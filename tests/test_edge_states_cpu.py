"""States at the u8 inventory limit, checked without a GPU.

The exported reference states never hold more than 12 of anything, so nothing there exercises the
one place where the kernels' state differs from the reference's: inventory counts are u8 in the
agent record (include/psk_craft.h) and float64 in the reference.  This module

  - derives such states from the exported ones (``edge_states``: counts in EDGE_COUNTS on the kinds
    that the next USE can touch), shared with tests/test_fused_states_gpu.py;
  - pins the C oracle (int32 counts) against the pure-Python port of the reference (float64
    counts, oracle/craft_ref_port.py) on them, so that the oracle is a trustworthy reference above
    count 12 as well;
  - states the documented overflow rule of psk_craft_step as a small model (``step_u8``) and checks
    it against the oracle wherever no count passes 255;
  - checks that the Python entry points reject caller state that does not fit the agent record
    before anything touches a device.
"""
import numpy as np
import pytest

from psketch_b200 import tables as T

EDGE_COUNTS = (13, 127, 128, 200, 254, 255)
MOVES = ((0, -1), (0, 1), (-1, 0), (1, 0))          # DOWN, UP, LEFT, RIGHT (worlds/craft.py:77-91)
USABLE = (T.KC_GRAB, T.KC_WORKSHOP, T.KC_WATER, T.KC_STONE)


def _recipes(tables):
    """(out, workshop, n_in, in0, cnt0, in1, cnt1, yield) in firing order."""
    return [tuple(int(v) for v in tables.recipes[r]) for r in range(tables.n_recipes)]


def _front(tables, x, y, d):
    fx, fy = x + MOVES[d][0], y + MOVES[d][1]
    return (fx, fy) if 0 <= fx < tables.W and 0 <= fy < tables.H else None


def edge_states(tables, S, n, seed):
    """n states derived from the exported states S: three quarters of them turned to face a cell that
    USE acts on (when one is adjacent), and inventory counts from EDGE_COUNTS (sometimes 0 or 1) on
    a few random carryable kinds plus every kind the next USE can touch: the faced grabbable kind,
    the inputs and outputs of the recipes of the faced workshop, the bridge in front of water and
    the axe in front of stone.  Returns dict(grid u8[n, C], inv i32[n, K], pos i32[n, 2], dir i32[n],
    src: the exported state each one came from)."""
    rng = np.random.RandomState(seed)
    H, kc = tables.H, tables.kind_class
    src = rng.randint(0, len(S["grid"]), size=n)
    grid = S["grid"][src].copy()
    inv = S["inv"][src].astype(np.int32)
    pos = S["pos"][src].astype(np.int32)
    dirs = S["dir"][src].astype(np.int32)
    carried = [k for k in range(1, tables.K) if k not in tables.cookbook.environment]
    recipes = _recipes(tables)
    for i in range(n):
        x, y = int(pos[i, 0]), int(pos[i, 1])
        if rng.rand() < 0.75:
            usable = [d for d in range(4) if _front(tables, x, y, d) is not None
                      and kc[grid[i, _front(tables, x, y, d)[0] * H + _front(tables, x, y, d)[1]]] in USABLE]
            if usable:
                dirs[i] = rng.choice(usable)
        f = _front(tables, x, y, int(dirs[i]))
        thing = int(grid[i, f[0] * H + f[1]]) if f is not None else 0
        kinds = set(int(k) for k in rng.choice(carried, size=rng.randint(1, 4), replace=False))
        if kc[thing] == T.KC_GRAB:
            kinds.add(thing)
        elif kc[thing] == T.KC_WORKSHOP:
            for out, ws, n_in, i0, _, i1, _, _ in recipes:
                if ws == thing:
                    kinds |= {out} | ({i0} if n_in > 0 else set()) | ({i1} if n_in > 1 else set())
        elif kc[thing] == T.KC_WATER and tables.bridge_kind:
            kinds.add(tables.bridge_kind)
        elif kc[thing] == T.KC_STONE and tables.axe_kind:
            kinds.add(tables.axe_kind)
        for k in sorted(kinds):
            inv[i, k] = rng.choice(EDGE_COUNTS) if rng.rand() < 0.85 else rng.randint(0, 2)
    return dict(grid=grid, inv=inv, pos=pos, dir=dirs, src=src)


def step_u8(tables, grid, inv, pos, dirs, action):
    """CraftState.step with the u8 inventory of the agent record, as psk_craft_step documents it
    (psk_craft.cu, step_env): a grab whose count is 255 clears the cell and keeps the count; a recipe
    whose output would pass 255 is skipped (its inputs stay) and the later recipes of the workshop
    still fire; both raise PSK_FLAG_INV_OVERFLOW.  Elsewhere the reference's rule.
    Returns (grid, inv, pos, dir, overflow bool[n], peak i32[n]); peak is the largest count the
    reference's own (unbounded) step reaches on the way, which can pass 255 even where its final
    counts do not: a later recipe may consume the output of an earlier one."""
    H, W, kc = tables.H, tables.W, tables.kind_class
    grid, inv = grid.copy(), inv.astype(np.int32)
    pos, dirs = pos.astype(np.int32), dirs.astype(np.int32)
    over = np.zeros(len(grid), bool)
    peak = inv.max(axis=1) if inv.shape[1] else np.zeros(len(grid), np.int32)
    recipes = _recipes(tables)
    for i in range(len(grid)):
        x, y, d, a = int(pos[i, 0]), int(pos[i, 1]), int(dirs[i]), int(action[i])
        if a < 4:
            dirs[i] = a
            tx, ty = x + MOVES[a][0], y + MOVES[a][1]
            if 0 <= tx < W and 0 <= ty < H and grid[i, tx * H + ty] == 0:
                pos[i] = (tx, ty)
        elif a == 4:
            f = _front(tables, x, y, d)
            if f is None:
                continue
            c = f[0] * H + f[1]
            thing = int(grid[i, c])
            if kc[thing] == T.KC_GRAB:
                peak[i] = max(peak[i], inv[i, thing] + 1)
                if inv[i, thing] == 255:
                    over[i] = True
                else:
                    inv[i, thing] += 1
                grid[i, c] = 0
            elif kc[thing] == T.KC_WORKSHOP:
                ref = inv[i].copy()                  # the reference's counts, unbounded
                for out, ws, n_in, i0, c0, i1, c1, yld in recipes:
                    if ws != thing:
                        continue
                    if not ((n_in > 0 and ref[i0] < c0) or (n_in > 1 and ref[i1] < c1)):
                        ref[out] += yld
                        ref[i0] -= c0 if n_in > 0 else 0
                        ref[i1] -= c1 if n_in > 1 else 0
                        peak[i] = max(peak[i], ref[out])
                    if (n_in > 0 and inv[i, i0] < c0) or (n_in > 1 and inv[i, i1] < c1):
                        continue
                    if inv[i, out] + yld > 255:
                        over[i] = True
                        continue
                    inv[i, out] += yld
                    if n_in > 0:
                        inv[i, i0] -= c0
                    if n_in > 1:
                        inv[i, i1] -= c1
            elif kc[thing] == T.KC_WATER and tables.bridge_kind and inv[i, tables.bridge_kind] > 0:
                grid[i, c] = 0
                inv[i, tables.bridge_kind] -= 1
            elif kc[thing] == T.KC_STONE and tables.axe_kind and inv[i, tables.axe_kind] > 0:
                grid[i, c] = 0
    return grid, inv, pos, dirs, over, peak


@pytest.fixture(params=["medium", "custom"])
def world(request, medium_tables, medium_states, custom_tables, custom_states):
    from oracle.craft_oracle import CraftOracle
    tables, S = {"medium": (medium_tables, medium_states), "custom": (custom_tables, custom_states)}[request.param]
    return tables, CraftOracle(tables), S


def test_edge_states_reach_the_limit(world):
    """The generator produces what the GPU tests rely on: every edge count, a faced grabbable kind at
    255, a faced workshop whose first fireable recipe overflows while a later one still fires, and
    steps that stay within 255."""
    tables, oracle, S = world
    E = edge_states(tables, S, 4096, seed=1)
    assert E["inv"].max() == 255 and E["inv"].min() >= 0
    for v in EDGE_COUNTS:
        assert (E["inv"] == v).sum() > 20, v
    use = np.full(len(E["grid"]), 4)
    g, iv, p, d, over, peak = step_u8(tables, E["grid"], E["inv"], E["pos"], E["dir"], use)
    og, oi, _, _, _ = oracle.step(E["grid"], E["inv"], E["pos"], E["dir"], use)
    grab_over = over & (g != E["grid"]).any(axis=1)
    recipe_over = over & (g == E["grid"]).all(axis=1)
    assert grab_over.sum() > 10 and recipe_over.sum() > 10
    # some overflowing workshop still fired another recipe
    assert ((iv != E["inv"]).any(axis=1) & recipe_over).sum() > 5
    # USE changed counts without passing 255, and reached 255 exactly
    assert (~over & (oi != E["inv"]).any(axis=1)).sum() > 100
    assert (~over & (oi == 255).any(axis=1) & (E["inv"] == 254).any(axis=1)).sum() > 5
    assert np.array_equal(over, peak > 255) and (oi.max(axis=1) <= peak).all()


def test_oracle_matches_the_reference_port_above_count_12(world):
    """C oracle (int32 counts) against the pure-Python port of the reference (float64 counts): features,
    step for all six actions (counts may pass 255 here, as in the reference), satisfies and the
    teacher for every task."""
    from oracle import craft_ref_port as port
    tables, oracle, S = world
    E = edge_states(tables, S, 160, seed=2)
    grid, inv, pos, dirs = E["grid"], E["inv"], E["pos"], E["dir"]
    n = len(grid)
    pw, teacher, tm = port.PortWorld(tables), port.PortTeacher(), tables.task_manager
    feats = oracle.features(grid, inv, pos, dirs)
    steps = [oracle.step(grid, inv, pos, dirs, np.full(n, a)) for a in range(6)]
    tids = list(range(1, tables.n_tasks))
    sat = {t: oracle.satisfies(grid, inv, pos, dirs, np.full(n, t)) for t in tids}
    exp = {t: oracle.expert(grid, inv, pos, dirs, np.full(n, t))[0] for t in tids}
    for i in range(n):
        s = port.PortState(pw, pw.onehot(grid[i]), (int(pos[i, 0]), int(pos[i, 1])), int(dirs[i]),
                           inv[i].astype(np.float64))
        assert np.array_equal(s.features(), feats[i].astype(np.float64)), i
        for a in range(6):
            _, s2 = s.step(a)
            g2, i2, p2, d2, _ = steps[a]
            assert np.array_equal(s2.grid.argmax(2) * (s2.grid.sum(2) > 0), g2[i].reshape(tables.W, tables.H)), (i, a)
            assert np.array_equal(s2.inventory, i2[i].astype(np.float64)), (i, a)
            assert s2.pos == tuple(p2[i]) and s2.dir == d2[i], (i, a)
        for t in tids:
            task = tm.by_id(t)
            v = s.satisfies(task)
            assert (2 if v is None else int(bool(v))) == sat[t][i], (i, t)
            try:
                a = teacher(task, s)
            except AssertionError:
                a = 255
            except TypeError:          # the reference's TypeError: the oracle's answer is the definition
                continue
            assert a == exp[t][i], (i, t)


def test_u8_step_rule_equals_the_oracle_below_the_limit(world):
    """step_u8 is the oracle wherever the oracle's counts stay <= 255 throughout the step, and flags
    exactly the rest; on those envs the faced grabbable cell is cleared with the count left at 255, or
    the overflowing recipe's output and inputs are unchanged."""
    tables, oracle, S = world
    E = edge_states(tables, S, 3000, seed=3)
    n = len(E["grid"])
    for a in range(6):
        act = np.full(n, a)
        g, iv, p, d, over, peak = step_u8(tables, E["grid"], E["inv"], E["pos"], E["dir"], act)
        og, oi, op, od, st = oracle.step(E["grid"], E["inv"], E["pos"], E["dir"], act)
        assert (st == 0).all()
        assert np.array_equal(over, peak > 255) and (oi.max(axis=1) <= peak).all(), a
        assert (over >= (oi.max(axis=1) > 255)).all(), a
        ok = ~over
        assert np.array_equal(g[ok], og[ok]) and np.array_equal(iv[ok], oi[ok]), a
        assert np.array_equal(p, op) and np.array_equal(d, od), a
        assert iv.max() <= 255 and iv.min() >= 0
        if a != 4:
            assert not over.any()
            continue
        grabbed = over & (g != E["grid"]).any(axis=1)
        for i in np.nonzero(grabbed)[0]:
            f = _front(tables, int(E["pos"][i, 0]), int(E["pos"][i, 1]), int(E["dir"][i]))
            thing = E["grid"][i, f[0] * tables.H + f[1]]
            assert g[i, f[0] * tables.H + f[1]] == 0 and iv[i, thing] == 255 == E["inv"][i, thing]


# ------------------------------------------------------------------------------------------------
# input validation: caller state that does not fit the agent record is rejected before any device
# work (these run without a GPU: the checks come before the first CUDA call)

def _good(medium_states, n=4):
    S = medium_states
    return dict(grid=S["grid"][:n], inv=S["inv"][:n].astype(np.int64), pos=S["pos"][:n].astype(np.int64),
                dirs=S["dir"][:n].astype(np.int64), task=np.full(n, 24))


BAD_STATES = [
    ("inv", (0, 3), 256), ("inv", (1, 0), 300), ("inv", (2, 5), -1), ("inv", (3, 2), 2.5),
    ("pos", (0, 0), 8), ("pos", (1, 1), 8), ("pos", (2, 0), -1), ("pos", (3, 1), 300),
    ("dirs", (0,), 4), ("dirs", (1,), -1),
    ("task", (0,), 27), ("task", (2,), -1),
]


@pytest.mark.parametrize("field,where,value", BAD_STATES)
def test_from_states_rejects_state_outside_the_record(field, where, value, medium_tables, medium_states):
    from psketch_b200.vec import VecCraft
    kw = _good(medium_states)
    kw[field] = kw[field].astype(np.float64) if isinstance(value, float) else kw[field].copy()
    kw[field][where] = value
    with pytest.raises(ValueError):
        VecCraft.from_states(medium_tables, kw["grid"], kw["inv"], kw["pos"], kw["dirs"], task=kw["task"])


BAD_INSTANCES = [("pos", (0, 0), 8), ("pos", (3, 1), -2), ("dirs", (1,), 7), ("task", (0,), 99),
                 ("task", (3,), -1), ("scen", (0,), 4), ("scen", (2,), -1)]


@pytest.mark.parametrize("entry", ["VecCraft", "HostCraft"])
@pytest.mark.parametrize("field,where,value", BAD_INSTANCES)
def test_instances_reject_state_outside_the_record(entry, field, where, value, medium_tables, medium_states):
    """VecCraft.from_instances and HostCraft: positions, facings, task ids and scenario indices."""
    kw = _good(medium_states)
    kw["scen"] = np.arange(4)
    kw[field] = kw[field].copy()
    kw[field][where] = value
    if entry == "VecCraft":
        from psketch_b200.vec import VecCraft as make
        call = lambda: make.from_instances(medium_tables, kw["grid"], kw["scen"], kw["pos"], kw["task"],
                                           init_dir=kw["dirs"])
    else:
        from psketch_b200.host import HostCraft as make
        call = lambda: make(medium_tables, kw["grid"], kw["scen"], kw["pos"], kw["task"], init_dir=kw["dirs"])
    with pytest.raises(ValueError):
        call()


def test_good_state_passes_validation(medium_tables, medium_states):
    from psketch_b200 import _lib
    kw = _good(medium_states)
    kw["inv"][0, 3] = 255
    kw["pos"][1] = (7, 7)
    kw["dirs"][2] = 3
    kw["task"][3] = 26
    _lib.check_agent_inputs(medium_tables, inv=kw["inv"], pos=kw["pos"], dirs=kw["dirs"], task=kw["task"],
                            scen_idx=np.arange(4), n_scen=4)


def test_facade_inventory_setter_rejects_counts_above_255(medium_tables, medium_states):
    from psketch_b200.worlds import craft as facade
    world = facade.CraftWorld(tables=medium_tables)
    s = world.init_state(medium_states["grid"][0], tuple(int(v) for v in medium_states["pos"][0]))
    inv = np.zeros(medium_tables.K)
    inv[7] = 300
    with pytest.raises(ValueError):
        s.inventory = inv
    inv[7] = 255
    s.inventory = inv
    assert s.inventory[7] == 255.0
