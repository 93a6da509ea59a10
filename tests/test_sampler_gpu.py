"""The Philox sampler kernels (psketch_b200/csrc/psk_scenario.cu) byte for byte against their C
restatement (oracle/sampler_oracle.c, pinned to the Philox known answers by
tests/test_sampler_cpu.py): scenarios at 8x8 and 10x10 with the stock and a custom cookbook, start
cells, random actions, and the entry points built on them (generate_dataset, CraftWorld).  Every
output buffer is poisoned before each call, and seeds, offsets and clocks reach past 2^32 and wrap
at 2^64.  Batches past one wave of the launch cap (WAVE) make the grid-stride loops go round."""
import ctypes

import numpy as np
import pytest

from oracle import sampler_oracle as so

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

WAVE = 148 * 16 * 128          # scenarios / groups per pass of the capped grid (= 148 * 8 * 256 action slots)
POISON = 0xA5
FAIL0 = 1000                   # fail_count starts here: the kernels add to it
U64 = 1 << 64


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _stream():
    from psketch_b200 import _lib
    return _lib.raw_stream(torch, torch.device("cuda", torch.cuda.current_device()))


@pytest.fixture(scope="module", params=["medium", "large", "custom"])
def world(request, medium_tables, large_tables, custom_tables):
    return {"medium": medium_tables, "large": large_tables, "custom": custom_tables}[request.param]


def _kernel_scenarios(tables, n, seed, offset, place_kinds):
    from psketch_b200 import _lib
    lib = _lib.load()
    ct = _lib.make_tables(tables)
    cs = so.cell_stride(tables.W, tables.H)
    pk = torch.from_numpy(np.asarray(list(place_kinds) + [POISON], np.uint8)).cuda()
    grid = torch.full((n, cs), POISON, dtype=torch.uint8, device="cuda")
    pos = torch.full((n, 2), POISON, dtype=torch.uint8, device="cuda")
    fails = torch.full((1,), FAIL0, dtype=torch.int32, device="cuda")
    rc = lib.psk_craft_sample_scenarios(ctypes.byref(ct), _ptr(grid), _ptr(pos), _ptr(pk), len(place_kinds),
                                        tables.cookbook.index["boundary"], ctypes.c_uint64(seed),
                                        ctypes.c_uint64(offset), n, cs, _ptr(fails), _stream())
    _lib.check(rc, "psk_craft_sample_scenarios")
    return grid.cpu().numpy(), pos.cpu().numpy(), int(fails.item()) - FAIL0


def _check_scenarios(tables, n, seed, offset, place_kinds):
    g, p, f = _kernel_scenarios(tables, n, seed, offset, place_kinds)
    og, op, of = so.sample_scenarios(tables.W, tables.H, place_kinds, tables.cookbook.index["boundary"],
                                     seed, offset, n)
    bad = np.flatnonzero((g != og).any(axis=1) | (p != op).any(axis=1))
    assert bad.size == 0, "scenario %d of n=%d seed=%d offset=%d differs: %s / %s vs oracle %s / %s" % (
        bad[0], n, seed, offset, g[bad[0]].tolist(), p[bad[0]].tolist(), og[bad[0]].tolist(), op[bad[0]].tolist())
    assert f == of, (n, seed, offset, f, of)
    return g, p, f


def _default(tables):
    from psketch_b200.data import default_placement
    return list(default_placement(tables))


def test_scenarios_batch_sizes_and_past_one_wave(world):
    pk = _default(world)
    for n in (1, 127, 128, 129, 4099):
        _, _, f = _check_scenarios(world, n, 123, 0, pk)
        assert f == 0
    big, _, f = _check_scenarios(world, WAVE + 4099, 123, 0, pk)
    assert f == 0
    # the stream depends on (seed, index + offset) only: a later launch is a slice of this one
    part, _, _ = _kernel_scenarios(world, 700, 123, WAVE - 300, pk)
    assert np.array_equal(part, big[WAVE - 300:WAVE + 400])


def test_scenarios_seeds_and_offsets(world):
    pk = _default(world)
    got = {}
    for seed in (0, 123, (1 << 32) + 123, U64 - 1):
        got[seed], _, f = _check_scenarios(world, 4099, seed, 0, pk)
        assert f == 0
    assert (got[123] != got[(1 << 32) + 123]).any(axis=1).mean() > 0.99     # the key's high word is used
    assert (got[0] != got[U64 - 1]).any(axis=1).mean() > 0.99
    # offsets whose streams cross into the high counter word, and wrap at 2^64
    start, _, _ = _kernel_scenarios(world, 6, 123, 0, pk)
    for seed in (123, U64 - 1):
        _check_scenarios(world, 8, seed, (1 << 32) - 3, pk)
        _check_scenarios(world, 8, seed, U64 - 2, pk)
    cross, _, _ = _kernel_scenarios(world, 8, 123, (1 << 32) - 3, pk)
    assert (cross[3:] != start[:5]).any(axis=1).all()        # streams 2^32.. are not streams 0..
    wrap, _, _ = _kernel_scenarios(world, 8, 123, U64 - 2, pk)
    assert np.array_equal(wrap[2:], start)                    # streams wrap at 2^64


def test_scenarios_place_lists_and_failure_path(world):
    K = world.K
    kinds = [k for k in range(2, K) if k != world.cookbook.index["boundary"]]
    C = world.W * world.H
    for pk, n in (([], 4099), ([kinds[0]], 4099), ([kinds[-1]], 129), (_default(world), 129)):
        _, _, f = _check_scenarios(world, n, 7, 11, pk)
        assert f == 0
    # lists that fit only sometimes, and lists that never fit (every row partial, start (0, 0))
    cycle = lambda m: [kinds[i % len(kinds)] for i in range(m)]
    some, never = (17, 30) if C == 64 else (33, 60)
    g, p, f = _check_scenarios(world, 1000, 123, 0, cycle(some))
    assert 0 < f < 1000
    failed = (p == 0).all(axis=1)
    assert failed.sum() == f
    placed = (g[:, :C].reshape(-1, world.W, world.H)[:, 1:-1, 1:-1] != 0).sum(axis=(1, 2))
    assert (placed[~failed] == some).all() and (placed[failed] <= some).all()
    g, p, f = _check_scenarios(world, 129, 5, U64 - 7, cycle(never))
    assert f == 129 and (p == 0).all()


def test_scenarios_public_entry_point(world):
    from psketch_b200 import data
    g, p, f = data.sample_scenarios(world, 4099, seed=99, offset=(1 << 32) - 1000)
    og, op, of = so.sample_for(world, 4099, 99, (1 << 32) - 1000)
    assert f == of == 0
    assert np.array_equal(g.cpu().numpy(), og) and np.array_equal(p.cpu().numpy(), op)
    with pytest.raises(ValueError):
        data.sample_scenarios(world, 4, seed=1, place_kinds=[0])


# ------------------------------------------------------------------------------- start cells
def _kernel_positions(tables, scen_grid, group_scen, per_group, seed, offset, cell_stride=None):
    from psketch_b200 import _lib
    lib = _lib.load()
    ct = _lib.make_tables(tables)
    sg = torch.from_numpy(np.ascontiguousarray(scen_grid)).cuda()
    gs = torch.from_numpy(np.asarray(group_scen, np.int32)).cuda()
    out = torch.full((len(gs), per_group, 2), POISON, dtype=torch.uint8, device="cuda")
    fails = torch.full((1,), FAIL0, dtype=torch.int32, device="cuda")
    rc = lib.psk_craft_sample_positions(ctypes.byref(ct), _ptr(sg), _ptr(gs), per_group, _ptr(out),
                                        ctypes.c_uint64(seed), ctypes.c_uint64(offset), len(gs),
                                        sg.shape[1] if cell_stride is None else cell_stride, _ptr(fails),
                                        _stream())
    if rc != _lib.PSK_OK:
        return rc
    return out.cpu().numpy(), int(fails.item()) - FAIL0


@pytest.mark.parametrize("name", ["medium", "large"])
def test_positions(name, medium_tables, large_tables):
    from psketch_b200 import _lib, data
    t = medium_tables if name == "medium" else large_tables
    W, H = t.W, t.H
    grid, _, f = so.sample_for(t, 64, 31)
    assert f == 0
    n_free = int((grid[0, :W * H] == 0).sum())
    assert (grid[:, :W * H] == 0).sum(axis=1).tolist() == [n_free] * 64
    rng = np.random.RandomState(4)
    gs = rng.randint(0, 64, size=300).astype(np.int32)          # repeated and out of order
    gs[:4] = [63, 0, 63, 5]
    for per_group in (1, 20, n_free, n_free + 3):
        for seed, offset in ((123, 0), ((1 << 32) + 7, (1 << 32) - 3), (U64 - 1, U64 - 100)):
            out, fails = _kernel_positions(t, grid, gs, per_group, seed, offset)
            want, wfails = so.sample_positions(W, H, grid, gs, per_group, seed, offset)
            assert np.array_equal(out, want), (per_group, seed, offset)
            assert fails == wfails == len(gs) * max(0, per_group - n_free)
            if per_group >= n_free:                 # every free cell once, then 255/255
                for g in (0, 1, 2, 3):
                    cells = {tuple(c) for c in out[g, :n_free]}
                    free = {(c // H, c % H) for c in np.flatnonzero(grid[gs[g], :W * H] == 0)}
                    assert cells == free
                    assert (out[g, n_free:] == 255).all()
    # past one wave of groups
    gs = rng.randint(0, 64, size=WAVE + 77).astype(np.int32)
    out, fails = _kernel_positions(t, grid, gs, 2, 9, 0)
    want, _ = so.sample_positions(W, H, grid, gs, 2, 9, 0)
    assert fails == 0 and np.array_equal(out, want)
    # the public entry point: same answer, PskError when a group cannot get its cells
    sg = torch.from_numpy(grid).cuda()
    got = data.sample_positions(t, sg, gs[:500], 20, 77, 5).cpu().numpy()
    assert np.array_equal(got, so.sample_positions(W, H, grid, gs[:500], 20, 77, 5)[0])
    with pytest.raises(_lib.PskError):
        data.sample_positions(t, sg, gs[:10], n_free + 1, 77)
    with pytest.raises(ValueError):
        data.sample_positions(t, sg, [0, 64], 1, 77)
    assert _kernel_positions(t, grid, gs[:10], 1, 1, 0, cell_stride=W * H - 1) == _lib.PSK_ERR_BADARG


# ------------------------------------------------------------------------------- random actions
def _kernel_actions(n, ticks, n_actions, seed, t, clock=None, block=True):
    from psketch_b200 import _lib
    lib = _lib.load()
    out = torch.full((ticks, n), POISON, dtype=torch.uint8, device="cuda")
    t_dev = None
    if clock is not None:
        t_dev = torch.tensor([clock - U64 if clock >= 1 << 63 else clock], dtype=torch.int64, device="cuda")
    dev = _ptr(t_dev) if t_dev is not None else None
    if block:
        rc = lib.psk_random_actions_block(_ptr(out), n, ticks, n_actions, ctypes.c_uint64(seed),
                                          ctypes.c_uint64(t), dev, _stream())
    else:
        assert ticks == 1
        rc = lib.psk_random_actions(_ptr(out), n, n_actions, ctypes.c_uint64(seed), ctypes.c_uint64(t), dev,
                                    _stream())
    if rc != _lib.PSK_OK:
        return rc
    return out.cpu().numpy()


def test_random_actions():
    from psketch_b200 import _lib
    for n_actions in (1, 2, 6, 7, 255):
        for n, ticks in ((1, 1), (129, 3), (4099, 8), (70001, 5)):             # 350,005 > one wave
            for seed, t in ((123, 0), ((1 << 32) + 123, (1 << 32) - 3), (U64 - 1, U64 - 3)):
                want = so.random_actions(n, ticks, n_actions, seed, t)
                assert np.array_equal(_kernel_actions(n, ticks, n_actions, seed, t), want), (n_actions, n, ticks)
                if ticks == 1 or n == 4099:
                    for k in range(0, ticks, 3):
                        got = _kernel_actions(n, 1, n_actions, seed, (t + k) % U64, block=False)
                        assert np.array_equal(got[0], want[k]), (n_actions, n, k)
        n = WAVE + 1234
        assert np.array_equal(_kernel_actions(n, 1, n_actions, 5, 17, block=False),
                              so.random_actions(n, 1, n_actions, 5, 17))
    for n_actions in (0, 256):
        assert _kernel_actions(8, 2, n_actions, 1, 0) == _lib.PSK_ERR_BADARG
        assert _kernel_actions(8, 1, n_actions, 1, 0, block=False) == _lib.PSK_ERR_BADARG
    # a device clock above 2^32 and one that wraps the counter
    for clock in ((1 << 32) + 5, U64 - 2):
        for t in (0, 3):
            want = so.random_actions(4099, 8, 6, 123, t + clock)
            assert np.array_equal(_kernel_actions(4099, 8, 6, 123, t, clock=clock), want)
            assert np.array_equal(_kernel_actions(4099, 1, 6, 123, t, clock=clock, block=False), want[:1])


def test_vec_random_actions_device_clock(medium_tables):
    from psketch_b200.vec import VecCraft
    grid, pos, _ = so.sample_for(medium_tables, 16, 3)
    n = 5000
    env = VecCraft.from_instances(medium_tables, grid[:, :64], np.arange(n) % 16, pos[np.arange(n) % 16],
                                  np.ones(n, np.int32))
    for clock in ((1 << 32) + 5, U64 - 2):
        env.stats[2] = clock - U64 if clock >= 1 << 63 else clock
        got = env.random_actions(t=4, seed=123, device_clock=True, ticks=6).cpu().numpy()
        assert np.array_equal(got, so.random_actions(n, 6, 6, 123, 4 + clock))
        got = env.random_actions(t=0, seed=9, device_clock=True).cpu().numpy()
        assert np.array_equal(got, so.random_actions(n, 1, 6, 9, clock)[0])


# ------------------------------------------------------------------------------- end to end
def _oracle_dataset_grids(tables, n_worlds, seed):
    """generate_dataset's rule: the first n_worlds distinct scenarios in (seed, offset) order,
    drawn 2 * n_worlds per launch."""
    C = tables.W * tables.H
    grids, seen, offset = [], set(), 0
    while len(grids) < n_worlds:
        g, _, f = so.sample_for(tables, 2 * n_worlds, seed, offset)
        assert f == 0
        offset += 2 * n_worlds
        for row in g[:, :C]:
            if row.tobytes() not in seen and len(grids) < n_worlds:
                seen.add(row.tobytes())
                grids.append(row)
    return np.stack(grids)


@pytest.mark.parametrize("name", ["medium", "large"])
def test_generate_dataset(name, medium_tables, large_tables):
    from psketch_b200 import data
    from oracle.craft_oracle import CraftOracle
    from test_oracle import _replay
    t = medium_tables if name == "medium" else large_tables
    n_worlds, n_pos, seed = 40, 20, 7
    packed = data.generate_dataset(t, n_worlds=n_worlds, n_pos=n_pos, seed=seed)
    grids = _oracle_dataset_grids(t, n_worlds, seed)
    assert np.array_equal(packed["grids"], grids)
    tasks = [tk.task_id for tk in t.task_manager.tasks if tk.goal_name in ("get", "make")]
    gs = np.repeat(np.arange(n_worlds, dtype=np.int32), len(tasks))
    sg = np.zeros((n_worlds, so.cell_stride(t.W, t.H)), np.uint8)
    sg[:, :t.W * t.H] = grids
    pos, f = so.sample_positions(t.W, t.H, sg, gs, n_pos, seed ^ 0x9E3779B97F4A7C15)
    assert f == 0 and np.array_equal(packed["inst_pos"], pos.reshape(-1, 2))
    ref, ln = packed["ref_actions"], packed["ref_len"]
    assert (ref[np.arange(len(ln)), ln - 1] == 5).all() and ln.max() < 64
    pad = np.where(ref == 255, 5, ref).astype(np.int32)
    assert _replay(CraftOracle(t), packed["grids"], packed["inst_env"], packed["inst_task"],
                   packed["inst_pos"], pad, ln) == 0


@pytest.mark.parametrize("name", ["craft_medium", "craft_large"])
def test_world_sample_scenario_follows_the_oracle(name):
    from psketch_b200.worlds import CraftWorld
    from psketch_b200.worlds.craft import _Struct
    world = CraftWorld(_Struct(world={"config": name}))
    W, H = world.tables.W, world.tables.H
    og, op, _ = so.sample_for(world.tables, 512, 123, 0)
    for k in range(300):                              # crosses a pool refill (256 per launch)
        grid, pos = world.sample_scenario()
        ids = grid.argmax(axis=2) * (grid.sum(axis=2) > 0)
        assert np.array_equal(ids.reshape(-1), og[k, :W * H]) and pos == tuple(op[k]), k
