"""The generic tier (psketch_b200/csrc/psk_craft_generic.cu): Craft worlds of any geometry of the
generic domain (1 <= W, H <= 64, odd windows of 1..9 cells per axis, at most 24 kinds) on every entry
point, compared byte for byte with the C oracle (oracle/craft_oracle.py):

  - thin boards, small and large windows, non-square grids and windows, up to 64x64 with a 9x9 window,
    with the stock cookbook (21 kinds) and tests/golden/custom (20 kinds);
  - step (every action, invalid bytes), features (f32, u8), satisfies (every task), the teacher with
    its distance, find_closest (every go-kind, several caps), reset;
  - the tick in all four orders and the byte-frame tick, the rollout (f32 and byte frames, a ring
    shorter than the rollout), HostCraft (state round trip and resident ticks);
  - n = 1, odd n, and batches past one wave of every grid-stride loop;
  - with the tuning key `generic` = 1 on the five built geometries: every output identical to the
    specialised kernels', on the reference's exported states and the stress families;
  - CraftWorld from a world yaml, teacher_rollouts, and guard bands around every buffer.

Every output buffer is poisoned before the call, so a row the kernel never wrote cannot match."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from test_edge_states_cpu import step_u8                                              # noqa: E402
from test_generic_geometry_cpu import board_states, generic_tables, good_tasks        # noqa: E402
from test_stress_limits_gpu import (POISON, _OracleTicks, _poisoned, run_expert,      # noqa: E402
                                    run_find_closest, tuning)
from test_stress_states_cpu import (all_families, concat, go_kinds, inventory_states,  # noqa: E402
                                    maze_states, random_states, ringless_states, stress_tables, take)

pytestmark = pytest.mark.gpu

KEYS = ("grid", "inv", "pos", "dir", "task")
# (W, H, window_w, window_h): thin boards, then the geometries of the generic domain's edges
GEOMETRIES = [(2, 9, 3, 1), (3, 12, 3, 3), (17, 3, 1, 5), (5, 7, 1, 1), (9, 9, 3, 3), (8, 8, 5, 5),
              (8, 8, 7, 7), (12, 12, 5, 5), (20, 13, 3, 5), (20, 13, 9, 1), (33, 17, 5, 5), (64, 64, 9, 9)]
BOOKS = ("stock", "custom")
TICKS, T_MAX = 7, 4


def _np(t):
    return t.cpu().numpy()


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _oracle(tables):
    from oracle.craft_oracle import CraftOracle
    return CraftOracle(tables)


def _env(tables, S, T=40):
    from psketch_b200.vec import VecCraft
    return VecCraft.from_states(tables, S["grid"], S["inv"], S["pos"], S["dir"], task=S["task"], max_timesteps=T)


def geometry_states(tables, seed):
    """The thin-board generator (any W, H) and the ringless family everywhere; the random, inventory
    and (square boards) maze families where the board is large enough for their item mix."""
    W, H = tables.W, tables.H
    parts = [board_states(tables, 67, seed), ringless_states(tables, seed + 1, n_near=20)]
    if min(W, H) >= 8:
        parts += [random_states(tables, 41, seed + 2), inventory_states(tables, 21, seed + 3)]
    if W == H and W >= 8:
        parts.append(maze_states(tables, 8, seed + 4))
    return concat([{k: np.asarray(p[k]).astype(np.int32) if k != "grid" else p[k] for k in KEYS} for p in parts])


def episode_states(tables, seed):
    """Episode starts: empty inventories, facing 0, a task the teacher answers."""
    S = geometry_states(tables, seed)
    S["inv"] = np.zeros_like(S["inv"])
    S["dir"] = np.zeros_like(S["dir"])
    S["task"] = np.random.RandomState(seed).choice(good_tasks(tables), size=len(S["grid"])).astype(np.int32)
    return S


@pytest.fixture(params=GEOMETRIES, ids=lambda g: "%dx%d_w%dx%d" % g)
def geometry(request):
    return request.param


@pytest.fixture(params=BOOKS)
def book(request):
    return request.param


def _setup(geometry, book, seed=0):
    tables = generic_tables(*geometry, book=book)
    return tables, _oracle(tables), geometry_states(tables, 1000 * sum(geometry) + seed + len(book))


# ------------------------------------------------------------------------------------------------
# primitives

def check_teacher(tables, o, S, tag):
    want_a, want_d, _ = o.expert(S["grid"], S["inv"], S["pos"], S["dir"], S["task"])
    env = _env(tables, S)
    for task in (None, S["task"]):
        a, d = run_expert(env, task)
        assert np.array_equal(a, want_a), (tag, np.flatnonzero(a != want_a)[:8])
        assert np.array_equal(d, want_d), (tag, np.flatnonzero(d != want_d)[:8])
        env.check_errors()
    return want_a, want_d


def check_closest(tables, o, S, kind, cap, tag):
    env = _env(tables, S)
    g, ln, seq = run_find_closest(env, kind, cap)
    og, ol, st, oseq = o.find_closest(S["grid"], S["pos"], S["dir"], kind, seq_cap=cap)
    ok = st != 2                            # status 2: the reference raised TypeError
    assert np.array_equal(ln[ok], ol[ok]), (tag, np.flatnonzero(ln[ok] != ol[ok])[:8])
    assert np.array_equal(g[ok], np.where(og < 0, 255, og)[ok]), tag
    if cap:
        assert np.array_equal(seq[ok], oseq[ok]), tag
    return ol


def check_step(tables, S, act, tag):
    bad = act > 5
    g, iv, p, d, over, _ = step_u8(tables, S["grid"], S["inv"], S["pos"], S["dir"], np.where(bad, 5, act))
    env = _env(tables, S)
    reward = _poisoned(env.n, torch.float32, env.device)
    env._reward = reward
    env.step(torch.from_numpy(act.astype(np.uint8)).to(env.device))
    assert (_np(reward) == 0).all(), tag
    assert np.array_equal(_np(env.cells), g), tag
    assert np.array_equal(_np(env.inventory).astype(np.int32), iv), tag
    assert np.array_equal(_np(env.pos).astype(np.int32), p), tag
    assert np.array_equal(_np(env.dir).astype(np.int32), d), tag
    if bad.any():
        with pytest.raises(Exception, match="Unexpected action"):
            env.check_errors()
    elif over.any():
        with pytest.raises(OverflowError):
            env.check_errors()
    else:
        env.check_errors()


def check_features(tables, o, S, tag):
    env = _env(tables, S)
    want = o.features(S["grid"], S["inv"], S["pos"], S["dir"])
    for impl in (0, 2):
        out = _poisoned((env.n, tables.n_features), torch.float32, env.device)
        env.features(out=out, impl=impl)
        assert np.array_equal(_np(out), want), (tag, impl)
    out = _poisoned((env.n, tables.n_features), torch.uint8, env.device)
    env.features_u8(out=out)
    assert np.array_equal(_np(out).astype(np.float32), want), (tag, "u8")


def check_satisfies(tables, o, S, tag):
    env = _env(tables, S)
    n = len(S["grid"])
    for t in range(1, tables.n_tasks):
        out = _poisoned(n, torch.uint8, env.device)
        tk = torch.full((n,), t, dtype=torch.uint8, device=env.device)
        with torch.cuda.device(env.device):
            assert env.lib.psk_craft_satisfies(ctypes.byref(env.ct), env._state(), _p(tk), _p(out), env._stream()) == 0
        want = o.satisfies(S["grid"], S["inv"], S["pos"], S["dir"], np.full(n, t))
        assert np.array_equal(_np(out).astype(np.int32), want), (tag, t)


def test_supported_and_feature_count(geometry, book):
    from psketch_b200 import _lib
    tables = generic_tables(*geometry, book=book)
    lib = _lib.load()
    ct = _lib.make_tables(tables)
    assert lib.psk_craft_supported(ctypes.byref(ct)) == 1
    assert lib.psk_craft_n_features(ctypes.byref(ct)) == tables.n_features


def test_teacher_and_find_closest(geometry, book):
    tables, o, S = _setup(geometry, book)
    a, d = check_teacher(tables, o, S, "all")
    assert (a < 4).any() and (a == 5).any() and (d > 0).any()
    n = len(S["grid"])
    for k in go_kinds(tables):
        check_closest(tables, o, S, np.full(n, k, np.int32), 0, ("kind", k))
    kind = np.random.RandomState(1).choice(go_kinds(tables), size=n).astype(np.int32)
    ol = check_closest(tables, o, S, kind, 0, "mixed kinds")
    L = int(np.median(ol[ol > 0])) if (ol > 0).any() else 1
    for cap in sorted({1, 31, 33, L, int(ol.max()) + 1}):
        check_closest(tables, o, S, kind, cap, ("cap", cap))


def test_satisfies_step_features(geometry, book):
    tables, o, S = _setup(geometry, book)
    check_satisfies(tables, o, S, "all")
    n = len(S["grid"])
    for a in range(6):
        check_step(tables, S, np.full(n, a), ("action", a))
    mixed = np.random.RandomState(2).choice(list(range(6)) + [6, 7, 100, 255], size=n)
    check_step(tables, S, mixed, "mixed with invalid bytes")
    check_features(tables, o, S, "all")


@pytest.mark.parametrize("geometry", [(9, 9, 3, 3), (20, 13, 3, 5)], ids=["9x9_w3x3", "20x13_w3x5"])
def test_batch_sizes(geometry):
    """n = 1, odd n, and past one wave of each grid-stride loop: 128-thread CTAs of one env per warp at
    16 CTAs per SM (teacher, find_closest, features) and 256-thread CTAs at 8 per SM (step,
    satisfies)."""
    tables, o, S = _setup(geometry, "stock")
    m = len(S["grid"])
    warp_wave, thread_wave = _sms() * 16 * 4, _sms() * 8 * 256
    rng = np.random.RandomState(7)

    def batch(k):
        return take(S, np.concatenate([rng.permutation(m) for _ in range(-(-k // m))])[:k])

    for k in (1, 3, 2 * warp_wave + 5):
        B = batch(k)
        check_teacher(tables, o, B, ("n", k))
        check_features(tables, o, B, ("n", k))
        kind = np.full(k, go_kinds(tables)[0], np.int32)
        check_closest(tables, o, B, kind, 5, ("n", k))
    B = batch(thread_wave + 7)
    B["inv"] = np.minimum(B["inv"], 200)             # no overflow: the oracle's step is the answer
    act = rng.randint(0, 6, size=len(B["grid"]))
    g, iv, p, d, _ = o.step(B["grid"], B["inv"], B["pos"], B["dir"], act)
    env = _env(tables, B)
    env.step(torch.from_numpy(act.astype(np.uint8)).to(env.device))
    env.check_errors()
    assert np.array_equal(_np(env.cells), g) and np.array_equal(_np(env.inventory).astype(np.int32), iv)
    assert np.array_equal(_np(env.pos).astype(np.int32), p) and np.array_equal(_np(env.dir).astype(np.int32), d)
    env = _env(tables, B)
    want = o.satisfies(B["grid"], B["inv"], B["pos"], B["dir"], B["task"])
    assert np.array_equal(_np(env.satisfies()).astype(np.int32), want)


# ------------------------------------------------------------------------------------------------
# ticks, rollouts, reset, host contexts

def _replay_ticks(tables, o, S, acts):
    ref = _OracleTicks(o, S["grid"], S["pos"], S["task"], T_MAX)
    return ref, [ref.tick(None if acts is None else acts[t]) for t in range(TICKS)]


def _actions(n, seed):
    return np.random.RandomState(seed).choice(6, size=(TICKS, n), p=[.2, .2, .2, .2, .15, .05]).astype(np.uint8)


@pytest.mark.parametrize("driver", ["teacher", "random"])
def test_tick_every_order(geometry, book, driver):
    """psk_craft_tick observe-then-step (f32 and bytes), the three-kernel pipeline, step-then-observe
    (f32 and bytes) and step-only-then-observe; each tick's outputs, the final state, the counters."""
    from psketch_b200.vec import VecCraft
    tables = generic_tables(*geometry, book=book)
    o = _oracle(tables)
    S = episode_states(tables, sum(geometry))
    n, nf, K = len(S["grid"]), tables.n_features, tables.K
    acts = None if driver == "teacher" else _actions(n, 3)
    ref, gold = _replay_ticks(tables, o, S, acts)
    assert sum(int(g["done"].sum()) for g in gold) > 0
    for mode in ("observe", "pipeline", "observe u8", "advance", "advance u8"):
        env = VecCraft.from_instances(tables, S["grid"], np.arange(n), S["pos"], S["task"], max_timesteps=T_MAX)
        u8, adv = mode.endswith("u8"), mode.startswith("advance")
        buf = _poisoned((n, nf), torch.uint8 if u8 else torch.float32, env.device)
        out = {k: _poisoned(n, torch.uint8, env.device) for k in ("expert", "done", "success")}

        def call(a):
            buf.fill_(POISON if u8 else -7.0)
            for v in out.values():
                v.fill_(POISON)
            env.tick(actions=a, features_out=buf, out=out, fused=mode != "pipeline", advance_first=adv)

        def observed(t, tag):
            assert np.array_equal(_np(out["expert"]), gold[t]["expert"]), tag
            assert np.array_equal(_np(buf).astype(np.float32), gold[t]["features"]), tag

        if adv:
            call(None)
            observed(0, (mode, "start"))
            assert not _np(out["done"]).any() and not _np(out["success"]).any()
        steps = TICKS - 1 if adv else TICKS
        for t in range(steps):
            tag = (mode, driver, t)
            call(acts[t] if acts is not None else (gold[t]["expert"] if adv else None))
            assert np.array_equal(_np(out["done"]), gold[t]["done"]), tag
            assert np.array_equal(_np(out["success"]), gold[t]["success"]), tag
            observed(t + 1 if adv else t, tag)
        env.check_errors()
        assert ref.state_equals(_np(env.cells), _np(env.agent), K, gold[steps - 1]["state"]), mode
        want = np.sum([(int(g["done"].sum()), int(g["success"].sum()), n) for g in gold[:steps]], axis=0)
        assert tuple(_np(env.stats)[:3]) == tuple(want), mode
    # step, then observe, without the episode rules (PSK_TICK_STEP_FIRST), f32 and bytes
    a = _actions(n, 4)[0]
    g, iv, p, d, _ = o.step(S["grid"], np.zeros((n, K), np.int32), S["pos"], np.zeros(n, np.int32), a)
    want_a, _, _ = o.expert(g, iv, p, d, S["task"])
    want_f = o.features(g, iv, p, d)
    for dt in (torch.float32, torch.uint8):
        env = VecCraft.from_instances(tables, S["grid"], np.arange(n), S["pos"], S["task"], max_timesteps=T_MAX)
        buf = _poisoned((n, nf), dt, env.device)
        ex = {"expert": _poisoned(n, torch.uint8, env.device)}
        env.step_observe(actions=torch.from_numpy(a).to(env.device), features_out=buf, out=ex)
        assert np.array_equal(_np(ex["expert"]).astype(np.int32), want_a), dt
        assert np.array_equal(_np(buf).astype(np.float32), want_f), dt
        assert np.array_equal(_np(env.cells), g), dt
        env.check_errors()


@pytest.mark.parametrize("driver", ["teacher", "random"])
def test_rollout_and_reset(geometry, book, driver):
    """psk_craft_rollout / _rollout_u8: TICKS ticks in one call into a 2-frame ring; then reset."""
    from psketch_b200.vec import VecCraft
    tables = generic_tables(*geometry, book=book)
    o = _oracle(tables)
    S = episode_states(tables, sum(geometry) + 1)
    n, nf, R = len(S["grid"]), tables.n_features, 2
    acts = None if driver == "teacher" else _actions(n, 5)
    ref, gold = _replay_ticks(tables, o, S, acts)
    for u8 in (False, True):
        env = VecCraft.from_instances(tables, S["grid"], np.arange(n), S["pos"], S["task"], max_timesteps=T_MAX)
        ring = _poisoned((R, n, nf), torch.uint8 if u8 else torch.float32, env.device)
        out = {k: _poisoned((TICKS, n), torch.uint8, env.device) for k in ("expert", "done", "success")}
        env.rollout(TICKS, actions=None if acts is None else torch.from_numpy(acts).cuda(), features_out=ring, out=out)
        for t in range(TICKS):
            for k in ("expert", "done", "success"):
                assert np.array_equal(_np(out[k][t]), gold[t][k]), (driver, u8, t, k)
        for t in (TICKS - 2, TICKS - 1):
            assert np.array_equal(_np(ring[t % R]).astype(np.float32), gold[t]["features"]), (driver, u8, t)
        env.check_errors()
        assert ref.state_equals(_np(env.cells), _np(env.agent), tables.K, gold[-1]["state"]), (driver, u8)
        assert tuple(_np(env.stats)[:3]) == tuple(ref.stats), (driver, u8)
        env.reset()
        assert np.array_equal(_np(env.cells), S["grid"]) and np.array_equal(_np(env.pos).astype(np.int32), S["pos"])


@pytest.mark.parametrize("geometry", [(3, 12, 3, 3), (9, 9, 3, 3), (20, 13, 3, 5)],
                         ids=["3x12_w3x3", "9x9_w3x3", "20x13_w3x5"])
def test_host_paths(geometry):
    """HostCraft with a chunk size that does not divide n: tick (state round trip) and tick_resident
    in every feature format and both orders; below the zero-copy size limit, so the generic tier's
    fallback to the copy route runs too."""
    from psketch_b200.host import HostCraft
    tables = generic_tables(*geometry)
    o = _oracle(tables)
    S0 = episode_states(tables, 11)
    n = 1000
    S = take(S0, np.random.RandomState(3).choice(len(S0["grid"]), n))
    K, C = tables.K, tables.W * tables.H
    acts = _actions(n, 6)
    ref = _OracleTicks(o, S["grid"], S["pos"], S["task"], T_MAX)
    gold = [ref.tick(acts[t]) for t in range(6)]
    for mode in ("tick", "f32", "u8", "f32_wire_u8", "advance f32", "advance u8"):
        h = HostCraft(tables, S["grid"], np.arange(n), S["pos"], S["task"], max_timesteps=T_MAX, chunk_envs=384,
                      host_threads=2)
        adv = mode.startswith("advance")
        fmt = mode.split()[-1]

        def call(a):
            h.expert[:] = POISON
            h.done[:] = POISON
            h.success[:] = POISON
            h.features[:] = -7.0
            h.features_u8[:] = POISON
            if mode == "tick":
                h.tick(actions=a)
            else:
                h.tick_resident(actions=a, features=fmt, advance_first=adv)

        def observed(t, tag):
            assert np.array_equal(h.expert, gold[t]["expert"]), tag
            f = h.features_u8.astype(np.float32) if fmt == "u8" else h.features
            assert np.array_equal(f, gold[t]["features"]), tag

        if adv:
            h.upload()
            call(None)
            observed(0, (mode, "start"))
        steps = 5 if adv else 6
        for t in range(steps):
            call(acts[t])
            assert np.array_equal(h.done, gold[t]["done"]) and np.array_equal(h.success, gold[t]["success"]), (mode, t)
            observed(t + 1 if adv else t, (mode, t))
        if mode != "tick":
            h.download(keep_resident=False)
        assert ref.state_equals(h.grid[:, :C], h.agent, K, gold[steps - 1]["state"]), mode
        h.close()


# ------------------------------------------------------------------------------------------------
# the generic tier forced on the five built geometries: identical to the specialised kernels

def _all_outputs(tables, S, acts):
    """Every entry point's outputs on S (poison-filled first), as numpy arrays."""
    from psketch_b200.vec import VecCraft
    n = len(S["grid"])
    res = {}
    env = _env(tables, S)
    res["expert"], res["dist"] = run_expert(env)
    kind = np.random.RandomState(0).choice(go_kinds(tables), size=n).astype(np.int32)
    res["goal"], res["len"], res["seq"] = run_find_closest(env, kind, 40)
    res["sat"] = _np(env.satisfies())
    f = _poisoned((n, tables.n_features), torch.float32, env.device)
    res["f32"] = _np(env.features(out=f))
    b = _poisoned((n, tables.n_features), torch.uint8, env.device)
    res["u8"] = _np(env.features_u8(out=b))
    snap = env.snapshot()
    env.step(torch.from_numpy(acts[0]).to(env.device))
    res["step"] = (_np(env.cells), _np(env.agent))
    env.restore(snap)
    E = take(S, np.arange(n))
    E["inv"] = np.zeros_like(E["inv"])
    for order in ("observe", "pipeline", "advance", "u8"):
        ep = VecCraft.from_instances(tables, E["grid"], np.arange(n), E["pos"], E["task"], max_timesteps=T_MAX)
        for t in range(4):
            fo = _poisoned((n, tables.n_features), torch.uint8 if order == "u8" else torch.float32, ep.device)
            o = ep.tick(actions=torch.from_numpy(acts[t]).to(ep.device), features_out=fo, fused=order != "pipeline",
                        advance_first=order == "advance")
            res[(order, t)] = (_np(o["expert"]), _np(o["done"]), _np(o["success"]), _np(fo))
        res[(order, "state")] = (_np(ep.cells), _np(ep.agent), _np(ep.stats))
    for u8 in (False, True):
        ep = VecCraft.from_instances(tables, E["grid"], np.arange(n), E["pos"], E["task"], max_timesteps=T_MAX)
        ring = _poisoned((2, n, tables.n_features), torch.uint8 if u8 else torch.float32, ep.device)
        o = ep.rollout(5, actions=torch.from_numpy(acts[:5]).to(ep.device), features_out=ring)
        res[("rollout", u8)] = (_np(o["expert"]), _np(o["done"]), _np(o["success"]), _np(ring), _np(ep.cells),
                                _np(ep.agent), _np(ep.stats))
    return res


def _forced_sets():
    import os
    from psketch_b200.tables import CraftTables
    here = os.path.dirname(os.path.abspath(__file__))
    out = []
    for name, cfg in (("craft_medium_states", "craft_medium"), ("craft_large_states", "craft_large")):
        d = np.load(os.path.join(here, "golden", name + ".npz"))
        tables = CraftTables(world_config=cfg)
        n = len(d["grid"])
        task = np.random.RandomState(1).choice(good_tasks(tables), size=n).astype(np.int32)
        out.append((name, tables, dict(grid=d["grid"], inv=d["inv"].astype(np.int32), pos=d["pos"].astype(np.int32),
                                       dir=d["dir"].astype(np.int32), task=task)))
    for size in (16, 32, 64):
        for bk in (("stock", "custom") if size == 16 else ("stock",)):
            S = all_families(size, bk)
            out.append(("stress%d_%s" % (size, bk), stress_tables(size, bk), {k: np.asarray(S[k]) for k in KEYS}))
    return out


@pytest.mark.parametrize("case", range(6))
def test_forced_generic_matches_specialised(case):
    name, tables, S = _forced_sets()[case]
    S = {k: (v.astype(np.int32) if k != "grid" else v) for k, v in S.items()}
    S["inv"] = np.minimum(S["inv"], 250)
    acts = np.random.RandomState(case).choice(6, size=(5, len(S["grid"]))).astype(np.uint8)
    with tuning(generic=-1):
        want = _all_outputs(tables, S, acts)
    with tuning(generic=1):
        got = _all_outputs(tables, S, acts)
    assert want.keys() == got.keys()
    for k in want:
        w, g = want[k], got[k]
        w, g = (w if isinstance(w, tuple) else (w,)), (g if isinstance(g, tuple) else (g,))
        for i, (a, b) in enumerate(zip(w, g)):
            assert a.dtype == b.dtype and np.array_equal(a, b), (name, k, i)


# ------------------------------------------------------------------------------------------------
# object API, teacher rollouts, guard bands

def test_craft_world_from_a_world_yaml(tmp_path, monkeypatch):
    """CraftWorld(config) with configs/worlds/<name>.yaml of a 20x13 world with a 3x5 window: the
    reference's object API on the generic tier."""
    from psketch_b200.teachers.demonstration import DemonstrationTeacher
    from psketch_b200.worlds.craft import CraftWorld
    (tmp_path / "configs" / "worlds").mkdir(parents=True)
    (tmp_path / "configs" / "worlds" / "wide.yaml").write_text(
        "WIDTH: 20\nHEIGHT: 13\nWINDOW_WIDTH: 3\nWINDOW_HEIGHT: 5\nN_WORKSHOPS: 3\nN_PRIMITIVES: 4\nN_WORLDS: 10\n")
    monkeypatch.chdir(tmp_path)

    class _Cfg(object):
        pass

    c = _Cfg()
    c.recipes = None
    c.world = _Cfg()
    c.world.config = "wide"
    c.trainer = _Cfg()
    c.trainer.hints = None
    world = CraftWorld(c)
    tables = world.tables
    assert (tables.W, tables.H, tables.win_w, tables.win_h) == (20, 13, 3, 5)
    assert world.n_features == 2 * 15 * tables.K + tables.K + 5
    o = _oracle(tables)
    S = take(episode_states(tables, 5), np.arange(40))
    K = tables.K
    teacher = DemonstrationTeacher()
    tm = tables.task_manager
    for i in range(len(S["grid"])):
        ids = S["grid"][i].reshape(20, 13)
        onehot = np.zeros((20, 13, K))
        xs, ys = np.nonzero(ids)
        onehot[xs, ys, ids[xs, ys]] = 1
        s = world.init_state(onehot, tuple(int(v) for v in S["pos"][i]))
        g, inv, pos, d = S["grid"][i:i + 1], np.zeros((1, K), np.int32), S["pos"][i:i + 1], np.zeros(1, np.int32)
        task = tm.by_id(int(S["task"][i]))
        for a in (1, 3, 4, 0, 2, 4):
            assert np.array_equal(s.features(), o.features(g, inv, pos, d)[0].astype(np.float64)), i
            sat = o.satisfies(g, inv, pos, d, S["task"][i:i + 1])[0]
            assert s.satisfies(task) == (None if sat == 2 else bool(sat)), i
            assert teacher(task, s) == o.expert(g, inv, pos, d, S["task"][i:i + 1])[0][0], i
            _, s = s.step(a)
            g, inv, pos, d, _ = o.step(g, inv, pos, d, np.array([a]))
            assert tuple(s.pos) == tuple(pos[0]) and s.dir == d[0], i
            assert np.array_equal(np.asarray(s.inventory), inv[0]), i


@pytest.mark.parametrize("geometry", [(9, 9, 3, 3), (33, 17, 5, 5)], ids=["9x9_w3x3", "33x17_w5x5"])
def test_teacher_rollouts(geometry):
    """teacher_rollouts at a new geometry: every episode ends in STOP, `satisfied` is the oracle's
    success flag of that episode (most get-tasks succeed), and the actions are the oracle's, tick by
    tick."""
    from psketch_b200.rollout import teacher_rollouts
    from psketch_b200.vec import VecCraft
    tables = generic_tables(*geometry)
    o = _oracle(tables)
    E = random_states(tables, 200, 21)
    n = len(E["grid"])
    get_tasks = [t.task_id for t in tables.task_manager.tasks if t.goal_name == "get"]
    task = np.random.RandomState(2).choice(get_tasks, size=n).astype(np.int32)
    T = 200
    env = VecCraft.from_instances(tables, E["grid"], np.arange(n), E["pos"], task, max_timesteps=T)
    acts, length, ok = teacher_rollouts(env, max_len=T)
    ref = _OracleTicks(o, E["grid"], E["pos"], task, T)
    first = np.full(n, -1)
    succ = np.zeros(n, bool)
    for t in range(int(length.max())):
        g = ref.tick()
        new = (g["done"] == 1) & (first < 0)
        first[new], succ[new] = t, g["success"][new] == 1
        live = t < length
        assert np.array_equal(acts[live, t], g["expert"][live]), t
    assert np.array_equal(length, first + 1)
    assert (acts[np.arange(n), length - 1] == 5).all()
    assert np.array_equal(ok, succ) and ok.mean() > 0.5


def test_guard_bands():
    """Every buffer of every generic entry point sits between 4 KB canaries: state rows, agent records,
    feature frames (f32, u8), teacher actions / distances, find_closest goal / length / sequences,
    satisfies, tick flags."""
    from psketch_b200 import _lib
    from psketch_b200.vec import VecCraft
    G = 4096
    for geometry in ((20, 13, 3, 5), (64, 64, 9, 9), (2, 9, 3, 1)):
        tables = generic_tables(*geometry)
        S = episode_states(tables, 31)
        S = take(S, np.arange(min(101, len(S["grid"]))))
        n, nf = len(S["grid"]), tables.n_features
        env = VecCraft.from_instances(tables, S["grid"], np.arange(n), S["pos"], S["task"], max_timesteps=T_MAX)
        dev = env.device

        def guarded(nbytes):
            t = torch.full((G + nbytes + G,), 0x5A, dtype=torch.uint8, device=dev)
            return t, t[G:G + nbytes]

        bufs = {}
        for name, nbytes in (("grid", n * env.cell_stride), ("agent", n * 32), ("f32", n * nf * 4), ("u8", n * nf),
                             ("act", n), ("dist", 2 * n), ("goal", 2 * n), ("len", 2 * n), ("seq", 37 * n),
                             ("sat", n), ("done", n), ("succ", n)):
            bufs[name] = guarded(nbytes)
        bufs["grid"][1].copy_(env.grid.view(-1))
        bufs["agent"][1].copy_(env.agent.view(-1))
        st = _lib.CraftStateC(bufs["grid"][1].data_ptr(), bufs["agent"][1].data_ptr(), n, env.cell_stride, 0)
        ct, s = ctypes.byref(env.ct), env._stream()
        lib = env.lib
        P = lambda k: ctypes.c_void_p(bufs[k][1].data_ptr())                                    # noqa: E731
        kind = env._u8(np.full(n, go_kinds(tables)[0]))
        acts = env._u8(np.random.RandomState(1).randint(0, 6, n))
        with torch.cuda.device(dev):
            assert lib.psk_craft_expert(ct, st, None, P("act"), P("dist"), _p(env.err_flags), s) == 0
            assert lib.psk_craft_find_closest(ct, st, _p(kind), P("goal"), P("len"), P("seq"), 37, s) == 0
            assert lib.psk_craft_satisfies(ct, st, None, P("sat"), s) == 0
            assert lib.psk_craft_features(ct, st, P("f32"), 0, s) == 0
            assert lib.psk_craft_features_u8(ct, st, P("u8"), s) == 0
            assert lib.psk_craft_step(ct, st, _p(acts), None, None, _p(env.err_flags), s) == 0
            for order in (1, 0, 2):
                assert lib.psk_craft_tick(ct, st, env._episodes(), _p(acts), P("f32"), P("act"), P("done"),
                                          P("succ"), _p(env.stats), _p(env.err_flags), order, s) == 0
                assert lib.psk_craft_tick_u8(ct, st, env._episodes(), _p(acts), P("u8"), P("act"), P("done"),
                                             P("succ"), _p(env.stats), _p(env.err_flags), order or 1, s) == 0
        torch.cuda.synchronize()
        for name, (whole, _) in bufs.items():
            w = _np(whole)
            assert (w[:G] == 0x5A).all() and (w[-G:] == 0x5A).all(), (geometry, name)
