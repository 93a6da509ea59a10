"""Every Craft entry point at 16x16, 32x32 and 64x64 (BASELINE configs[4]) on the edge families of
tests/test_stress_states_cpu.py, stock and custom cookbook (20 kinds: the runtime-K feature
kernels), compared exactly with the C oracle (oracle/craft_oracle.py):

  - the teacher on leaf pairs inside one warp, odd and even batch sizes, and past one wave of the
    grid-stride loops (the wave is taken from the device's SM count);
  - find_closest for every go-kind: length, goal (the last goal cell when none is reachable,
    255/255 when the kind is absent), the action sequence at several caps and the 255 fill;
  - satisfies, step (all actions, invalid bytes, both step variants, past one wave), features
    (impl 0 and 2, bytes);
  - the tick (both orders, f32 and byte frames), the rollout with a ring shorter than the rollout,
    and HostCraft, replayed tick by tick with teacher and random actions through auto-resets.

Every output buffer is poisoned before the call, so a row the kernel never wrote cannot match."""
import contextlib
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from test_edge_states_cpu import step_u8                        # noqa: E402
from test_stress_states_cpu import (BOOKS, SIZES, all_families, concat, family, go_kinds,  # noqa: E402
                                    good_tasks, stress_oracle, stress_tables, take)

pytestmark = pytest.mark.gpu

POISON = 0xA5


@contextlib.contextmanager
def tuning(**knobs):
    from psketch_b200 import _lib
    old = _lib.set_tuning(**knobs)
    try:
        yield
    finally:
        _lib.set_tuning(**old)


def _np(t):
    return t.cpu().numpy()


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _env(tables, S, T=40):
    from psketch_b200.vec import VecCraft
    return VecCraft.from_states(tables, S["grid"], S["inv"], S["pos"], S["dir"], task=S["task"], max_timesteps=T)


def _poisoned(shape, dtype, dev):
    t = torch.empty(shape, dtype=dtype, device=dev)
    if dtype == torch.float32:
        t.fill_(-7.0)
    elif dtype == torch.int16:
        t.fill_(-12345)
    else:
        t.fill_(POISON)
    return t


def run_expert(env, task=None):
    """psk_craft_expert into poisoned buffers: (action i32, dist i32)."""
    act = _poisoned(env.n, torch.uint8, env.device)
    dist = _poisoned(env.n, torch.int16, env.device)
    with torch.cuda.device(env.device):
        rc = env.lib.psk_craft_expert(ctypes.byref(env.ct), env._state(), _p(env._u8(task)), _p(act), _p(dist),
                                      _p(env.err_flags), env._stream())
    assert rc == 0
    return _np(act).astype(np.int32), _np(dist).astype(np.int32)


def run_find_closest(env, kind, seq_cap):
    goal = _poisoned((env.n, 2), torch.uint8, env.device)
    length = _poisoned(env.n, torch.int16, env.device)
    seq = _poisoned((env.n, seq_cap), torch.uint8, env.device) if seq_cap else None
    with torch.cuda.device(env.device):
        rc = env.lib.psk_craft_find_closest(ctypes.byref(env.ct), env._state(), _p(env._u8(kind)), _p(goal),
                                            _p(length), _p(seq), int(seq_cap), env._stream())
    assert rc == 0
    return _np(goal).astype(np.int32), _np(length).astype(np.int32), None if seq is None else _np(seq)


def check_expert(tables, oracle, S, tag):
    """Teacher action and distance, task from the agent record and from an explicit array."""
    want_a, want_d, _ = oracle.expert(S["grid"], S["inv"], S["pos"], S["dir"], S["task"])
    env = _env(tables, S)
    for task in (None, S["task"]):
        a, d = run_expert(env, task)
        assert np.array_equal(a, want_a), (tag, np.flatnonzero(a != want_a)[:8])
        assert np.array_equal(d, want_d), (tag, np.flatnonzero(d != want_d)[:8])
        env.check_errors()
    return want_a, want_d


@pytest.fixture(params=BOOKS)
def book(request):
    return request.param


@pytest.fixture(params=SIZES)
def size(request):
    return request.param


# ------------------------------------------------------------------------------------------------
# teacher

def test_expert_on_every_family_and_leaf_pair(size, book):
    """Every family; the paired leaf batch (envs 2i / 2i+1 share a warp at 16x16) whole and cut to
    n = 1, 2, 3 and to odd and even lengths, and with every pair in the other order and shifted by one
    env, so that each case also meets the other cases across a warp's two halves the other way."""
    tables, o = stress_tables(size, book), stress_oracle(size, book)
    S = all_families(size, book)
    a, d = check_expert(tables, o, S, "all")
    assert d.max() > {16: 60, 32: 255, 64: 1000}[size] and (a == 4).any() and (a == 5).any()
    L = family(size, book, "leaf")
    n = len(L["grid"])
    for m in (1, 2, 3, n - 1, n, n - 3):
        check_expert(tables, o, take(L, np.arange(m)), ("leaf", m))
    rev = np.arange(n).reshape(-1, 2)[:, ::-1].reshape(-1)          # every pair in the other order
    check_expert(tables, o, take(L, rev[1:]), "leaf shifted by one")


def _wave_batch(size, book, n, seed):
    """n envs drawn (a seeded permutation, tiled) from every family, so that no two neighbours of a
    warp or of a grid-stride pass are copies of each other."""
    S = all_families(size, book)
    m = len(S["grid"])
    rng = np.random.RandomState(seed)
    idx = np.concatenate([rng.permutation(m) for _ in range(-(-n // m))])[:n]
    return take(S, idx)


def test_expert_and_find_closest_past_one_wave(size, book):
    """The grid-stride loops of the warp-per-env kernels (4 warps x 16 CTAs per SM) and of the
    two-envs-per-warp kernel (twice as many envs per pass) run a second and third pass."""
    sms = _sms()
    wave = sms * 16 * 4
    n = {16: 2 * (2 * wave) + 1, 32: 2 * wave + 3, 64: wave + 5}[size]
    tables, o = stress_tables(size, book), stress_oracle(size, book)
    S = _wave_batch(size, book, n, seed=size)
    check_expert(tables, o, S, ("wave", n))
    env = _env(tables, S)
    kind = np.where(S["target"] > 0, S["target"], go_kinds(tables)[0]).astype(np.int32)
    g, ln, _ = run_find_closest(env, kind, 0)
    og, ol, st, _ = o.find_closest(S["grid"], S["pos"], S["dir"], kind, seq_cap=0)
    ok = st != 2
    assert np.array_equal(ln[ok], ol[ok])
    assert np.array_equal(g[ok], np.where(og < 0, 255, og)[ok])


# ------------------------------------------------------------------------------------------------
# find_closest

def _check_closest(env, o, S, kind, cap, tag):
    g, ln, seq = run_find_closest(env, kind, cap)
    og, ol, st, oseq = o.find_closest(S["grid"], S["pos"], S["dir"], kind, seq_cap=cap)
    ok = st != 2                            # status 2: the reference raised TypeError
    assert np.array_equal(ln[ok], ol[ok]), (tag, np.flatnonzero(ln[ok] != ol[ok])[:8])
    assert np.array_equal(g[ok], np.where(og < 0, 255, og)[ok]), tag
    if cap:
        assert np.array_equal(seq[ok], oseq[ok]), tag
    return ol, st, og


def test_find_closest_every_kind_and_cap(size, book):
    tables, o = stress_tables(size, book), stress_oracle(size, book)
    S = concat([family(size, book, f) for f in ("random", "open", "ringless", "leaf", "inventory")])
    env = _env(tables, S)
    n = len(S["grid"])
    seen = dict(unreachable=0, absent=0, facing=0)
    for k in go_kinds(tables):
        ol, st, og = _check_closest(env, o, S, np.full(n, k, np.int32), 0, ("kind", k))
        seen["absent"] += int(((og[:, 0] < 0) & (st == 1)).sum())
        seen["unreachable"] += int(((og[:, 0] >= 0) & (st == 1)).sum())
        seen["facing"] += int((ol == 0).sum())
    assert min(seen.values()) > 0, seen
    # sequences towards each env's own target, capped below, at and above path lengths
    kind = np.where(S["target"] > 0, S["target"], go_kinds(tables)[0]).astype(np.int32)
    ol, _, _ = _check_closest(env, o, S, kind, 0, "target")
    L = int(np.median(ol[ol > 0]))
    for cap in sorted({0, 1, 31, 33, L - 1, L, L + 1, int(ol.max()) + 1}):
        _check_closest(env, o, S, kind, cap, ("cap", cap))
    # the mazes: sequences of hundreds / thousands of actions
    M = family(size, book, "maze")
    envm = _env(tables, M)
    ol, _, _ = _check_closest(envm, o, M, M["target"], 0, "maze")
    Lm = int(ol.max())
    assert Lm > {16: 60, 32: 255, 64: 1000}[size]
    for cap in (33, Lm, Lm + 1):
        _check_closest(envm, o, M, M["target"], cap, ("maze cap", cap))


# ------------------------------------------------------------------------------------------------
# satisfies, step, features

def test_satisfies_every_task(size, book):
    tables, o = stress_tables(size, book), stress_oracle(size, book)
    S = all_families(size, book)
    env = _env(tables, S)
    n = len(S["grid"])
    for t in range(1, tables.n_tasks):
        out = _poisoned(n, torch.uint8, env.device)
        tk = torch.full((n,), t, dtype=torch.uint8, device=env.device)
        with torch.cuda.device(env.device):
            assert env.lib.psk_craft_satisfies(ctypes.byref(env.ct), env._state(), _p(tk), _p(out), env._stream()) == 0
        want = o.satisfies(S["grid"], S["inv"], S["pos"], S["dir"], np.full(n, t))
        assert np.array_equal(_np(out).astype(np.int32), want), t


BAD_BYTES = (6, 7, 100, 254, 255)


def _check_step(tables, S, act, tag):
    """One psk_craft_step of `act` on S in every step variant: next state as step_u8 (the oracle's
    step with the u8 inventory rule); envs with an invalid byte keep their state, and the batch raises
    'Unexpected action' (or OverflowError when only a count overflowed)."""
    bad = act > 5
    g, iv, p, d, over, _ = step_u8(tables, S["grid"], S["inv"], S["pos"], S["dir"], np.where(bad, 5, act))
    env = _env(tables, S)
    snap = env.snapshot()
    for sv in (0, 1, 2):
        with tuning(step_variant=sv):
            env.restore(snap)
            env.step(torch.from_numpy(act.astype(np.uint8)).to(env.device))
            assert np.array_equal(_np(env.cells), g), (tag, sv)
            assert np.array_equal(_np(env.inventory).astype(np.int32), iv), (tag, sv)
            assert np.array_equal(_np(env.pos).astype(np.int32), p), (tag, sv)
            assert np.array_equal(_np(env.dir).astype(np.int32), d), (tag, sv)
            if bad.any():
                with pytest.raises(Exception, match="Unexpected action"):
                    env.check_errors()
            elif over.any():
                with pytest.raises(OverflowError):
                    env.check_errors()
            else:
                env.check_errors()


def test_step_every_action(size, book):
    tables = stress_tables(size, book)
    S = all_families(size, book)
    n = len(S["grid"])
    for a in range(6):
        _check_step(tables, S, np.full(n, a), ("action", a))
    rng = np.random.RandomState(size)
    mixed = rng.choice(list(range(6)) + list(BAD_BYTES), size=n)
    _check_step(tables, S, mixed, "mixed with invalid bytes")
    for b in BAD_BYTES:
        _check_step(tables, take(S, np.arange(5)), np.full(5, b), ("bad", b))
    # the grid-stride loop of the step kernel: 256-thread CTAs x 8 per SM (variant 0) and 64 x 32
    if size == 16 and book == "stock":
        o = stress_oracle(size, book)
        N = _sms() * 8 * 256 + 7
        W = _wave_batch(size, book, N, seed=5)
        W["inv"] = np.minimum(W["inv"], 200)       # no overflow: the oracle's step is the answer
        act = rng.randint(0, 6, size=N)
        env = _env(tables, W)
        snap = env.snapshot()
        g, iv, p, d, _ = o.step(W["grid"], W["inv"], W["pos"], W["dir"], act)
        for sv in (0, 1):
            with tuning(step_variant=sv):
                env.restore(snap)
                env.step(torch.from_numpy(act.astype(np.uint8)).to(env.device))
                env.check_errors()
                assert np.array_equal(_np(env.cells), g) and np.array_equal(_np(env.inventory).astype(np.int32), iv), sv
                assert np.array_equal(_np(env.pos).astype(np.int32), p) and np.array_equal(_np(env.dir).astype(np.int32), d), sv


def test_features_every_family(size, book):
    """impl 0 (vector store), impl 2 (TMA store) and the byte rows on every family; the ringless
    family puts the 9x9 window off the grid on every side."""
    tables, o = stress_tables(size, book), stress_oracle(size, book)
    for f in ("ringless", "random", "maze", "open", "leaf", "inventory"):
        S = family(size, book, f)
        env = _env(tables, S)
        want = o.features(S["grid"], S["inv"], S["pos"], S["dir"])
        for impl in (0, 2):
            out = _poisoned((env.n, tables.n_features), torch.float32, env.device)
            env.features(out=out, impl=impl)
            assert np.array_equal(_np(out), want), (f, impl)
        out = _poisoned((env.n, tables.n_features), torch.uint8, env.device)
        env.features_u8(out=out)
        assert np.array_equal(_np(out).astype(np.float32), want), (f, "u8")


# ------------------------------------------------------------------------------------------------
# multi-tick paths, replayed against the oracle

class _OracleTicks(object):
    """The rollout loop body of trainers/imitation.py:42-73 (with auto-reset) on the CPU oracle, one
    tick at a time, with the per-env done / success flags the kernels also report."""

    def __init__(self, oracle, grids, ipos, itask, max_timesteps):
        self.o, self.T = oracle, max_timesteps
        n = len(grids)
        self.init_grid = np.ascontiguousarray(grids)
        self.init_pos = np.asarray(ipos).astype(np.int32)
        self.task = np.asarray(itask).astype(np.int32)
        self.grid = self.init_grid.copy()
        self.inv = np.zeros((n, oracle.K), np.int32)
        self.pos = self.init_pos.copy()
        self.dir = np.zeros(n, np.int32)
        self.timer = np.full(n, max_timesteps, np.int32)
        self.stats = np.zeros(3, np.int64)

    def tick(self, actions=None):
        o = self.o
        expert, _, _ = o.expert(self.grid, self.inv, self.pos, self.dir, self.task)
        feats = o.features(self.grid, self.inv, self.pos, self.dir)
        act = expert if actions is None else np.asarray(actions).astype(np.int32)
        self.timer -= 1
        done = (act == 5) | (self.timer <= 0)
        succ = done & (o.satisfies(self.grid, self.inv, self.pos, self.dir, self.task) == 1)
        g2, i2, p2, d2, _ = o.step(self.grid, self.inv, self.pos, self.dir, np.where(done, 5, act).astype(np.int32))
        self.grid = np.where(done[:, None], self.init_grid, g2)
        self.inv = np.where(done[:, None], 0, i2).astype(np.int32)
        self.pos = np.where(done[:, None], self.init_pos, p2).astype(np.int32)
        self.dir = np.where(done, 0, d2).astype(np.int32)
        self.timer = np.where(done, self.T, self.timer).astype(np.int32)
        self.stats += (int(done.sum()), int(succ.sum()), len(done))
        return dict(expert=expert.astype(np.uint8), done=done.astype(np.uint8),
                    success=succ.astype(np.uint8), features=feats,
                    state=tuple(a.copy() for a in (self.grid, self.inv, self.pos, self.dir, self.timer)))

    @staticmethod
    def state_equals(grid, agent, K, state):
        """A device state (cells, agent records) against a state returned by tick()."""
        g, inv, pos, d, timer = state
        return (np.array_equal(grid, g) and np.array_equal(agent[:, :K].astype(np.int32), inv)
                and np.array_equal(agent[:, 24:26].astype(np.int32), pos)
                and np.array_equal(agent[:, 26].astype(np.int32), d)
                and np.array_equal(agent[:, 28].astype(np.int32), timer))


TICKS, T_MAX = 9, 4


def _episodes(size, book, n=None):
    """Episode starts: every family but the inventory one (episodes start with nothing), tasks with
    a defined teacher answer, facing 0."""
    S = concat([family(size, book, f) for f in ("random", "open", "ringless", "leaf", "maze")])
    if n is not None:
        S = take(S, np.random.RandomState(n).permutation(len(S["grid"]))[:n])
    ok = np.isin(S["task"], good_tasks(stress_tables(size, book)))
    assert ok.all()
    return S


def _actions(n, seed):
    return np.random.RandomState(seed).choice(6, size=(TICKS, n), p=[.2, .2, .2, .2, .15, .05]).astype(np.uint8)


@pytest.mark.parametrize("driver", ["teacher", "random"])
def test_tick_replay_both_orders(size, book, driver):
    """psk_craft_tick (observe, then step; and step, then observe), f32 and byte frames, and the
    three-kernel pipeline: every tick's outputs, then the final state and the counters."""
    from psketch_b200.vec import VecCraft
    tables, o = stress_tables(size, book), stress_oracle(size, book)
    S = _episodes(size, book)
    n, nf, K = len(S["grid"]), tables.n_features, tables.K
    acts = None if driver == "teacher" else _actions(n, size)
    ref = _OracleTicks(o, S["grid"], S["pos"], S["task"], T_MAX)
    gold = [ref.tick(None if acts is None else acts[t]) for t in range(TICKS)]
    assert sum(int(g["done"].sum()) for g in gold) > n // 4          # auto-resets happen
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

        if adv:                     # the first observation, no step; then step t and observe t + 1
            call(None)
            observed(0, (mode, driver, "start"))
            assert not _np(out["done"]).any() and not _np(out["success"]).any()
        steps = TICKS - 1 if adv else TICKS
        for t in range(steps):
            tag = (mode, driver, t)
            a = acts[t] if acts is not None else (gold[t]["expert"] if adv else None)
            call(a)
            assert np.array_equal(_np(out["done"]), gold[t]["done"]), tag
            assert np.array_equal(_np(out["success"]), gold[t]["success"]), tag
            observed(t + 1 if adv else t, tag)
        env.check_errors()
        assert ref.state_equals(_np(env.cells), _np(env.agent), K, gold[steps - 1]["state"]), mode
        want = np.sum([(int(g["done"].sum()), int(g["success"].sum()), n) for g in gold[:steps]], axis=0)
        assert tuple(_np(env.stats)[:3]) == tuple(want), mode


@pytest.mark.parametrize("driver", ["teacher", "random"])
def test_rollout_replay(size, book, driver):
    """psk_craft_rollout and _rollout_u8 at these sizes: T = 5 ticks in one call, a 2-frame feature
    ring, teacher-driven or with an action block; every tick, the ring, the final state, the stats."""
    from psketch_b200.vec import VecCraft
    tables, o = stress_tables(size, book), stress_oracle(size, book)
    S = _episodes(size, book)
    n, nf, Tk, R = len(S["grid"]), tables.n_features, 5, 2
    acts = None if driver == "teacher" else _actions(n, size + 1)[:Tk]
    ref = _OracleTicks(o, S["grid"], S["pos"], S["task"], T_MAX)
    gold = [ref.tick(None if acts is None else acts[t]) for t in range(Tk)]
    for u8 in (False, True):
        env = VecCraft.from_instances(tables, S["grid"], np.arange(n), S["pos"], S["task"], max_timesteps=T_MAX)
        ring = _poisoned((R, n, nf), torch.uint8 if u8 else torch.float32, env.device)
        out = {k: _poisoned((Tk, n), torch.uint8, env.device) for k in ("expert", "done", "success")}
        env.rollout(Tk, actions=None if acts is None else torch.from_numpy(acts).cuda(), features_out=ring, out=out)
        tag = (driver, u8)
        for t in range(Tk):
            for k in ("expert", "done", "success"):
                assert np.array_equal(_np(out[k][t]), gold[t][k]), (tag, t, k)
        for t in (Tk - 2, Tk - 1):
            assert np.array_equal(_np(ring[t % R]).astype(np.float32), gold[t]["features"]), (tag, t)
        env.check_errors()
        assert ref.state_equals(_np(env.cells), _np(env.agent), tables.K, gold[-1]["state"]), tag
        assert tuple(_np(env.stats)[:3]) == tuple(ref.stats), tag


@pytest.mark.parametrize("size", [16, 32])
def test_host_paths(size, book):
    """HostCraft with a chunk size that does not divide n: tick (state round trip) and tick_resident
    with every feature format, observe-then-step and step-then-observe; host frames poisoned first."""
    from psketch_b200.host import HostCraft
    tables, o = stress_tables(size, book), stress_oracle(size, book)
    n = 1000
    S = _episodes(size, book, n=n)
    K, C = tables.K, tables.W * tables.H
    acts = _actions(n, 3)
    ref = _OracleTicks(o, S["grid"], S["pos"], S["task"], T_MAX)
    gold = [ref.tick(acts[t]) for t in range(6)]
    for mode in ("tick", None, "f32", "u8", "f32_wire_u8", "advance f32", "advance u8", "advance f32_wire_u8",
                 "advance None"):
        h = HostCraft(tables, S["grid"], np.arange(n), S["pos"], S["task"], max_timesteps=T_MAX, chunk_envs=384,
                      host_threads=2)
        adv = mode is not None and mode.startswith("advance")
        fmt = mode.split()[1] if adv else mode
        fmt = None if fmt == "None" else fmt

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
            if fmt is not None:
                f = h.features_u8.astype(np.float32) if fmt == "u8" else h.features
                assert np.array_equal(f, gold[t]["features"]), tag

        if adv:
            h.upload()
            call(None)
            observed(0, (size, mode, "start"))
        steps = 5 if adv else 6
        for t in range(steps):
            tag = (size, mode, t)
            call(acts[t])
            assert np.array_equal(h.done, gold[t]["done"]) and np.array_equal(h.success, gold[t]["success"]), tag
            observed(t + 1 if adv else t, tag)
        if mode != "tick":
            h.download(keep_resident=False)
        assert ref.state_equals(h.grid[:, :C], h.agent, K, gold[steps - 1]["state"]), mode
        want = np.sum([(int(g["done"].sum()), int(g["success"].sum()), n) for g in gold[:steps]], axis=0)
        assert tuple(h.stats[:3].astype(np.int64)) == tuple(want), mode
        h.close()


def test_sampler_rejects_enlarged_grids(size):
    """The scenario sampler is built for 8x8 and 10x10 only: other sizes raise, nothing is returned."""
    from psketch_b200 import _lib, data
    with pytest.raises(_lib.PskError):
        data.sample_scenarios(stress_tables(size), 16, seed=1)
