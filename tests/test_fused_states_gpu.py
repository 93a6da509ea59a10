"""The kernels that do the work — the fused tick (every CTA shape, store path, persistent grid and
launch mode), its byte-frame form, the multi-tick rollout and the host-buffer paths — on the states
exported from the reference (tests/golden/craft_*_states.npz: water, stone, bridge and axe in the
inventory, all four facings, answers for every task) and at the u8 inventory limit.

Expected values come straight from the golden arrays where the reference answered (features, step
results for every action, satisfies, teacher action) and from the C oracle elsewhere (the teacher
where the reference raised TypeError, observations after a step, multi-tick rollouts, counts above
12 — tests/test_edge_states_cpu.py pins the oracle against the reference's code there).  Every
comparison is exact and runs on the device."""
import contextlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from test_craft_gpu import ERR_TYPE, ROLLOUT_VARIANTS           # noqa: E402
from test_edge_states_cpu import edge_states, step_u8           # noqa: E402

pytestmark = pytest.mark.gpu

AG_TASK, AG_TIMER = 27, 28
TICK_SHAPES = {0: "64+2", 1: "128+4", 2: "32+1", 3: "64+4", 4: "32+2"}
MIN_ENVS = 160000        # persistent grids loop over super-tiles above ~148 x per_sm x NE envs


@contextlib.contextmanager
def tuning(**knobs):
    from psketch_b200 import _lib
    old = _lib.set_tuning(**knobs)
    try:
        yield
    finally:
        _lib.set_tuning(**old)


_ARRAYS = {}


def _arrays(S):
    """npz members are re-read on every access: load each fixture once."""
    key = id(S)
    if key not in _ARRAYS:
        _ARRAYS[key] = {k: S[k] for k in S.files}
    return _ARRAYS[key]


class Ref(object):
    """n (state, task) pairs of exported states, each env starting over at a DIFFERENT exported
    state (a permutation) with its own task, and the expected outcome of one tick for any action."""

    def __init__(self, tables, oracle, S, ii, tt, T=40, seed=0):
        S = _arrays(S)
        self.tables, self.oracle, self.S = tables, oracle, S
        self.n = n = len(ii)
        self.ii, self.tt, self.T = ii, tt.astype(np.int32), T
        self.C, self.K, self.cs = tables.W * tables.H, tables.K, ((tables.W * tables.H + 63) // 64) * 64
        self.perm = np.random.RandomState(seed).permutation(n)
        self.grid = S["grid"][ii]
        self.inv, self.pos, self.dir = S["inv"][ii], S["pos"][ii], S["dir"][ii]
        self.agent0 = self._agent(self.inv, self.pos, self.dir, T)
        self.init_agent = self.agent0[self.perm].copy()
        self.init_agent[:, AG_TASK] = self.tt
        golden = S["expert"][ii, tt]
        o_act, _, _ = oracle.expert(self.grid, self.inv.astype(np.int32), self.pos.astype(np.int32),
                                    self.dir.astype(np.int32), self.tt)
        ok = golden != ERR_TYPE
        assert np.array_equal(o_act[ok], golden[ok])
        self.expert = np.where(ok, golden, o_act).astype(np.uint8)   # TypeError: the oracle's answer
        self.feats = S["features"][ii]
        self.sat = S["satisfies"][ii, tt]
        self._dev = {}
        self._obs = {}

    def _agent(self, inv, pos, dirs, timer):
        a = np.zeros((len(inv), 32), np.uint8)
        a[:, :self.K] = inv
        a[:, 24:26] = pos
        a[:, 26] = dirs
        a[:, AG_TASK] = self.tt
        a[:, AG_TIMER] = timer
        return a

    def slots(self):
        """(name, action u8[n]): the teacher's action, then every action forced."""
        return [("teacher", self.expert)] + [("a%d" % a, np.full(self.n, a, np.uint8)) for a in range(6)]

    def after(self, act, timer=None):
        """State after one tick with `act` from a timer of `timer`: (grid u8[n, C], agent u8[n, 32],
        done, success)."""
        timer = self.T if timer is None else timer
        S, ii, act = self.S, self.ii, act.astype(np.int64)
        done = (act == 5) | (timer - 1 <= 0)
        succ = done & (self.sat == 1)
        grid = S["step_grid"][ii, act]
        agent = self._agent(S["step_inv"][ii, act], S["step_pos"][ii, act], S["step_dir"][ii, act], timer - 1)
        grid[done] = self.grid[self.perm][done]
        agent[done] = self.init_agent[done]
        return grid, agent, done.astype(np.uint8), succ.astype(np.uint8)

    def observed_after(self, name, act):
        """Teacher action and feature row (u8) of the state after the tick, from the oracle."""
        if name not in self._obs:
            g, a, _, _ = self.after(act)
            inv, pos, d = a[:, :self.K].astype(np.int32), a[:, 24:26].astype(np.int32), a[:, 26].astype(np.int32)
            e, _, _ = self.oracle.expert(g, inv, pos, d, self.tt)
            f = self.oracle.features(g, inv, pos, d)
            assert f.max() <= 255
            self._obs[name] = (e.astype(np.uint8), f.astype(np.uint8))
        return self._obs[name]

    def dev(self, key, make):
        """Device copy of a host array, uploaded once."""
        if key not in self._dev:
            self._dev[key] = torch.from_numpy(np.ascontiguousarray(make())).cuda()
        return self._dev[key]

    def make_env(self, lo=0, hi=None):
        """VecCraft over pairs [lo, hi) with the permuted episode starts."""
        from psketch_b200.vec import VecCraft
        hi = self.n if hi is None else hi
        sl = slice(lo, hi)
        env = VecCraft.from_states(self.tables, self.grid[sl], self.inv[sl], self.pos[sl], self.dir[sl],
                                   task=self.tt[sl], max_timesteps=self.T)
        scen = np.zeros((hi - lo, self.cs), np.uint8)
        scen[:, :self.C] = self.grid[self.perm][sl]
        env.scen_grid = torch.from_numpy(scen).to(env.device)
        env.init_agent = torch.from_numpy(self.init_agent[sl].copy()).to(env.device)
        return env


def _pairs(tables, oracle, S, min_envs=0, seed=0):
    """Every (state, task) pair whose teacher answer is defined (not the reference's assertion),
    tiled to at least min_envs."""
    S = _arrays(S)
    E = S["expert"]
    ii, tt = np.nonzero(E[:, 1:] != 255)
    tt = tt + 1
    o_act, _, _ = oracle.expert(S["grid"][ii], S["inv"][ii].astype(np.int32), S["pos"][ii].astype(np.int32),
                                S["dir"][ii].astype(np.int32), tt)
    keep = o_act != 255                    # TypeError states on which the oracle's walk asserts
    ii, tt = ii[keep], tt[keep]
    reps = max(1, -(-min_envs // len(ii)))
    return np.tile(ii, reps), np.tile(tt, reps)


_REFS = {}


def _ref(which, tables, oracle, S):
    if which not in _REFS:
        ii, tt = _pairs(tables, oracle, S, 0 if which == "medium" else MIN_ENVS)
        _REFS[which] = Ref(tables, oracle, S, ii, tt, seed={"medium": 1, "large": 2, "custom": 3}[which])
    return _REFS[which]


@pytest.fixture(params=["medium", "large", "custom"])
def ref(request, medium_tables, medium_oracle, medium_states, large_tables, large_oracle, large_states,
        custom_tables, custom_oracle, custom_states):
    w = request.param
    tables, oracle, S = {"medium": (medium_tables, medium_oracle, medium_states),
                         "large": (large_tables, large_oracle, large_states),
                         "custom": (custom_tables, custom_oracle, custom_states)}[w]
    R = _ref(w, tables, oracle, S)
    R.which = w
    return R


def _start(R, env, lo=0):
    """Device copies of the start state of pairs [lo, lo + env.n) in env's layout."""
    sl = slice(lo, lo + env.n)
    grid, agent = env.grid.clone(), env.agent.clone()
    grid[:, :R.C] = R.dev(("grid", lo, lo + env.n), lambda: R.grid[sl])
    agent.copy_(R.dev(("agent", lo, lo + env.n), lambda: R.agent0[sl]))
    return grid, agent


def check_one_tick(R, env, tag, fused=True, u8=False, orders=("observe", "advance"), timer1=True, lo=0):
    """Every slot (teacher action, forced 0..5) from the exported states, in the given tick orders,
    then the teacher's action with timer 1: outputs, next state, counters and flags."""
    n = env.n
    hi = lo + n
    sl = slice(lo, hi)
    nf = R.tables.n_features
    start_grid, start_agent = _start(R, env, lo)
    buf = torch.empty((n, nf), dtype=torch.uint8 if u8 else torch.float32, device=env.device)
    gold_f = R.dev(("feats", lo, hi), lambda: R.feats[sl])
    gold_e = R.dev(("expert", lo, hi), lambda: R.expert[sl])
    runs = [(o, name, act, R.T) for o in orders for name, act in R.slots()]
    if timer1:
        runs.append(("observe", "timer1", R.expert, 1))
    for order, name, act, timer in runs:
        t = "%s %s %s timer %d" % (tag, order, name, timer)
        env.grid.copy_(start_grid)
        env.agent.copy_(start_agent)
        if timer != R.T:
            env.agent[:, AG_TIMER] = timer
        env.stats.zero_()
        buf.fill_(77 if u8 else -1.0)
        adv = order == "advance"
        out = env.tick(actions=R.dev(("act", name, lo, hi), lambda: act[sl]), features_out=buf, fused=fused,
                       advance_first=adv)
        g, a, done, succ = R.after(act, timer)
        assert torch.equal(out["done"], R.dev(("done", name, timer, lo, hi), lambda: done[sl])), t
        assert torch.equal(out["success"], R.dev(("succ", name, timer, lo, hi), lambda: succ[sl])), t
        assert torch.equal(env.cells, R.dev(("g", name, timer, lo, hi), lambda: g[sl])), t
        assert torch.equal(env.agent, R.dev(("a", name, timer, lo, hi), lambda: a[sl])), t
        st = env.stats.tolist()
        assert st[:3] == [int(done[sl].sum()), int(succ[sl].sum()), n], t
        if adv:
            e_after, f_after = R.observed_after(name, act)
            want_e = R.dev(("e_after", name, lo, hi), lambda: e_after[sl])
            want_f = R.dev(("f_after", name, lo, hi), lambda: f_after[sl])
            raises = bool((e_after[sl] == 255).any())
        else:
            want_e, want_f, raises = gold_e, gold_f, False
        assert torch.equal(out["expert"], want_e), t
        assert torch.equal(buf, want_f if u8 else want_f.float()), t
        if raises:                                # the new state's teacher asserts (base.py:23-24)
            with pytest.raises(AssertionError):
                env.check_errors()
        else:
            env.check_errors()


# ------------------------------------------------------------------------------------------------
# A1: one tick against the reference's own answers

def test_fused_tick_every_variant(ref):
    """psk_craft_tick, fused: every CTA shape x store path x persistent grid (large: the one 64+2
    shape), tick_pdl=0, and the three-kernel pipeline."""
    R = ref
    env = R.make_env()
    variants = sorted(TICK_SHAPES) if R.which != "large" else [-1]
    for v in variants:
        for tma in (0, 1):
            for persist in (0, 1):
                with tuning(tick_variant=v, tick_tma=tma, tick_persist=persist):
                    check_one_tick(R, env, "%s variant %d tma %d persist %d" % (R.which, v, tma, persist))
    with tuning(tick_pdl=0):
        check_one_tick(R, env, "%s pdl 0" % R.which)
    check_one_tick(R, env, "%s pipeline" % R.which, fused=False, orders=("observe",))


def test_byte_frame_rollout_and_persistent_features(ref):
    """psk_craft_tick_u8 in both orders (both grid forms), psk_craft_rollout / _u8 with ticks = 1 over
    every rollout variant, and psk_craft_features with a persistent grid, impl 0, 1, 2."""
    R = ref
    env = R.make_env()
    for persist in (0, 1):
        with tuning(tick_persist=persist):
            check_one_tick(R, env, "%s u8 persist %d" % (R.which, persist), u8=True)
    nf, n = R.tables.n_features, R.n
    start_grid, start_agent = _start(R, env)
    gold_f, gold_e = R.dev(("feats", 0, n), lambda: R.feats), R.dev(("expert", 0, n), lambda: R.expert)
    variants = ROLLOUT_VARIANTS if R.which != "large" else [(-1, -1)]
    for variant, tma in variants:
        for u8 in (False, True):
            if u8 and (variant, tma) != (-1, -1):     # the byte frame has one CTA shape
                continue
            ring = torch.empty((1, n, nf), dtype=torch.uint8 if u8 else torch.float32, device=env.device)
            with tuning(rollout_variant=variant, rollout_tma=tma):
                for name, act in R.slots() + [("timer1", R.expert)]:
                    t = "%s rollout %d tma %d u8 %d %s" % (R.which, variant, tma, u8, name)
                    timer = 1 if name == "timer1" else R.T
                    env.grid.copy_(start_grid)
                    env.agent.copy_(start_agent)
                    env.agent[:, AG_TIMER] = timer
                    env.stats.zero_()
                    ring.fill_(77 if u8 else -1.0)
                    out = env.rollout(1, actions=R.dev(("act", name, 0, n), lambda: act)[None], features_out=ring)
                    g, a, done, succ = R.after(act, timer)
                    assert torch.equal(out["expert"][0], gold_e), t
                    assert torch.equal(ring[0], gold_f if u8 else gold_f.float()), t
                    assert torch.equal(out["done"][0], R.dev(("done", name, timer, 0, n), lambda: done)), t
                    assert torch.equal(out["success"][0], R.dev(("succ", name, timer, 0, n), lambda: succ)), t
                    assert torch.equal(env.cells, R.dev(("g", name, timer, 0, n), lambda: g)), t
                    assert torch.equal(env.agent, R.dev(("a", name, timer, 0, n), lambda: a)), t
                    assert env.stats.tolist()[:3] == [int(done.sum()), int(succ.sum()), n], t
                    env.check_errors()
    env.grid.copy_(start_grid)
    env.agent.copy_(start_agent)
    with tuning(feat_persist=1):
        for impl in (0, 1, 2):
            f = env.features(impl=impl)
            assert torch.equal(f, gold_f.float()), (R.which, "features impl", impl)
        assert torch.equal(env.features_u8(), gold_f), (R.which, "features_u8")


@pytest.mark.parametrize("n", [1, 33, 4099])
def test_ragged_slices_through_the_tick_variants(n, medium_tables, medium_oracle, medium_states):
    R = _ref("medium", medium_tables, medium_oracle, medium_states)
    lo = 1000
    env = R.make_env(lo, lo + n)
    for v in sorted(TICK_SHAPES):
        for tma in (0, 1):
            with tuning(tick_variant=v, tick_tma=tma):
                check_one_tick(R, env, "n %d variant %d tma %d" % (n, v, tma), lo=lo, timer1=False)
    check_one_tick(R, env, "n %d u8" % n, u8=True, lo=lo, timer1=False)


def _host_ref(medium_tables, medium_oracle, medium_states, n, N=10000, seed=5):
    """The first n of a 10,000-state slice of the medium states, one task per state (seeded) among
    those whose teacher answer is defined."""
    S = _arrays(medium_states)
    rng = np.random.RandomState(seed)
    ii = np.arange(N)
    ok = S["expert"][ii, 1:] != 255
    tt = np.array([rng.choice(np.nonzero(row)[0]) + 1 for row in ok])
    o_act, _, _ = medium_oracle.expert(S["grid"][ii], S["inv"][ii].astype(np.int32), S["pos"][ii].astype(np.int32),
                                       S["dir"][ii].astype(np.int32), tt)
    keep = np.nonzero(o_act != 255)[0][:n]
    return Ref(medium_tables, medium_oracle, medium_states, ii[keep], tt[keep], seed=seed)


@pytest.mark.parametrize("n", [10000, 2000])
def test_host_paths_on_exported_states(n, medium_tables, medium_oracle, medium_states):
    """psk_craft_host_tick with the state in the pinned arrays, and upload() + tick_resident in every
    feature format and both orders; 10,000 envs take the copy route, 2,000 the zero-copy route."""
    import ctypes
    from psketch_b200.host import HostCraft
    R = _host_ref(medium_tables, medium_oracle, medium_states, n)
    n, o, K = R.n, medium_oracle, R.K
    env = HostCraft(R.tables, R.grid, np.arange(n), R.pos, R.tt, max_timesteps=R.T, chunk_envs=1024, host_threads=2)
    scen = np.zeros((n, R.cs), np.uint8)
    scen[:, :R.C] = R.grid[R.perm]
    ptr = lambda a: ctypes.c_void_p(a.ctypes.data)
    idx = np.arange(n, dtype=np.int32)
    assert env.lib.psk_craft_host_set_episodes(env.ctx, ptr(scen), n, ptr(idx), ptr(R.init_agent), n) == 0
    for name, act in R.slots() + [("timer1", R.expert)]:
        timer = 1 if name == "timer1" else R.T
        g, ag, done, succ = R.after(act, timer)
        inv, pos, dd = ag[:, :K].astype(np.int32), ag[:, 24:26].astype(np.int32), ag[:, 26].astype(np.int32)
        for mode in ("tick", "f32", "u8", "f32_wire_u8", None, "advance"):
            t = (n, name, mode)
            env.grid[:, :R.C] = R.grid
            env.agent[:] = R.agent0
            env.agent[:, AG_TIMER] = timer
            env.expert[:] = 77
            env.done[:] = 77
            env.features[:] = -1.0
            before = env.stats.copy()
            want_e, want_f = R.expert, R.feats.astype(np.float32)
            if mode == "advance":
                want_e = o.expert(g, inv, pos, dd, R.tt)[0].astype(np.uint8)
                want_f = o.features(g, inv, pos, dd)
            raises = pytest.raises(AssertionError) if (want_e == 255).any() else contextlib.nullcontext()
            a = act.copy()
            with raises:
                if mode == "tick":
                    env.tick(actions=a)
                else:
                    env.upload()
                    fmt = "f32" if mode == "advance" else mode
                    if fmt == "u8":
                        env.features_u8[:] = 77
                    env.tick_resident(actions=a, features=fmt, advance_first=mode == "advance")
            if mode != "tick":
                env.download(keep_resident=False)
            assert np.array_equal(env.done, done) and np.array_equal(env.success, succ), t
            assert np.array_equal(env.grid[:, :R.C], g) and np.array_equal(env.agent, ag), t
            d = (env.stats - before).astype(np.int64)
            assert tuple(d[:3]) == (int(done.sum()), int(succ.sum()), n), t
            assert np.array_equal(env.expert, want_e), t
            if mode in ("tick", "f32", "f32_wire_u8", "advance"):
                assert np.array_equal(env.features, want_f), t
            elif mode == "u8":
                assert np.array_equal(env.features_u8.astype(np.float32), want_f), t
    env.close()


# ------------------------------------------------------------------------------------------------
# A2: several ticks from exported states

class StartTicks(object):
    """The rollout tick (trainers/imitation.py:42-73, auto-reset) on the C oracle, for episodes that
    start at arbitrary states: grid, inventory, position and facing of the start state."""

    def __init__(self, oracle, grid, inv, pos, dirs, task, start, T):
        self.o, self.T = oracle, T
        self.s_grid, self.s_inv = grid[start].copy(), inv[start].astype(np.int32)
        self.s_pos, self.s_dir = pos[start].astype(np.int32), dirs[start].astype(np.int32)
        self.grid, self.inv = grid.copy(), inv.astype(np.int32)
        self.pos, self.dir = pos.astype(np.int32), dirs.astype(np.int32)
        self.task = task.astype(np.int32)
        self.timer = np.full(len(grid), T, np.int32)
        self.stats = np.zeros(3, np.int64)

    def tick(self, actions=None):
        o = self
        e, _, _ = o.o.expert(o.grid, o.inv, o.pos, o.dir, o.task)
        f = o.o.features(o.grid, o.inv, o.pos, o.dir)
        act = e if actions is None else actions.astype(np.int32)
        o.timer = o.timer - 1
        done = (act == 5) | (o.timer <= 0)
        succ = done & (o.o.satisfies(o.grid, o.inv, o.pos, o.dir, o.task) == 1)
        g, i, p, d, _ = o.o.step(o.grid, o.inv, o.pos, o.dir, np.where(done, 5, act).astype(np.int32))
        o.grid = np.where(done[:, None], o.s_grid, g)
        o.inv = np.where(done[:, None], o.s_inv, i).astype(np.int32)
        o.pos = np.where(done[:, None], o.s_pos, p).astype(np.int32)
        o.dir = np.where(done, o.s_dir, d).astype(np.int32)
        o.timer = np.where(done, o.T, o.timer).astype(np.int32)
        o.stats += (int(done.sum()), int(succ.sum()), len(done))
        return e.astype(np.uint8), f.astype(np.uint8), done.astype(np.uint8), succ.astype(np.uint8)


@pytest.mark.parametrize("which", ["medium", "custom"])
@pytest.mark.parametrize("driver", ["teacher", "random"])
def test_multi_tick_from_exported_states(which, driver, medium_tables, medium_oracle, medium_states,
                                         custom_tables, custom_oracle, custom_states):
    """T = 8 ticks from exported states, episodes restarting at other exported states: teacher-driven
    (timer 40), and random actions with timer 5 (resets inside the launch).  Every rollout variant
    (9-frame ring) and 8 fused ticks: each tick's outputs, the final state and the counters."""
    from psketch_b200.vec import VecCraft
    tables, oracle, S = {"medium": (medium_tables, medium_oracle, medium_states),
                         "custom": (custom_tables, custom_oracle, custom_states)}[which]
    A = _arrays(S)
    ii, tt = _pairs(tables, oracle, S)
    rng = np.random.RandomState(41)
    pick = rng.choice(len(ii), size=min(len(ii), 65536 + 37), replace=False)
    ii, tt = ii[pick], tt[pick]
    Tk, RING = 8, 9
    timer = 40 if driver == "teacher" else 5
    acts = None if driver == "teacher" else rng.choice(6, size=(Tk, len(ii)), p=[.19, .19, .19, .19, .2, .04]).astype(np.uint8)
    args = (A["grid"][ii], A["inv"][ii], A["pos"][ii], A["dir"][ii], tt)

    start = rng.permutation(len(ii))
    keep_idx = np.arange(len(ii))
    for attempt in range(6):
        orc = StartTicks(oracle, *args, start, timer)
        ticks = [orc.tick(None if acts is None else acts[t][keep_idx]) for t in range(Tk)]
        bad = np.zeros(len(keep_idx), bool)
        for e, _, _, _ in ticks:
            bad |= e == 255                 # the teacher asserts on some later state: leave those out
        if not bad.any():
            break
        keep = np.nonzero(~bad)[0]
        keep_idx = keep_idx[keep]
        args = tuple(x[keep] for x in args)
        start = np.argsort(np.argsort(start[keep]))      # ranks: a permutation of the kept envs
    assert not bad.any()
    n = len(keep_idx)
    grid, inv, pos, dirs, task = args
    nf, C = tables.n_features, tables.W * tables.H
    cs = ((C + 63) // 64) * 64
    init = np.zeros((n, 32), np.uint8)
    init[:, :tables.K] = inv[start]
    init[:, 24:26], init[:, 26], init[:, AG_TASK], init[:, AG_TIMER] = pos[start], dirs[start], task, timer
    scen = np.zeros((n, cs), np.uint8)
    scen[:, :C] = grid[start]
    d_acts = None if acts is None else torch.from_numpy(np.ascontiguousarray(acts[:, keep_idx])).cuda()

    def fresh():
        env = VecCraft.from_states(tables, grid, inv, pos, dirs, task=task, max_timesteps=timer)
        env.scen_grid = torch.from_numpy(scen).to(env.device)
        env.init_agent = torch.from_numpy(init).to(env.device)
        return env

    def check_final(env, tag):
        assert np.array_equal(env.cells.cpu().numpy(), orc.grid), tag
        assert np.array_equal(env.inventory.cpu().numpy().astype(np.int32), orc.inv), tag
        assert np.array_equal(env.pos.cpu().numpy().astype(np.int32), orc.pos), tag
        assert np.array_equal(env.dir.cpu().numpy().astype(np.int32), orc.dir), tag
        assert np.array_equal(env.timer.cpu().numpy().astype(np.int32), orc.timer), tag
        assert np.array_equal(env.task.cpu().numpy().astype(np.int32), task), tag
        assert tuple(env.stats.tolist()[:3]) == tuple(orc.stats), tag
        env.check_errors()

    gold = [tuple(torch.from_numpy(x).cuda() for x in tk) for tk in ticks]
    variants = ROLLOUT_VARIANTS if tables.W * tables.H == 64 else [(-1, -1)]
    ring = torch.empty((RING, n, nf), dtype=torch.float32, device="cuda")
    for variant, tma in variants:
        with tuning(rollout_variant=variant, rollout_tma=tma):
            env = fresh()
            ring.fill_(-1.0)
            out = env.rollout(Tk, actions=d_acts, features_out=ring)
            tag = "%s %s rollout %d tma %d" % (which, driver, variant, tma)
            for t, (e, f, done, succ) in enumerate(gold):
                assert torch.equal(out["expert"][t], e), (tag, t)
                assert torch.equal(ring[t], f.float()), (tag, t)
                assert torch.equal(out["done"][t], done) and torch.equal(out["success"][t], succ), (tag, t)
            assert bool((ring[Tk] == -1.0).all()), tag
            check_final(env, tag)
    env = fresh()
    for t, (e, f, done, succ) in enumerate(gold):
        out = env.tick(actions=None if d_acts is None else d_acts[t])
        tag = "%s %s fused tick" % (which, driver)
        assert torch.equal(out["expert"], e) and torch.equal(out["features"], f.float()), (tag, t)
        assert torch.equal(out["done"], done) and torch.equal(out["success"], succ), (tag, t)
    check_final(env, "%s %s fused tick" % (which, driver))


# ------------------------------------------------------------------------------------------------
# A3: the teacher's assertion through every fused path

def test_teacher_assertion_on_every_fused_path(medium_tables, medium_states):
    """Tasks 1-4 and 6 (leaves that are neither 'use' nor 'go') make the reference assert: expert 255
    and AssertionError through the fused tick, the byte frame, the rollout and the host paths."""
    from psketch_b200.host import HostCraft
    from psketch_b200.vec import VecCraft
    S = _arrays(medium_states)
    n = 4099
    task = np.resize([1, 2, 3, 4, 6], n)
    assert (S["expert"][np.arange(n), task] == 255).all()
    args = (S["grid"][:n], S["inv"][:n], S["pos"][:n], S["dir"][:n])
    nf = medium_tables.n_features
    for path in ("tick", "tick_u8", "advance", "rollout", "rollout_u8"):
        env = VecCraft.from_states(medium_tables, *args, task=task)
        if path == "tick":
            e = env.tick()["expert"]
        elif path == "advance":
            e = env.tick(advance_first=True)["expert"]
        elif path == "tick_u8":
            e = env.tick(features_out=torch.empty((n, nf), dtype=torch.uint8, device=env.device))["expert"]
        else:
            dt = torch.uint8 if path == "rollout_u8" else torch.float32
            e = env.rollout(1, features_out=torch.empty((1, n, nf), dtype=dt, device=env.device))["expert"][0]
        assert bool((e == 255).all()), path
        with pytest.raises(AssertionError):
            env.check_errors()
    for m in (n, 64):                              # copy route, zero-copy route
        env = HostCraft(medium_tables, S["grid"][:m], np.arange(m), S["pos"][:m], task[:m], init_dir=S["dir"][:m])
        with pytest.raises(AssertionError):
            env.tick()
        assert (env.expert == 255).all()
        env.reset_resident()
        with pytest.raises(AssertionError):
            env.tick_resident(features="f32")
        assert (env.expert == 255).all()
        env.close()


# ------------------------------------------------------------------------------------------------
# A4: the u8 inventory limit

def _edge_batch(tables, oracle, S, n, seed):
    """Edge states with one task each whose teacher answer is defined on the state."""
    E = edge_states(tables, _arrays(S), n, seed)
    rng = np.random.RandomState(seed)
    m = len(E["grid"])
    ok = np.stack([oracle.expert(E["grid"], E["inv"], E["pos"], E["dir"], np.full(m, t))[0] != 255
                   for t in range(1, tables.n_tasks)], axis=1)
    task = np.array([rng.choice(np.nonzero(row)[0]) + 1 if row.any() else 0 for row in ok], np.int32)
    keep = task > 0
    E = {k: v[keep] for k, v in E.items()}
    E["task"] = task[keep]
    return E


@pytest.mark.parametrize("which", ["medium", "custom"])
def test_inventory_limit_on_every_path(which, medium_tables, medium_oracle, medium_states, custom_tables,
                                       custom_oracle, custom_states):
    """Counts 13..255 on the kinds the next USE touches.  Features, satisfies and the teacher equal the
    oracle (int32 counts); a step whose counts stay <= 255 equals the oracle on every path; a step that
    would pass 255 raises PSK_FLAG_INV_OVERFLOW -> OverflowError and leaves the documented state (the
    grab clears the cell and keeps 255, the overflowing recipe is skipped, later ones still fire) — the
    same on psk_craft_step (every variant), the fused tick (every shape, both orders), the byte frame,
    the rollout kernel, the host paths and the Craft façade."""
    from psketch_b200.host import HostCraft
    from psketch_b200.vec import VecCraft
    tables, oracle, S = {"medium": (medium_tables, medium_oracle, medium_states),
                         "custom": (custom_tables, custom_oracle, custom_states)}[which]
    E = _edge_batch(tables, oracle, S, 3000, seed=7)
    grid, inv, pos, dirs, task = E["grid"], E["inv"], E["pos"], E["dir"], E["task"]
    n, C, K, nf = len(grid), tables.W * tables.H, tables.K, tables.n_features
    T = 40
    env = VecCraft.from_states(tables, grid, inv, pos, dirs, task=task, max_timesteps=T)
    snap = env.snapshot()
    # ---- observations: every feature builder, satisfies and the teacher for every task
    want_f = oracle.features(grid, inv, pos, dirs)
    assert want_f.max() == 255
    for impl in (0, 1, 2):
        assert np.array_equal(env.features(impl=impl).cpu().numpy(), want_f), impl
    assert np.array_equal(env.features_u8().cpu().numpy().astype(np.float32), want_f)
    with tuning(feat_persist=1):
        assert np.array_equal(env.features().cpu().numpy(), want_f)
    for t in range(1, tables.n_tasks):
        tk = torch.full((n,), t, dtype=torch.uint8, device=env.device)
        assert np.array_equal(env.satisfies(tk).cpu().numpy(), oracle.satisfies(grid, inv, pos, dirs, np.full(n, t))), t
        o_e = oracle.expert(grid, inv, pos, dirs, np.full(n, t))[0]
        assert np.array_equal(env.expert(tk).cpu().numpy().astype(np.int32), o_e), t
        if (o_e == 255).any():
            with pytest.raises(AssertionError):
                env.check_errors()
        env.check_errors()
    o_exp = oracle.expert(grid, inv, pos, dirs, task)[0].astype(np.uint8)
    sat = oracle.satisfies(grid, inv, pos, dirs, task)
    # ---- one step / tick per action on every path
    for a in range(6):
        act = np.full(n, a, np.uint8)
        g, iv, p, d, over, _ = step_u8(tables, grid, inv, pos, dirs, act)
        og, oi, op, od, _ = oracle.step(grid, inv, pos, dirs, act.astype(np.int32))
        ok = ~over
        assert np.array_equal(g[ok], og[ok]) and np.array_equal(iv[ok], oi[ok])
        assert over.any() == (a == 4)
        want_agent = np.zeros((n, 32), np.uint8)
        want_agent[:, :K], want_agent[:, 24:26], want_agent[:, 26] = iv, p, d
        want_agent[:, AG_TASK] = task

        def check_state(env, tag, tick):
            # a tick counts the timer down; STOP ends the episode, which from_states restarts at the
            # state itself (step_u8 leaves it unchanged for STOP), timer full again
            w = want_agent.copy()
            w[:, AG_TIMER] = T - 1 if tick and a != 5 else T
            assert np.array_equal(env.cells.cpu().numpy(), g), tag
            assert np.array_equal(env.agent.cpu().numpy(), w), tag

        def check_flags(raise_fn, tag):
            if over.any():
                with pytest.raises(OverflowError):
                    raise_fn()
            else:
                raise_fn()

        # psk_craft_step, every variant
        for sv in (0, 1, 2):
            with tuning(step_variant=sv):
                env.restore(snap)
                env.step(torch.from_numpy(act).to(env.device))
                check_state(env, ("step", sv, a), tick=False)
                check_flags(env.check_errors, ("step", sv, a))
        if over.any():                     # the envs that stay within 255 alone: the oracle, no flag
            sub = VecCraft.from_states(tables, grid[ok], inv[ok], pos[ok], dirs[ok], task=task[ok])
            sub.step(torch.from_numpy(act[ok]).to(sub.device))
            sub.check_errors()
            assert np.array_equal(sub.cells.cpu().numpy(), og[ok])
            assert np.array_equal(sub.inventory.cpu().numpy().astype(np.int32), oi[ok])
        # the rollout tick, every CTA shape and order, the byte frame and the pipeline
        d_act = torch.from_numpy(act).to(env.device)
        tick_runs = [("shape %d" % v, dict(tick_variant=v), False, False) for v in sorted(TICK_SHAPES)]
        tick_runs += [("advance", {}, True, False), ("u8", {}, False, True), ("u8 advance", {}, True, True),
                      ("pipeline", None, False, False)]
        for name, knobs, adv, u8 in tick_runs:
            tag = (name, a)
            with tuning(**(knobs or {})):
                env.restore(snap)
                env.stats.zero_()
                fo = torch.empty((n, nf), dtype=torch.uint8, device=env.device) if u8 else None
                out = env.tick(actions=d_act, features_out=fo, fused=knobs is not None, advance_first=adv)
                check_state(env, tag, tick=True)
                done = np.full(n, a == 5)
                assert np.array_equal(out["done"].cpu().numpy(), done.astype(np.uint8)), tag
                assert np.array_equal(out["success"].cpu().numpy(), (done & (sat == 1)).astype(np.uint8)), tag
                assert env.stats.tolist()[:3] == [int(done.sum()), int((done & (sat == 1)).sum()), n], tag
                f = out["features"].cpu().numpy().astype(np.float32)
                if adv:
                    cur = (env.cells.cpu().numpy(), env.inventory.cpu().numpy().astype(np.int32),
                           env.pos.cpu().numpy().astype(np.int32), env.dir.cpu().numpy().astype(np.int32))
                    e_after = oracle.expert(*cur, task)[0]
                    assert np.array_equal(out["expert"].cpu().numpy().astype(np.int32), e_after), tag
                    assert np.array_equal(f, oracle.features(*cur)), tag
                    if (e_after == 255).any():      # the teacher's assertion comes first
                        with pytest.raises(AssertionError):
                            env.check_errors()
                        continue
                else:
                    assert np.array_equal(out["expert"].cpu().numpy(), o_exp), tag
                    assert np.array_equal(f, want_f), tag
                check_flags(env.check_errors, tag)
        rollouts = [(-1, -1), (0, 1), (4, 0)] if C == 64 else [(-1, -1)]
        for variant, tma in rollouts:
            for u8 in (False, True):
                with tuning(rollout_variant=variant, rollout_tma=tma):
                    env.restore(snap)
                    ring = torch.empty((1, n, nf), dtype=torch.uint8 if u8 else torch.float32, device=env.device)
                    out = env.rollout(1, actions=d_act[None], features_out=ring)
                    tag = ("rollout", variant, tma, u8, a)
                    check_state(env, tag, tick=True)
                    assert np.array_equal(out["expert"][0].cpu().numpy(), o_exp), tag
                    assert np.array_equal(ring[0].cpu().numpy().astype(np.float32), want_f), tag
                    check_flags(env.check_errors, tag)
        # host paths: state round trip, resident (copy route and, at 500 envs, zero-copy)
        for m in (n, 500):
            h = HostCraft(tables, grid[:m], np.arange(m), pos[:m], task[:m], init_dir=dirs[:m], max_timesteps=T)
            for mode in ("tick", "resident"):
                h.grid[:, :C] = grid[:m]
                h.agent[:] = 0
                h.agent[:, :K], h.agent[:, 24:26], h.agent[:, 26] = inv[:m], pos[:m], dirs[:m]
                h.agent[:, AG_TASK], h.agent[:, AG_TIMER] = task[:m], T
                tag = ("host", m, mode, a)
                with pytest.raises(OverflowError) if over[:m].any() else contextlib.nullcontext():
                    if mode == "tick":
                        h.tick(actions=act[:m])
                    else:
                        h.upload()
                        h.tick_resident(actions=act[:m], features="f32")
                if mode == "resident":
                    h.download(keep_resident=False)
                assert np.array_equal(h.expert, o_exp[:m]) and np.array_equal(h.features, want_f[:m]), tag
                if a == 5:       # HostCraft restarts at its own episode start (empty inventory)
                    continue
                assert np.array_equal(h.grid[:, :C], g[:m]), tag
                assert np.array_equal(h.agent[:, :K], iv[:m]) and np.array_equal(h.agent[:, 24:26], p[:m]), tag
                assert np.array_equal(h.agent[:, 26], d[:m]) and (h.agent[:, AG_TIMER] == T - 1).all(), tag
            h.close()
    # ---- the Craft façade: the same rule, the same exception
    from psketch_b200.worlds import craft as facade
    act = np.full(n, 4)
    g, iv, p, d, over, _ = step_u8(tables, grid, inv, pos, dirs, act)
    for sel in (np.nonzero(~over)[0][:40], np.nonzero(over)[0][:3]):
        world = facade.CraftWorld(tables=tables)
        kids = []
        for i in sel:
            s = world.init_state(grid[i], tuple(int(v) for v in pos[i]), dir=int(dirs[i]))
            s.inventory = inv[i]
            kids.append(s.step(4)[1])
        if over[sel].any():
            with pytest.raises(OverflowError):
                kids[0].features()
            continue
        for s, i in zip(kids, sel):
            assert np.array_equal(s.cells, g[i]) and np.array_equal(s.inventory, iv[i].astype(np.float64)), i
