"""Light kernels (psk_light.cu) on every state of scenarios beyond the 60 reference ones: the
generator's draws of all 17 goals up to 7 keys and every board shape and goal room, and synthetic
records up to the C ABI's limits (8 keys, 8 doors, 31 x 31 boards, goal rooms in column / row 4,
shared doors, keys on wall openings, door cells and shared cells), one batch, max_keys = 8.
The scenario sets are built in tests/test_light_limits_cpu.py.

Everything is compared with oracle/light_oracle.c, whose step / features / satisfies are pinned to
the reference's exported states and whose orc_light_expert is the brute-force specification of
the teacher:
  * step (5 actions), features, satisfies and reset on every state, exactly;
  * the teacher table against the shortest-path equations through the oracle's step, in numpy on
    the kernel's own dense table; the table lookup, the per-env search kernel and (on a sample) the
    brute force give the same answers;
  * psk_light_tick on every state with the teacher's and each forced action; psk_light_tick and
    psk_light_rollout over mixed ragged batches against a numpy replay on the oracle;
  * the table, states and outputs inside a canary arena at 8 keys, and a table built with max_keys
    below a scenario's n_keys, whose lookups must answer 255 / -2 instead of reading past it.
"""
import time
from types import SimpleNamespace

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from test_light_limits_cpu import generator_set, oracle_of, records, synthetic_set   # noqa: E402

ALLOWED = np.asarray([0, 1, 2, 3, 4, 254, 255])
INF = 1 << 20


def _scenarios():
    return [sc for _, _, sc in generator_set()] + [sc for _, sc in synthetic_set()]


def _cells(c):
    """(wall u8[32, 32], lock i64[32, 32]: keys locking a door at the cell) of a record."""
    rows = np.asarray(list(c.walls), np.uint64)
    wall = ((rows[:, None] >> np.arange(32, dtype=np.uint64)[None, :]) & 1).astype(np.uint8)
    doors = np.zeros((32, 32), np.int64)
    for d in range(c.n_doors):
        doors[c.doors[2 * d], c.doors[2 * d + 1]] += 1
    lock = np.zeros((32, 32), np.int64)
    for k in range(c.n_keys):
        tx, ty = c.keys[4 * k + 2], c.keys[4 * k + 3]
        if doors[tx, ty]:
            lock[tx, ty] |= 1 << k
    return wall, lock, doors


def all_states(recs, locked_doors=False):
    """Every (scenario, x, y, key mask) of every scenario: each cell one can stand on (no wall, no
    door locked by a key of the mask) under each key subset.  ``locked_doors``: the door cells
    under the masks that lock them instead (reachable only through set_state)."""
    scen, st = [], []
    for si, c in enumerate(recs):
        wall, lock, _ = _cells(c)
        free = np.argwhere(wall == 0)
        lk = lock[free[:, 0], free[:, 1]]
        ms = np.arange(1 << c.n_keys)
        hit = (ms[:, None] & lk[None, :]) != 0
        m_i, c_i = np.nonzero(hit if locked_doors else ~hit)
        scen.append(np.full(len(m_i), si, np.int32))
        st.append(np.column_stack([free[c_i], ms[m_i]]).astype(np.int32))
    return np.concatenate(scen), np.concatenate(st)


def table_views(v):
    """The kernel's teacher table as numpy: dist u16[S, 2^max_keys, 32, 32], the per-cell maps
    u8[S, 3, 32, 32] (keys locking a door here, keys lying here, doors here), act u8[S, 2^max_keys, 32, 32]."""
    S, cap = v.scen.shape[0], 1 << v.max_keys
    t = v.teacher_table().cpu().numpy().view(np.uint16).reshape(S, -1)
    assert t.shape[1] == cap * 1024 + 1536 + cap * 512
    dist = t[:, :cap * 1024].reshape(S, cap, 32, 32)
    aux = np.ascontiguousarray(t[:, cap * 1024:cap * 1024 + 1536]).view(np.uint8).reshape(S, 3, 32, 32)
    act = np.ascontiguousarray(t[:, cap * 1024 + 1536:]).view(np.uint8).reshape(S, cap, 32, 32)
    return dist, aux, act


def _u8(a):
    return np.asarray(a).astype(np.uint8)


@pytest.fixture(scope="module")
def W():
    from psketch_b200.worlds.light import VecLight
    scens = _scenarios()
    recs = records(scens)
    si, st = all_states(recs)
    xsi, xst = all_states(recs, locked_doors=True)
    v = VecLight(scens, si)
    assert v.max_keys == 8
    dist, aux, act = table_views(v)
    init = np.asarray([[c.init_x, c.init_y, (1 << c.n_keys) - 1] for c in recs], np.int32)
    names = {name: len(generator_set()) + i for i, (name, _) in enumerate(synthetic_set())}
    return SimpleNamespace(scens=scens, recs=recs, o=oracle_of(recs), si=si, st=st, xsi=xsi, xst=xst, v=v,
                           dist=dist, aux=aux, act=act, init=init, names=names,
                           nk=np.asarray([c.n_keys for c in recs]))


def replay_tick(o, act, init, si, cur, a_in, max_timesteps, cap=None):
    """One psk_light_tick on the oracle.  cur i32[n, 4] = x, y, mask, steps; act: teacher answers
    [S, cap, 32, 32] (a mask >= cap answers 255)."""
    x, y, m, e = cur.T
    cap = act.shape[1] if cap is None else cap
    ref = np.where(m < cap, act[si, np.minimum(m, cap - 1), x, y], 255).astype(np.int32)
    feat, sat, _ = o.run(si, cur[:, :3])
    a = ref if a_in is None else np.asarray(a_in, np.int32)
    elapsed = e + 1
    done = (a >= 5) | (elapsed >= max_timesteps)
    succ = done & (sat == 1)
    _, _, nxt = o.run(si, cur[:, :3], np.where(done, 0, a))
    new = np.where(done[:, None], np.column_stack([init[si], np.zeros(len(si), np.int32)]),
                   np.column_stack([nxt, elapsed]))
    return ref, feat, done, succ, new.astype(np.int32)


def _check_tick(out, v, want, what):
    ref, feat, done, succ, new = want
    assert np.array_equal(out["expert"].cpu().numpy().astype(np.int32), ref), what
    if out.get("features") is not None:
        assert np.array_equal(out["features"].cpu().numpy(), feat), what
    assert np.array_equal(out["done"].cpu().numpy().astype(bool), done), what
    assert np.array_equal(out["success"].cpu().numpy().astype(bool), succ), what
    assert np.array_equal(v.state.cpu().numpy().astype(np.int32), new), what


def test_step_features_satisfies_reset_on_every_state(W):
    v = W.v
    si = np.concatenate([W.si, W.xsi])
    st = np.concatenate([W.st, W.xst])
    n = len(si)
    assert len(W.si) > 500000 and len(W.xsi) > 4000
    v.reset()
    got = v.state.cpu().numpy().astype(np.int32)
    assert np.array_equal(got[:, :3], W.init[W.si]) and not got[:, 3].any()
    v.scen_idx = si
    v.n = n
    v.state = torch.zeros((n, 4), dtype=torch.uint8, device=v.device)
    st4 = np.zeros((n, 4), np.uint8)
    st4[:, :3] = st
    v.set_state(st4)
    feat, sat, _ = W.o.run(si, st)
    assert np.array_equal(v.features().cpu().numpy(), feat)
    assert np.array_equal(v.satisfies().cpu().numpy(), sat)
    for a in range(5):
        v.set_state(st4)
        v.step(np.full(n, a, np.uint8))
        _, _, nxt = W.o.run(si, st, np.full(n, a))
        assert np.array_equal(v.state.cpu().numpy().astype(np.int32)[:, :3], nxt), a
    v.check_errors()
    # the edges are in the set: two keys on one cell, two locked / open doors on one cell, a key on
    # a wall opening (feature 0 although it lies underfoot)
    assert feat[:, 8].max() == 3 and feat[:, 0].max() == 2 and feat[:, 4].max() == 2
    wk = W.names["wall_and_door_keys"]
    on = (si == wk) & (st[:, 0] == 6) & (st[:, 1] == 1) & (st[:, 2] & 1 == 1)
    assert on.any() and not feat[on, 8:].any()


def test_teacher_table_cell_maps(W):
    for si, c in enumerate(W.recs):
        _, lock, doors = _cells(c)
        keys = np.zeros((32, 32), np.int64)
        for k in range(c.n_keys):
            keys[c.keys[4 * k], c.keys[4 * k + 1]] |= 1 << k
        assert np.array_equal(W.aux[si, 0], lock), si
        assert np.array_equal(W.aux[si, 1], keys), si
        assert np.array_equal(W.aux[si, 2], doors), si


def test_teacher_table_solves_the_shortest_path_equations(W):
    """dist = 0 exactly in the goal room; dist = 1 + min over the actions that change the state of
    dist(successor); unreachable states have only unreachable successors; the action is the
    smallest index attaining the minimum; the lookup kernel returns the table's entries."""
    si, st, v = W.si, W.st, W.v
    n = len(si)
    x, y, m = st.T
    D = W.dist[si, m, x, y].astype(np.int64)
    A = W.act[si, m, x, y].astype(np.int64)
    unreachable = D == 0xFFFF
    _, sat, _ = W.o.run(si, st)
    assert np.array_equal(D == 0, sat == 1) and np.array_equal(A == 254, sat == 1)
    succ = np.full((5, n), INF, np.int64)
    for a in range(5):
        _, _, nxt = W.o.run(si, st, np.full(n, a))
        moved = (nxt != st).any(axis=1)
        d = W.dist[si, nxt[:, 2], nxt[:, 0], nxt[:, 1]].astype(np.int64)
        succ[a] = np.where(moved & (d != 0xFFFF), d, INF)
    best = succ.min(axis=0)
    assert np.array_equal(unreachable, (best >= INF) & (sat == 0))
    assert (A[unreachable] == 255).all()
    ok = ~unreachable & (sat == 0)
    assert np.array_equal(D[ok], 1 + best[ok])
    assert np.array_equal(A[ok], succ[:, ok].argmin(axis=0))
    # the set reaches far: long plans, unreachable states and USE as the best action at 8 keys
    big = W.nk[si] == 8
    assert D[ok & big].max() > 40 and unreachable[big].any() and (A[ok & big] == 4).any()
    # the lookup kernel
    st4 = np.zeros((n, 4), np.uint8)
    st4[:, :3] = st
    v.scen_idx = si
    v.n = n
    v.state = torch.zeros((n, 4), dtype=torch.uint8, device=v.device)
    v.set_state(st4)
    act, dist = (t.cpu().numpy().astype(np.int64) for t in v.expert())
    assert np.array_equal(act, A)
    assert np.array_equal(dist, np.where(unreachable, -1, D))


def test_search_kernel_equals_the_table(W):
    """psk_light_expert (one backward flood per env) against the table.  Every state of the
    scenarios with up to 6 keys, every third state of those with 7 and 8 (one warp per CTA there)."""
    from psketch_b200.worlds.light import VecLight
    idx = np.arange(len(W.si))
    sel = idx[(W.nk[W.si] <= 6) | (idx % 3 == 0)]
    si, st = W.si[sel], W.st[sel]
    v = VecLight(W.scens, si)
    st4 = np.zeros((len(sel), 4), np.uint8)
    st4[:, :3] = st
    v.set_state(st4)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    act, dist = v.expert(search=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    x, y, m = st.T
    D = W.dist[si, m, x, y].astype(np.int64)
    want_d = np.where(D == 0xFFFF, -1, D)
    act, dist = act.cpu().numpy().astype(np.int64), dist.cpu().numpy().astype(np.int64)
    co = si == W.names["colocated_keys"]
    assert co.sum() > 1000
    assert np.array_equal(dist[co], want_d[co]) and np.array_equal(act[co], W.act[si, m, x, y][co])
    assert np.array_equal(dist, want_d)
    assert np.array_equal(act, W.act[si, m, x, y])
    print("search kernel: %d states (%d at 8 keys) in %.3f s" % (len(sel), int((W.nk[si] == 8).sum()), dt))


def test_brute_force_on_a_sample(W):
    """orc_light_expert (forward BFS from every successor) on ~2,000 states: every scenario, both
    key extremes, a share of unreachable states."""
    rng = np.random.RandomState(3)
    x, y, m = W.st.T
    D = W.dist[W.si, m, x, y].astype(np.int64)
    pick = [rng.choice(np.flatnonzero(W.si == s), 15, replace=False) for s in range(len(W.recs))]
    pick.append(rng.choice(np.flatnonzero(D == 0xFFFF), 200, replace=False))
    pick.append(rng.choice(np.flatnonzero((W.nk[W.si] == 8) & (D != 0xFFFF)), 300, replace=False))
    sel = np.unique(np.concatenate(pick))
    assert len(sel) > 1500
    want_a, want_d = W.o.expert(W.si[sel], W.st[sel])
    got_d = np.where(D[sel] == 0xFFFF, -1, D[sel])
    assert np.array_equal(got_d, want_d)
    assert np.array_equal(W.act[W.si[sel], m[sel], x[sel], y[sel]].astype(np.int64), want_a)


def test_tick_on_every_state(W):
    """psk_light_tick from every state (locked door cells included), step counters spread over
    0..254: the teacher's action, each forced action, and a random mix with bad action bytes."""
    v = W.v
    si = np.concatenate([W.si, W.xsi])
    st = np.concatenate([W.st, W.xst])
    n = len(si)
    rng = np.random.RandomState(5)
    cur = np.column_stack([st, rng.randint(0, 255, n)]).astype(np.int32)
    v.scen_idx = si
    v.n = n
    v.state = torch.zeros((n, 4), dtype=torch.uint8, device=v.device)
    mixed = rng.choice([0, 1, 2, 3, 4, 4, 5, 200, 255], n)
    for a_in, T in ((None, 255), (None, 1), (0, 200), (1, 37), (2, 255), (3, 100), (4, 255), (mixed, 128)):
        v.set_state(_u8(cur))
        v.stats = None
        a_in = None if a_in is None else np.asarray(a_in) + np.zeros(n, np.int32)
        out = v.tick(actions=None if a_in is None else _u8(a_in), max_timesteps=T)
        want = replay_tick(W.o, W.act, W.init, si, cur, a_in, T)
        _check_tick(out, v, want, (None if a_in is None else a_in[:3], T))
        s = v.stats.cpu().numpy()
        assert (s[0], s[1], s[2]) == (int(want[2].sum()), int(want[3].sum()), n)


def test_tick_and_rollout_replay_on_mixed_batches(W):
    """Ragged batches mixing 0..8 keys, half of the envs from reset and half from random states:
    psk_light_rollout (feature ring shorter than the launch) then psk_light_tick, teacher-driven and
    with random actions (bad bytes included), max_timesteps 1, 23 and 255, against the replay."""
    from psketch_b200.worlds.light import VecLight
    rng = np.random.RandomState(7)
    for n, T, R, max_t in ((1, 5, 2, 255), (33, 9, 4, 1), (4099, 12, 5, 23), (70001, 8, 3, 255)):
        rows = rng.randint(0, len(W.si), n)
        for i, name in enumerate(("no_keys", "eight_keys_path")[:n]):
            rows[i] = rng.choice(np.flatnonzero(W.si == W.names[name]))
        si = W.si[rows]
        assert 0 in W.nk[si] and (n == 1 or 8 in W.nk[si])
        v = VecLight(W.scens, si)
        v._table = W.v._table
        cur = np.column_stack([W.st[rows], rng.randint(0, 100, n)]).astype(np.int32)
        fresh = rng.rand(n) < 0.5
        cur[fresh] = np.column_stack([W.init[si[fresh]], np.zeros(int(fresh.sum()), np.int32)])
        for teacher in (True, False):
            v.set_state(_u8(cur))
            v.stats = None
            acts = None if teacher else rng.choice([0, 1, 2, 3, 4] * 6 + [9], size=(T, n)).astype(np.uint8)
            ring = torch.full((R, n, 12), -1.0, device=v.device)
            got = v.rollout(T, actions=None if acts is None else torch.from_numpy(acts).to(v.device),
                            features_out=ring, max_timesteps=max_t)
            tot = np.zeros(3, np.int64)
            frames = {}
            for t in range(T):
                ref, feat, done, succ, cur = replay_tick(W.o, W.act, W.init, si, cur,
                                                         None if acts is None else acts[t], max_t)
                frames[t % R] = feat
                tot += (int(done.sum()), int(succ.sum()), n)
                for k, w in (("expert", ref), ("done", done), ("success", succ)):
                    assert np.array_equal(got[k][t].cpu().numpy().astype(w.dtype), w), (n, teacher, t, k)
            for r, feat in frames.items():
                assert np.array_equal(ring[r].cpu().numpy(), feat), (n, teacher, r)
            assert np.array_equal(v.state.cpu().numpy().astype(np.int32), cur), (n, teacher)
            assert tuple(v.stats.cpu().numpy()[:3]) == tuple(tot), (n, teacher)
            for t in range(3):
                a_in = None if teacher else rng.randint(0, 5, n).astype(np.uint8)
                out = v.tick(actions=a_in, max_timesteps=max_t)
                want = replay_tick(W.o, W.act, W.init, si, cur, a_in, max_t)
                _check_tick(out, v, want, (n, teacher, "tick", t))
                cur = want[4]


def _carve_env(v, arena, n):
    v.state = arena.carve((n, 4), torch.uint8)
    v.stats = arena.carve((4,), torch.int64).zero_()


def test_kernels_stay_inside_their_buffers_at_8_keys(W):
    """The synthetic set (8 keys, max_keys 8): teacher table, state, lookup, tick and rollout
    outputs carved out of a canary arena; results equal ordinary allocations, the guard bands stay
    intact and no teacher answer is a canary byte."""
    from psketch_b200.worlds.light import VecLight
    from test_bounds_gpu import Arena
    synth = [sc for _, sc in synthetic_set()]
    first = len(generator_set())
    rng = np.random.RandomState(8)
    rows = rng.choice(np.flatnonzero(W.si >= first), 4099, replace=False)
    si, st4 = W.si[rows] - first, np.zeros((4099, 4), np.uint8)
    st4[:, :3] = W.st[rows]
    n, T, R = len(si), 6, 4
    v, ref = VecLight(synth, si), VecLight(synth, si)
    assert v.max_keys == 8
    nbytes = v.lib.psk_light_teacher_table_bytes(len(synth), 8)
    arena = Arena(nbytes + n * (4 + 2 + 1 + 48 * (R + 1) + 3 * (T + 1)) + 64 * 1024, v.device)
    v._table = arena.carve((nbytes // 2,), torch.int16)
    _carve_env(v, arena, n)
    rc = v.lib.psk_light_teacher_build(v._p(v.scen), len(synth), 8, v._p(v._table), v._stream())
    assert rc == 0
    assert torch.equal(v._table, ref.teacher_table()) and arena.guards_intact()
    for obj in (v, ref):
        obj.set_state(st4)
    act, dist = arena.carve((n,), torch.uint8), arena.carve((n,), torch.int16)
    rc = v.lib.psk_light_expert_table(v._p(v.scen), v._p(v.scen_idx), v._p(v.state), v._p(v._table), 8,
                                      v._p(act), v._p(dist), n, v._stream())
    assert rc == 0
    a2, d2 = ref.expert()
    assert torch.equal(act, a2) and torch.equal(dist, d2) and arena.guards_intact()
    assert np.isin(act.cpu().numpy(), ALLOWED).all()
    out = dict(expert=arena.carve((n,), torch.uint8), done=arena.carve((n,), torch.uint8),
               success=arena.carve((n,), torch.uint8))
    feats = arena.carve((n, 12), torch.float32)
    for t in range(3):
        a = ref.tick(max_timesteps=9)
        b = v.tick(features_out=feats, out=out, max_timesteps=9)
        for k in ("expert", "done", "success", "features"):
            assert torch.equal(a[k], b[k]), (t, k)
        assert torch.equal(v.state, ref.state) and arena.guards_intact()
        assert np.isin(b["expert"].cpu().numpy(), ALLOWED).all()
    ring = arena.carve((R, n, 12), torch.float32)
    rout = dict(expert=arena.carve((T, n), torch.uint8), done=arena.carve((T, n), torch.uint8),
                success=arena.carve((T, n), torch.uint8))
    got = v.rollout(T, features_out=ring, out=rout, max_timesteps=9)
    for t in range(T):
        want = ref.tick(max_timesteps=9)
        for k in ("expert", "done", "success"):
            assert torch.equal(got[k][t], want[k]), (t, k)
        if t >= T - R:
            assert torch.equal(ring[t % R], want["features"]), t
    assert torch.equal(v.state, ref.state) and torch.equal(v.stats, ref.stats) and arena.guards_intact()
    assert np.isin(rout["expert"].cpu().numpy(), ALLOWED).all()


def test_masks_outside_the_table_answer_255(W):
    """A table built with max_keys = 3 for a batch whose last scenario has 8 keys: reset gives its
    envs all 8 key bits, which have no layer in the table.  The lookup, tick and rollout answer 255 /
    dist -2 there (as the search kernel does) instead of reading past the table, which is carved
    from a canary arena with nothing after it; envs of the other scenarios get the answers of a
    table built for them alone.  Mask bits above a scenario's keys, written past set_state, the same."""
    from psketch_b200.worlds.light import VecLight
    from test_bounds_gpu import Arena
    names = dict(synthetic_set())
    small = [names[k] for k in ("no_keys", "init_is_goal", "key_behind_its_door", "goal_row_4")]
    scens = small + [names["eight_keys_path"]]
    recs = records(scens)
    o = oracle_of(recs)
    si_s, st_s = all_states(recs[:-1])
    rng = np.random.RandomState(12)
    big = rng.choice(1 << 8, 3000)
    si = np.concatenate([si_s, np.full(3000 + 64, 4, np.int32)])
    st = np.concatenate([st_s, np.column_stack([np.full(3000, 3), np.full(3000, 3), big]),
                         np.tile([3, 3, 255], (64, 1))]).astype(np.int32)
    n = len(si)
    v, ref = VecLight(scens, si), VecLight(small, si_s)
    v.max_keys = 3
    assert ref.max_keys == 3
    nbytes = v.lib.psk_light_teacher_table_bytes(len(scens), 3)
    arena = Arena(n * (4 + 2 + 1 + 48 + 3) + 8 * 1024 + nbytes + 512 * 1024, v.device)
    _carve_env(v, arena, n)
    act, dist = arena.carve((n,), torch.uint8), arena.carve((n,), torch.int16)
    out = dict(expert=arena.carve((n,), torch.uint8), done=arena.carve((n,), torch.uint8),
               success=arena.carve((n,), torch.uint8))
    feats = arena.carve((n, 12), torch.float32)
    v._table = arena.carve((nbytes // 2,), torch.int16)         # last: canary bytes behind it
    assert arena.buf.numel() - arena.top > 300 * 1024
    assert v.lib.psk_light_teacher_build(v._p(v.scen), len(scens), 3, v._p(v._table), v._stream()) == 0
    block = nbytes // 2 // len(scens)
    assert torch.equal(v._table[:4 * block], ref.teacher_table()) and arena.guards_intact()
    cur = np.column_stack([st, np.zeros(n, np.int32)])
    v.set_state(_u8(cur))
    ref.set_state(_u8(cur[:len(si_s)]))

    def lookup():
        rc = v.lib.psk_light_expert_table(v._p(v.scen), v._p(v.scen_idx), v._p(v.state), v._p(v._table), 3,
                                          v._p(act), v._p(dist), n, v._stream())
        assert rc == 0
        return act.cpu().numpy().astype(np.int64), dist.cpu().numpy().astype(np.int64)
    a, d = lookup()
    a_s, d_s = (t.cpu().numpy().astype(np.int64) for t in ref.expert())
    outside = st[:, 2] >= 8
    assert outside.sum() > 2500
    assert np.array_equal(a[:len(si_s)], a_s) and np.array_equal(d[:len(si_s)], d_s)
    assert (a[outside] == 255).all() and (d[outside] == -2).all()
    assert np.isin(a, ALLOWED).all() and arena.guards_intact()
    # the same envs through the search kernel (max_keys 3: the 8-key scenario is not searched)
    a_q, d_q = (t.cpu().numpy().astype(np.int64) for t in v.expert(search=True))
    assert np.array_equal(a_q[:len(si_s)], a_s) and np.array_equal(d_q[:len(si_s)], d_s)
    assert (a_q[len(si_s):] == 255).all() and (d_q[len(si_s):] == -2).all()
    # tick from these states, teacher-driven and forced, then reset puts every 8-key env outside
    _, _, act_s = table_views(v)
    for a_in in (None, rng.randint(0, 5, n)):
        v.set_state(_u8(cur))
        got = v.tick(actions=None if a_in is None else _u8(a_in), features_out=feats, out=out, max_timesteps=50)
        want = replay_tick(o, act_s, np.asarray([[c.init_x, c.init_y, (1 << c.n_keys) - 1] for c in recs]),
                           si, cur, a_in, 50)
        _check_tick(got, v, want, a_in is None)
        assert arena.guards_intact()
    v.reset()
    a, d = lookup()
    assert (a[si == 4] == 255).all() and (d[si == 4] == -2).all()
    got = v.rollout(3, max_timesteps=50)
    assert (got["expert"].cpu().numpy()[:, si == 4] == 255).all() and got["done"].cpu().numpy()[:, si == 4].all()
    # mask bits the scenario does not have: set_state refuses them, the kernels stay inside the table
    bad = cur.copy()
    bad[:len(si_s), 2] |= 0x80
    before = v.state.clone()
    with pytest.raises(ValueError, match="bits at or above"):
        v.set_state(_u8(bad))
    assert torch.equal(v.state, before)
    v.state.copy_(torch.from_numpy(_u8(bad)).to(v.device))
    a, d = lookup()
    assert (a[:len(si_s)] == 255).all() and (d[:len(si_s)] == -2).all() and arena.guards_intact()
    a_q, d_q = (t.cpu().numpy().astype(np.int64) for t in v.expert(search=True))
    assert (a_q == 255).all() and (d_q == -2).all()


def test_veclight_rejects_states_it_has_no_table_entry_for(W):
    from psketch_b200.worlds.light import VecLight
    names = dict(synthetic_set())
    v = VecLight([names["no_keys"], names["goal_row_4"]], [0, 1, 1])
    good = np.asarray([[18, 6, 0, 0], [6, 30, 7, 254], [1, 1, 0, 3]], np.uint8)
    v.set_state(good)
    for row, col, val, what in ((0, 0, 19, "off its 19 x 7 board"), (0, 1, 7, "off its 19 x 7 board"),
                                (0, 2, 1, "bits at or above its scenario's 0 keys"),
                                (1, 2, 8, "bits at or above its scenario's 3 keys"),
                                (2, 3, 255, "step counter 255")):
        bad = good.copy()
        bad[row, col] = val
        with pytest.raises(ValueError, match=what):
            v.set_state(bad)
        assert np.array_equal(v.state.cpu().numpy(), good)
    with pytest.raises(ValueError, match="scenario indices"):
        v.scen_idx = [0, 2, 1]
    assert v.scen_idx.cpu().numpy().tolist() == [0, 1, 1]
