"""The C oracle (oracle/craft_oracle.c) against the restatement of the reference's numpy code
(oracle/craft_ref_port.py) at geometries no other test covers: non-square grids, thin boards and
non-square odd windows.  The GPU tests of the generic tier (tests/test_generic_geometry_gpu.py)
compare the kernels with the oracle, so this pins the oracle itself there: features, step for all
six actions, satisfies for every task, and the teacher.

Boards stay at most 250 cells, so that the port's 1000-slot BFS queue (teachers/base.py:42) holds
every (position, direction) state.  Also checked without a GPU: the library's answer to
psk_craft_supported / psk_craft_n_features over the generic domain, and that even windows, which the
library rejects, break the reference's own features()."""
import ctypes
import functools
import os

import numpy as np
import pytest

from oracle.craft_ref_port import MOVES, PortTeacher, PortWorld

CUSTOM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "custom")

# (W, H, window_w, window_h)
GEOMETRIES = [(5, 7, 1, 3), (7, 4, 3, 5), (6, 9, 5, 1), (3, 11, 3, 3), (2, 9, 3, 1), (9, 5, 7, 3),
              (12, 3, 9, 5), (1, 6, 3, 3), (15, 13, 3, 9)]
BOOKS = ("stock", "custom")


@functools.lru_cache(maxsize=None)
def generic_tables(W, H, ww, wh, book="stock"):
    from psketch_b200.tables import Cookbook, CraftTables, TaskManager
    cfg = dict(WIDTH=W, HEIGHT=H, WINDOW_WIDTH=ww, WINDOW_HEIGHT=wh, N_WORKSHOPS=3, N_PRIMITIVES=1, N_WORLDS=1)
    if book == "stock":
        return CraftTables(world_config=cfg)
    return CraftTables(Cookbook(os.path.join(CUSTOM, "recipes.yaml")),
                       TaskManager(os.path.join(CUSTOM, "hints.yaml")), cfg)


def good_tasks(tables):
    """Task ids whose teacher answer is defined everywhere (no leaf other than use / go)."""
    return [t.task_id for t in tables.task_manager.tasks if t.goal_name in ("get", "make", "makeat", "go")]


def board_states(tables, n, seed, density=0.3, ring=False):
    """n states on any board, thin ones included: a random fill of every kind but 0 at `density`
    (inside a boundary ring with `ring`), the agent on a free cell facing any way, small inventories (a
    fifth of the envs hold counts up to 255 on every kind), and tasks the teacher answers."""
    rng = np.random.RandomState(seed)
    W, H, K = tables.W, tables.H, tables.K
    grid = np.where(rng.rand(n, W * H) < density, rng.randint(1, K, size=(n, W * H)), 0).astype(np.uint8)
    lo = 1 if ring else 0
    pos = np.stack([rng.randint(lo, W - lo, n), rng.randint(lo, H - lo, n)], 1).astype(np.int32)
    if ring:
        g = grid.reshape(n, W, H)
        g[:, 0, :] = g[:, W - 1, :] = g[:, :, 0] = g[:, :, H - 1] = tables.cookbook.index["boundary"]
    grid[np.arange(n), pos[:, 0] * H + pos[:, 1]] = 0
    inv = (rng.randint(0, 3, size=(n, K)) * (rng.rand(n, K) < 0.3)).astype(np.int32)
    inv[::5] = rng.randint(0, 256, size=inv[::5].shape)
    inv[:, 0] = 0
    return dict(grid=grid, inv=inv, pos=pos, dir=rng.randint(0, 4, n).astype(np.int32),
                task=rng.choice(good_tasks(tables), size=n).astype(np.int32))


def _port_states(tables, S):
    world = PortWorld(tables)
    out = []
    for i in range(len(S["grid"])):
        s = world.init_state(world.onehot(S["grid"][i]), S["pos"][i], int(S["dir"][i]))
        s.inventory = S["inv"][i].astype(np.float64)
        out.append(s)
    return out


def _ids(tables, port_state):
    """Port one-hot grid -> kind ids u8[W*H] (x-major)."""
    g = port_state.grid
    return (g.argmax(axis=2) * (g.max(axis=2) > 0)).reshape(-1).astype(np.uint8)


@pytest.fixture(params=GEOMETRIES, ids=lambda g: "%dx%d_w%dx%d" % g)
def geometry(request):
    return request.param


@pytest.fixture(params=BOOKS)
def book(request):
    return request.param


def _setup(geometry, book, n=60, seed=0, ring=False):
    from oracle.craft_oracle import CraftOracle
    tables = generic_tables(*geometry, book=book)
    S = board_states(tables, n, seed=sum(geometry) * 7919 + len(book) * 31 + seed, ring=ring)
    return tables, CraftOracle(tables), S, _port_states(tables, S)


def test_features(geometry, book):
    tables, o, S, P = _setup(geometry, book)
    want = np.stack([p.features() for p in P]).astype(np.float32)
    got = o.features(S["grid"], S["inv"], S["pos"], S["dir"])
    assert got.shape == (len(P), tables.n_features)
    assert np.array_equal(got, want)


def test_step_every_action(geometry, book):
    tables, o, S, P = _setup(geometry, book)
    for a in range(6):
        g, inv, pos, d, status = o.step(S["grid"], S["inv"], S["pos"], S["dir"], np.full(len(P), a))
        assert (status == 0).all()
        for i, p in enumerate(P):
            if a < 4 and not (0 <= p.pos[0] + MOVES[a][0] < tables.W and 0 <= p.pos[1] + MOVES[a][1] < tables.H):
                continue        # the reference indexes off the grid here; the oracle blocks (documented)
            _, q = p.step(a)
            assert np.array_equal(g[i], _ids(tables, q)), (a, i)
            assert np.array_equal(inv[i], q.inventory.astype(np.int32)), (a, i)
            assert tuple(pos[i]) == tuple(q.pos) and d[i] == q.dir, (a, i)
    _, _, _, _, status = o.step(S["grid"], S["inv"], S["pos"], S["dir"], np.full(len(P), 6))
    assert (status == -1).all()
    with pytest.raises(Exception, match="Unexpected action"):
        P[0].step(6)


def test_satisfies_every_task(geometry, book):
    tables, o, S, P = _setup(geometry, book)
    tm = tables.task_manager
    for t in range(1, tables.n_tasks):
        got = o.satisfies(S["grid"], S["inv"], S["pos"], S["dir"], np.full(len(P), t))
        task = tm.by_id(t)
        for i, p in enumerate(P):
            x, y = p.pos
            dx, dy = MOVES[p.dir]
            if task.goal_name == "go" and not (0 <= x + dx < tables.W and 0 <= y + dy < tables.H):
                continue        # the reference indexes off the grid here; the oracle reads 0 (documented)
            want = p.satisfies(task)
            want = 2 if want is None else int(bool(want))
            assert got[i] == want, (t, i)


def test_teacher(geometry, book):
    """Inside a boundary ring (the reference's search indexes off the grid without one), so boards
    at least 3 cells wide each way."""
    if min(geometry[:2]) < 3:
        pytest.skip("no interior inside a boundary ring")
    tables, o, S, P = _setup(geometry, book, n=80, seed=1, ring=True)
    tm = tables.task_manager
    act, dist, status = o.expert(S["grid"], S["inv"], S["pos"], S["dir"], S["task"])
    teacher = PortTeacher()
    checked = 0
    for i, p in enumerate(P):
        if status[i] == 2:
            continue        # the reference raises TypeError (documented in craft_oracle.c)
        assert act[i] == teacher(tm.by_id(int(S["task"][i])), p), i
        checked += 1
    assert checked > len(P) // 2
    assert (act < 4).any() and (act == 5).any() and (dist > 0).any()


def test_even_windows_break_the_reference_features():
    """block_reduce pads a window of ww^2 + 1 cells per axis, and the reference's features() then
    fails its own length check; the port fails the same way (its block max only takes shapes that
    divide evenly).  This is why the library keeps windows odd."""
    for ww, wh in ((2, 3), (3, 4), (4, 4)):
        tables = generic_tables(7, 6, ww, wh)
        S = board_states(tables, 2, seed=ww * 10 + wh)
        with pytest.raises((AssertionError, ValueError)):
            _port_states(tables, S)[0].features()


def test_library_domain():
    """psk_craft_supported / psk_craft_n_features: 1 <= W, H <= 64, odd windows 1..9 per axis,
    1..24 kinds; everything else unsupported (-1 features)."""
    from psketch_b200 import _lib
    lib = _lib.load()
    base = _lib.make_tables(generic_tables(9, 9, 3, 3))

    def ask(**kw):
        c = _lib.CraftTablesC()
        ctypes.memmove(ctypes.byref(c), ctypes.byref(base), ctypes.sizeof(c))
        for k, v in kw.items():
            setattr(c, k, v)
        return lib.psk_craft_supported(ctypes.byref(c)), lib.psk_craft_n_features(ctypes.byref(c))

    K = base.n_kinds
    for W, H, ww, wh in [(1, 1, 1, 1), (64, 64, 9, 9), (2, 64, 9, 1), (64, 3, 1, 7), (20, 13, 3, 5),
                         (8, 8, 3, 3), (10, 10, 5, 5), (8, 8, 5, 5), (33, 17, 5, 5)]:
        assert ask(width=W, height=H, window_w=ww, window_h=wh) == (1, 2 * ww * wh * K + K + 5), (W, H, ww, wh)
    for kw in [dict(width=0), dict(height=65), dict(width=65), dict(window_w=2), dict(window_h=4),
               dict(window_w=11), dict(window_h=0), dict(window_w=-1), dict(n_kinds=25), dict(n_kinds=0)]:
        assert ask(**kw) == (0, -1), kw
