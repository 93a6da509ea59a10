"""Light world beyond the 60 reference scenarios, host side (no GPU): the scenario sets that
tests/test_light_limits_gpu.py runs the kernels on, and the input checks of VecLight.

Two sets.  The GENERATOR set is drawn from LightWorld with reseeded random streams: three draws of
each of the 17 goals, then whatever draws a seed search finds for the board shapes and goal rooms the
first draws missed and for the rare six- and seven-key draws.  The SYNTHETIC set is built directly as
psk_light_scenario records and reaches what the C ABI accepts but the generator never makes: 8 keys
and 8 doors on a 31 x 31 board, goal rooms in column / row 4, several keys for one door, keys whose
target is no door, keys on room-wall and door cells, two doors on one cell, several keys on one cell.
"""
import functools

import numpy as np
import pytest

from psketch_b200.worlds.light import LIGHT_GOALS, ROOM_H, ROOM_W, LightScenario, LightWorld, _walk


def _extent(goal):
    l = r = u = d = 0
    for x, y in _walk(goal):
        l, r, u, d = min(l, x), max(r, x), min(u, y), max(d, y)
    return l, r, u, d


def generator_limits():
    """Every board shape and goal room LightWorld.sample_scenario_with_goal can draw: each side of
    the goal path's bounding box grows by randint(2) rooms (worlds/light.py:65-68)."""
    shapes, rooms = set(), set()
    for g in LIGHT_GOALS:
        l, r, u, d = _extent(g)
        gx, gy = list(_walk(g))[-1]
        for el, er, eu, ed in np.ndindex(2, 2, 2, 2):
            shapes.add((ROOM_W * (r - l + 1 + el + er) + 1, ROOM_H * (d - u + 1 + eu + ed) + 1))
            rooms.add((-l + el + gx, -u + eu + gy))
    return shapes, rooms


def _draw(goal, seed):
    w = LightWorld()
    w.random = np.random.RandomState(seed)
    return w.sample_scenario_with_goal(goal)


@functools.lru_cache(maxsize=None)
def generator_set():
    """[(goal, seed, LightScenario)]: draws of the host generator picked by searching seeds."""
    out = [(g, seed, _draw(g, seed)) for g in LIGHT_GOALS for seed in range(3)]
    shapes, rooms = generator_limits()
    seen_s = {sc.walls.shape for _, _, sc in out}
    seen_r = {tuple(sc.goal_room) for _, _, sc in out}
    seed = 3
    while not (shapes <= seen_s and rooms <= seen_r):
        for g in LIGHT_GOALS:
            sc = _draw(g, seed)
            if sc.walls.shape not in seen_s or tuple(sc.goal_room) not in seen_r:
                out.append((g, seed, sc))
                seen_s.add(sc.walls.shape)
                seen_r.add(tuple(sc.goal_room))
        seed += 1
    # six or seven keys: seven need seven doors, the three of a three-room goal path and four extra
    # ones, and each door gets its key with probability 1/2 -- about one draw in a thousand
    want = {6: 2, 7: 2}
    seed = 0
    while any(want.values()):
        for g in (g for g in LIGHT_GOALS if len(g) == 3):
            sc = _draw(g, seed)
            if want.get(len(sc.keys)):
                want[len(sc.keys)] -= 1
                out.append((g, seed, sc))
        seed += 1
    return tuple(out)


class KeyList(list):
    """Keys as a list of ((kx, ky), (door x, door y)): unlike the reference's dict keyed by position
    it can hold several keys on one cell.  LightScenario.to_c only needs ``items()`` and ``len``."""

    def items(self):
        return list(self)


def board(rooms_x, rooms_y):
    walls = np.zeros((ROOM_W * rooms_x + 1, ROOM_H * rooms_y + 1))
    walls[0::ROOM_W, :] = 1
    walls[:, 0::ROOM_H] = 1
    return walls


def door_right(rx, ry):
    """The door cell between room (rx, ry) and room (rx + 1, ry)."""
    return (ROOM_W * (rx + 1), ROOM_H * ry + ROOM_H // 2)


def door_down(rx, ry):
    """The door cell between room (rx, ry) and room (rx, ry + 1)."""
    return (ROOM_W * rx + ROOM_W // 2, ROOM_H * (ry + 1))


def cell(rx, ry, i, j):
    """Interior cell (i, j) in 0..4 of room (rx, ry)."""
    return (ROOM_W * rx + 1 + i, ROOM_H * ry + 1 + j)


def scenario(walls, doors, keys, init_room, goal_room):
    walls = walls.copy()
    for d in doors:
        walls[d] = 0
    return LightScenario(walls, list(doors), KeyList(keys), init_room, goal_room, None)


def _eight_key_path(rng):
    """8 keys and 8 doors on a 31 x 31 board, goal room in the far corner: a path of rooms
    (0,0) .. (4,0) .. (4,4); the key of the k-th door lies in a random room before it."""
    path = [(x, 0) for x in range(5)] + [(4, y) for y in range(1, 5)]
    doors = [door_right(*path[k]) if path[k + 1][1] == path[k][1] else door_down(*path[k]) for k in range(8)]
    keys, used = [], set()
    for k in range(8):
        while True:
            c = cell(*path[rng.randint(k + 1)], rng.randint(5), rng.randint(5))
            if c not in used:
                break
        used.add(c)
        keys.append((c, doors[k]))
    return scenario(board(5, 5), doors, keys, (0, 0), (4, 4))


def _eight_key_random(rng):
    """8 of the 40 inner doors of a 5 x 5-room board and 8 keys in random rooms, two of them on one
    cell; most key subsets and many rooms cannot reach the goal room (4, 2)."""
    all_doors = [door_right(x, y) for x in range(4) for y in range(5)] + \
                [door_down(x, y) for x in range(5) for y in range(4)]
    doors = [all_doors[i] for i in rng.choice(len(all_doors), 8, replace=False)]
    cells = [cell(rng.randint(5), rng.randint(5), rng.randint(5), rng.randint(5)) for _ in range(7)]
    cells.append(cells[3])
    keys = [(cells[k], doors[rng.randint(8)]) for k in range(8)]
    return scenario(board(5, 5), doors, keys, (0, 4), (4, 2))


@functools.lru_cache(maxsize=None)
def synthetic_set():
    """[(name, scenario)] of records the C ABI accepts and the generator never makes."""
    rng = np.random.RandomState(11)
    out = [("eight_keys_path", _eight_key_path(rng)), ("eight_keys_random", _eight_key_random(rng))]
    # goal room in row 4 of a 1 x 5-room board (7 x 31)
    doors = [door_down(0, y) for y in range(4)]
    out.append(("goal_row_4", scenario(board(1, 5), doors, [(cell(0, 0, 4, 4), doors[0]),
                                                            (cell(0, 1, 0, 0), doors[1]),
                                                            (cell(0, 0, 2, 2), doors[3])], (0, 0), (0, 4))))
    # two keys lock door A, three keys lock door B; a key whose target is an interior cell and one
    # whose target is a wall cell; a key-free detour (0,0) -> (0,1) -> (1,1)
    A, B, C = door_right(0, 0), door_down(1, 0), door_right(1, 1)
    doors = [A, B, C, door_down(0, 0), door_right(0, 1)]
    keys = [(cell(0, 0, 0, 4), A), (cell(0, 0, 4, 0), A), (cell(0, 0, 1, 1), B), (cell(1, 0, 2, 2), B),
            (cell(0, 1, 3, 3), B), (cell(0, 0, 2, 2), cell(1, 1, 2, 2)), (cell(1, 0, 0, 0), (6, 1))]
    out.append(("shared_doors", scenario(board(3, 3), doors, keys, (0, 0), (2, 1))))
    # a key on an opening of a room wall that is no door (its feature is 0), a key on a door cell,
    # two doors on one cell (both locked by one key)
    walls = board(2, 2)
    walls[6, 1] = 0                                              # opening between (0,0) and (1,0)
    D0, D1, D2 = door_right(0, 0), door_down(0, 0), door_down(1, 0)
    keys = [((6, 1), D1), (D0, D2), (cell(0, 0, 3, 3), D0), (cell(1, 0, 1, 1), D2)]
    out.append(("wall_and_door_keys", scenario(walls, [D0, D1, D2, D2], keys, (0, 0), (1, 1))))
    # the only way into the goal room is a door whose key lies inside it
    D = door_right(0, 0)
    out.append(("key_behind_its_door", scenario(board(2, 1), [D], [(cell(1, 0, 2, 2), D), (cell(0, 0, 0, 0), D)],
                                                (0, 0), (1, 0))))
    # init room = goal room
    D = door_down(1, 0)
    out.append(("init_is_goal", scenario(board(2, 2), [D, door_right(0, 1)], [(cell(1, 1, 1, 1), D)], (1, 0), (1, 0))))
    # no keys at all, next to the 8-key ones in the same batch
    out.append(("no_keys", scenario(board(3, 1), [door_right(0, 0), door_right(1, 0)], [], (0, 0), (2, 0))))
    # two keys on one cell and three keys on another (two of those for the same door): one USE
    # picks up every key lying on the cell
    D0, D1, D2, D3 = door_right(0, 0), door_down(0, 0), door_right(1, 0), door_down(2, 0)
    doors = [D0, D1, D2, D3, door_right(0, 1), door_right(1, 1)]
    k1, k2 = cell(0, 0, 1, 1), cell(1, 0, 2, 2)
    keys = [(k1, D0), (k1, D1), (k2, D2), (k2, D3), (k2, D2), (cell(0, 1, 0, 0), door_right(1, 1))]
    out.append(("colocated_keys", scenario(board(3, 2), doors, keys, (0, 0), (2, 1))))
    # goal room in column 4, keys everywhere on the way, on a 31 x 13 board
    doors = [door_right(x, 0) for x in range(4)] + [door_down(2, 0), door_right(2, 1), door_right(3, 1)]
    keys = [(cell(x, 0, x, 4 - x), doors[x]) for x in range(4)] + [(cell(2, 1, 1, 1), doors[6])]
    out.append(("goal_column_4", scenario(board(5, 2), doors, keys, (0, 0), (4, 1))))
    return tuple(out)


def records(scens):
    return [s.to_c() for s in scens]


# ---------------------------------------------------------------------------------------------


def test_generator_set_reaches_the_generator_limits():
    gen = generator_set()
    shapes, rooms = generator_limits()
    assert {sc.walls.shape for _, _, sc in gen} == shapes and len(shapes) == 21
    assert {(7, 31), (31, 7), (13, 31)} <= shapes
    assert {tuple(sc.goal_room) for _, _, sc in gen} == rooms
    assert {(0, 3), (3, 0), (3, 1)} <= rooms
    per_goal = {g: sum(1 for g2, _, _ in gen if g2 == g) for g in LIGHT_GOALS}
    assert min(per_goal.values()) >= 3 and len(per_goal) == 17
    n_keys = [len(sc.keys) for _, _, sc in gen]
    assert max(n_keys) == 7 and n_keys.count(7) >= 2 and n_keys.count(6) >= 2
    assert max(len(sc.doors) for _, _, sc in gen) == 7
    # the seed search reproduces: a draw depends only on (goal, seed)
    g, seed, sc = gen[-1]
    again = _draw(g, seed)
    assert np.array_equal(again.walls, sc.walls) and again.keys == sc.keys and again.doors == sc.doors


def test_synthetic_set_covers_the_abi_edges():
    recs = dict((name, sc.to_c()) for name, sc in synthetic_set())
    assert len(recs) == len(synthetic_set())

    def keys(c):
        return [tuple(c.keys[4 * k:4 * k + 4]) for k in range(c.n_keys)]

    def doors(c):
        return [tuple(c.doors[2 * d:2 * d + 2]) for d in range(c.n_doors)]
    big = recs["eight_keys_path"]
    assert (big.n_keys, big.n_doors, big.board_w, big.board_h) == (8, 8, 31, 31)
    assert recs["eight_keys_random"].n_keys == 8
    assert any(c.goal_rx == 4 for c in recs.values()) and any(c.goal_ry == 4 for c in recs.values())
    targets = [k[2:] for k in keys(recs["shared_doors"])]
    assert sorted(targets.count(t) for t in set(targets))[-2:] == [2, 3]
    assert any(t not in doors(recs["shared_doors"]) for t in targets)
    wk = recs["wall_and_door_keys"]
    on = [k[:2] for k in keys(wk)]
    assert (6, 1) in on and (6, 1) not in doors(wk) and any(p in doors(wk) for p in on)
    assert len(doors(wk)) - len(set(doors(wk))) == 1
    ii = recs["init_is_goal"]
    assert (ii.init_x // ROOM_W, ii.init_y // ROOM_H) == (ii.goal_rx, ii.goal_ry)
    assert recs["no_keys"].n_keys == 0
    on = [k[:2] for k in keys(recs["colocated_keys"])]
    assert sorted(on.count(p) for p in set(on))[-2:] == [2, 3]
    assert sum(on.count(p) for p in set(on) if on.count(p) > 1) >= 2


def test_oracle_use_picks_up_every_key_on_the_cell():
    """light_oracle.c (pinned against the reference) removes every live key underfoot in one USE;
    the reference cannot hold two keys on one cell, so this is the rule the kernels follow."""
    name, sc = [x for x in synthetic_set() if x[0] == "colocated_keys"][0]
    o = oracle_of(records([sc]))
    kx, ky = sc.keys[2][0]
    _, _, nxt = o.run(np.zeros(2, np.int32), np.asarray([[kx, ky, 0x3F], [kx, ky, 0x2B]]), np.full(2, 4))
    assert nxt.tolist() == [[kx, ky, 0x23], [kx, ky, 0x23]]


def oracle_of(recs):
    """LightOracle over psk_light_scenario records (walls beyond the board are 1, as to_c pads them)."""
    from oracle.light_oracle import LightOracle
    S = len(recs)
    rows = np.asarray([list(c.walls) for c in recs], np.uint64).reshape(S, 32)
    walls = ((rows[:, :, None] >> np.arange(32, dtype=np.uint64)[None, None, :]) & 1).astype(np.uint8)
    assert walls[:, 31, :].all() and walls[:, :, 31].all()
    doors = np.asarray([list(c.doors) for c in recs], np.int32).reshape(S, 8, 2)
    keys = np.asarray([list(c.keys) for c in recs], np.int32).reshape(S, 8, 4)
    return LightOracle(walls[:, :31, :31], np.asarray([[c.board_w, c.board_h] for c in recs]), doors,
                       [c.n_doors for c in recs], keys, [c.n_keys for c in recs],
                       np.asarray([[c.goal_rx, c.goal_ry] for c in recs]))


def test_check_light_inputs():
    from psketch_b200 import _lib
    board = np.asarray([[13, 7], [31, 31]])
    n_keys = np.asarray([2, 8])
    si = np.asarray([0, 1, 1])
    good = np.asarray([[12, 6, 3, 0], [30, 30, 255, 254], [0, 0, 0, 17]])
    _lib.check_light_inputs(board, n_keys, si, good)
    _lib.check_light_inputs(board, n_keys, [], np.zeros((0, 4)))
    with pytest.raises(ValueError, match="scenario indices"):
        _lib.check_light_inputs(board, n_keys, [0, 2])
    with pytest.raises(ValueError, match="scenario indices"):
        _lib.check_light_inputs(board, n_keys, [-1, 0])
    for col, val, what in ((0, 13, "off its 13 x 7 board"), (1, 7, "off its 13 x 7 board"),
                           (2, 4, "bits at or above its scenario's 2 keys"),
                           (3, 255, "step counter 255")):
        bad = good.copy()
        bad[0, col] = val
        with pytest.raises(ValueError, match=what):
            _lib.check_light_inputs(board, n_keys, si, bad)
    with pytest.raises(ValueError, match="0..255"):
        _lib.check_light_inputs(board, n_keys, si, good + [[0, 0, 0, -1], [0] * 4, [0] * 4])
    with pytest.raises(ValueError, match="0..255"):
        _lib.check_light_inputs(board, n_keys, si, good + [[0, 0, 300, 0], [0] * 4, [0] * 4])
    with pytest.raises(ValueError, match="shape"):
        _lib.check_light_inputs(board, n_keys, si, good[:2])
    with pytest.raises(ValueError, match="whole numbers"):
        _lib.check_light_inputs(board, n_keys, si, good + 0.5)


def test_veclight_checks_scenario_indices_before_any_device_work():
    from psketch_b200.worlds.light import VecLight
    scens = [sc for _, sc in synthetic_set()]
    with pytest.raises(ValueError, match="scenario indices"):
        VecLight(scens, [0, len(scens)])
    with pytest.raises(ValueError, match="scenario indices"):
        VecLight(scens, [-1])
