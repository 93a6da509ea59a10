"""Enlarged-grid Craft states (16x16, 32x32 and 64x64, BASELINE configs[4]) that reach the edges of
the warp-cooperative teacher kernels, checked without a GPU.

The kernels behind these sizes (psk_craft.cu: RowBoard / bfs_rows with one or two rows per lane,
HalfRows / bfs_half_rows with two envs per warp, craft_find_closest_rows_kernel, the windowed
feature gather) have edges that random boards rarely reach.  This module holds a seeded generator of
states in six families, shared with tests/test_stress_limits_gpu.py:

  random     the mix of tests/test_stress_gpu.py: a boundary ring, items, 15-40 % stone;
  maze       serpentine corridors with one- or two-cell gaps and one goal at the far end, reachable
             or walled off (distances above 255 on 32x32 and above 1,000 on 64x64);
  open       no obstacles, goal cells placed symmetric about the agent (mirrored in x, in y, and on
             both sides of a lane or slot boundary of the 64x64 layout): ties in the goal and in the
             first action;
  ringless   no boundary ring, agents on every edge cell facing every way, and 0-4 cells from
             each edge, items on the edges;
  leaf       the teacher's leaf is USE, STOP (task satisfied), GO short / long / unreachable, or
             the agent already faces the goal; ``paired_leaf_batch`` orders them so that envs 2i and
             2i+1 (one warp of the two-envs-per-warp kernel) cover every ordered pair of cases;
  inventory  counts up to 255 on every kind, the last kinds of the cookbook included.

The tests below check through the C oracle that each family reaches its edge, so that a generator
that stopped doing so fails here instead of weakening the GPU tests.
"""
import functools
import itertools
import os

import numpy as np
import pytest


SIZES = (16, 32, 64)
BOOKS = ("stock", "custom")
FAMILIES = ("random", "maze", "open", "ringless", "leaf", "inventory")
LEAF_CASES = ("use", "stop", "facing", "short", "long", "unreachable")
INV_COUNTS = (0, 1, 13, 127, 128, 200, 254, 255)
MOVES = ((0, -1), (0, 1), (-1, 0), (1, 0))          # DOWN, UP, LEFT, RIGHT (worlds/craft.py:77-91)
CUSTOM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "custom")


@functools.lru_cache(maxsize=None)
def stress_tables(size, book="stock"):
    """CraftTables of a size x size world, 3x3 window, with the stock or the custom cookbook
    (tests/golden/custom: 20 kinds, so the runtime-K feature kernels run)."""
    from psketch_b200.tables import Cookbook, CraftTables, TaskManager
    cfg = dict(WIDTH=size, HEIGHT=size, WINDOW_WIDTH=3, WINDOW_HEIGHT=3, N_WORKSHOPS=3,
               N_PRIMITIVES=size // 4, N_WORLDS=1)
    if book == "stock":
        return CraftTables(world_config=cfg)
    return CraftTables(Cookbook(os.path.join(CUSTOM, "recipes.yaml")),
                       TaskManager(os.path.join(CUSTOM, "hints.yaml")), cfg)


@functools.lru_cache(maxsize=None)
def stress_oracle(size, book="stock"):
    from oracle.craft_oracle import CraftOracle
    return CraftOracle(stress_tables(size, book))


def _kind(tables, name):
    return tables.cookbook.index[name]


def go_kinds(tables):
    """Kinds some hint leaf walks to (go[X]), in id order."""
    tm = tables.task_manager
    return sorted(set(_kind(tables, t.goal_arg) for t in tm.tasks if t.goal_name == "go"))


def task_id(tables, goal):
    return tables.task_manager[goal].task_id


def good_tasks(tables):
    """Task ids whose teacher answer is defined everywhere (no leaf other than use / go)."""
    return [t.task_id for t in tables.task_manager.tasks if t.goal_name in ("get", "make", "makeat", "go")]


def _go_task(tables, kind, rng):
    """A task whose first leaf is go[kind] on a state with nothing in the inventory."""
    name = tables.cookbook.index.get(kind)
    cands = ["go[%s]" % name, "get[%s]" % name, "makeat[%s]" % name]
    cands = [c for c in cands if c in tables.task_manager.tasks_by_goal]
    return task_id(tables, cands[rng.randint(len(cands))])


class _Batch(object):
    """States under construction: grid u8[n, W, H] kind ids, inventory, position, facing, task."""

    def __init__(self, tables, n, ring=True):
        self.t = tables
        W, H, K = tables.W, tables.H, tables.K
        self.grid = np.zeros((n, W, H), np.uint8)
        if ring:
            b = _kind(tables, "boundary")
            self.grid[:, 0, :] = self.grid[:, W - 1, :] = self.grid[:, :, 0] = self.grid[:, :, H - 1] = b
        self.inv = np.zeros((n, K), np.int32)
        self.pos = np.zeros((n, 2), np.int32)
        self.dir = np.zeros(n, np.int32)
        self.task = np.zeros(n, np.int32)
        self.target = np.zeros(n, np.int32)        # the kind the env's task walks to first (0: none)
        self.case = np.array([""] * n, dtype=object)

    def done(self, family):
        n = len(self.grid)
        for i in range(n):                          # the agent stands on a free cell
            self.grid[i, self.pos[i, 0], self.pos[i, 1]] = 0
        return dict(grid=self.grid.reshape(n, -1).copy(), inv=self.inv, pos=self.pos, dir=self.dir,
                    task=self.task, target=self.target, case=self.case, family=np.array([family] * n, dtype=object))


def _scatter(B, i, rng, free_cells, counts):
    """Places counts {kind: c} on random cells of free_cells (a list of (x, y)); returns the rest."""
    order = rng.permutation(len(free_cells))
    k = 0
    for kind, c in counts.items():
        for _ in range(c):
            if k >= len(order):
                return []
            x, y = free_cells[order[k]]
            B.grid[i, x, y] = kind
            k += 1
    return [free_cells[j] for j in order[k:]]


def _items(tables, rng, size, wall_frac):
    """Kind counts of the random mix: a few of every go-kind, water, and wall_frac stone."""
    W, H = tables.W, tables.H
    c = {}
    for name in ("iron", "grass", "wood"):
        c[_kind(tables, name)] = rng.randint(1, size // 2)
    for w in range(3):
        c[_kind(tables, "workshop%d" % w)] = 1
    if _kind(tables, "gem"):
        c[_kind(tables, "gem")] = rng.randint(0, 3)
    c[_kind(tables, "water")] = rng.randint(0, 4)
    c[_kind(tables, "stone")] = int(wall_frac * (W - 2) * (H - 2))
    return c


def _interior(W, H, ring=True):
    lo = 1 if ring else 0
    return [(x, y) for x in range(lo, W - lo) for y in range(lo, H - lo)]


def random_states(tables, n, seed):
    rng = np.random.RandomState(seed)
    W, H = tables.W, tables.H
    B = _Batch(tables, n)
    tasks = good_tasks(tables)
    cells = _interior(W, H)
    for i in range(n):
        rest = _scatter(B, i, rng, cells, _items(tables, rng, W, rng.uniform(0.15, 0.4)))
        B.pos[i] = rest[0]
        for _ in range(rng.randint(0, 4)):
            B.inv[i, rng.randint(7, tables.K)] += 1
    B.dir[:] = rng.randint(0, 4, size=n)
    B.task[:] = rng.choice(tasks, size=n)
    return B.done("random")


def _maze(B, i, rng, kind, reachable, transform):
    """Serpentine corridors: walls on every other column x = 2, 4, ..., W-4, each with a gap of one
    or two cells, alternately at the top and at the bottom; the agent starts in the first corridor,
    one goal cell of `kind` sits at the far end of the last one.  Not reachable: the last gap is
    closed.  `transform` (0-7) mirrors / transposes the board so corridors run both ways."""
    W, H = B.t.W, B.t.H
    wall = _kind(B.t, "boundary")
    stone = _kind(B.t, "stone")
    g = B.grid[i]
    xs = list(range(2, W - 3, 2))
    for j, x in enumerate(xs):
        g[x, 1:H - 1] = stone if rng.rand() < 0.3 else wall
        gap = rng.randint(1, 3)
        ys = range(H - 1 - gap, H - 1) if j % 2 == 0 else range(1, 1 + gap)
        if reachable or j < len(xs) - 1:
            for y in ys:
                g[x, y] = 0
    last_gap_top = (len(xs) - 1) % 2 == 0
    gx, gy = W - 2, (1 if last_gap_top else H - 2)
    g[gx, gy] = kind
    ax, ay = 1, rng.randint(1, H - 1)
    if transform & 1:
        g[:] = g[::-1, :].copy()
        gx, ax = W - 1 - gx, W - 1 - ax
    if transform & 2:
        g[:] = g[:, ::-1].copy()
        gy, ay = H - 1 - gy, H - 1 - ay
    if transform & 4:
        g[:] = g.T.copy()
        gx, gy, ax, ay = gy, gx, ay, ax
    B.pos[i] = (ax, ay)
    return gx, gy


def maze_states(tables, n, seed):
    """Half of them reachable; goal kinds and tasks vary."""
    rng = np.random.RandomState(seed)
    B = _Batch(tables, n)
    kinds = go_kinds(tables)
    for i in range(n):
        kind = kinds[rng.randint(len(kinds))]
        reachable = i % 2 == 0
        _maze(B, i, rng, kind, reachable, rng.randint(8))
        B.task[i] = _go_task(tables, kind, rng)
        B.target[i] = kind
        B.case[i] = "long" if reachable else "unreachable"
    B.dir[:] = rng.randint(0, 4, size=n)
    return B.done("maze")


def open_states(tables, n, seed):
    """An empty room; goal cells at the images of one offset under the mirrors about the agent, and
    (one env in two) goal pairs that straddle a lane / slot boundary of the 64-row layout: rows 2l and
    2l+1 (two slots of one lane) or 2l+1 and 2l+2 (two lanes), offset so that both are equally far.
    A quarter of the envs have the agent sealed in a box, so every goal is unreachable."""
    rng = np.random.RandomState(seed)
    W, H = tables.W, tables.H
    B = _Batch(tables, n)
    kinds = go_kinds(tables)
    wall = _kind(tables, "boundary")

    def put(i, x, y, kind):
        if 1 <= x < W - 1 and 1 <= y < H - 1 and (x, y) != tuple(B.pos[i]):
            B.grid[i, x, y] = kind

    for i in range(n):
        kind = kinds[rng.randint(len(kinds))]
        ax, ay = rng.randint(2, W - 2), rng.randint(2, H - 2)
        B.pos[i] = (ax, ay)
        if i % 2 == 0:
            r = max(2, min(W, H) // 2 - 1)
            dx, dy = rng.randint(0, r), rng.randint(0, r)
            if dx == 0 and dy == 0:
                dx = 1
            for sx, sy in ((1, 1), (-1, 1), (1, -1), (-1, -1)):
                if rng.rand() < 0.8:
                    put(i, ax + sx * dx, ay + sy * dy, kind)
        else:
            l = rng.randint(1, W // 2 - 2)
            x0 = 2 * l + rng.randint(2)                # rows (x0, x0 + 1): one lane or two
            ax = x0 + rng.randint(2)
            d = rng.randint(3, H // 2 - 1)
            ay = rng.randint(d + 1, H - d - 1)
            B.pos[i] = (ax, ay)
            s = rng.choice([-1, 1])
            # equally far from (ax, ay): (ax, ay + s d) and (other row, ay + s (d - 1))
            put(i, ax, ay + s * d, kind)
            put(i, 2 * x0 + 1 - ax, ay + s * (d - 1), kind)
            if rng.rand() < 0.5:
                put(i, ax, ay - s * d, kind)
        if i % 4 == 3:
            x, y = B.pos[i]
            for ddx in (-1, 0, 1):
                for ddy in (-1, 0, 1):
                    if (ddx or ddy) and 0 <= x + ddx < W and 0 <= y + ddy < H:
                        B.grid[i, x + ddx, y + ddy] = wall
        B.task[i] = _go_task(tables, kind, rng)
        B.target[i] = kind
    B.dir[:] = rng.randint(0, 4, size=n)
    return B.done("open")


def ringless_positions(W, H):
    """Every edge cell, then every cell 1-4 cells from an edge (and no nearer to another edge)."""
    edge = [(x, y) for x in range(W) for y in range(H) if min(x, y, W - 1 - x, H - 1 - y) == 0]
    near = [(x, y) for x in range(W) for y in range(H) if 1 <= min(x, y, W - 1 - x, H - 1 - y) <= 4]
    return edge, near


def ringless_states(tables, seed, n_near=None):
    """No boundary ring: the agent on every edge cell with every facing, then on cells 1-4 from an
    edge; items (go-kinds, water, stone) cover about 8 % of the cells, a third of them on the edges."""
    rng = np.random.RandomState(seed)
    W, H = tables.W, tables.H
    edge, near = ringless_positions(W, H)
    starts = [(p, d) for p in edge for d in range(4)]
    near = [near[j] for j in rng.permutation(len(near))[:n_near or len(near)]]
    starts += [(p, rng.randint(4)) for p in near]
    n = len(starts)
    B = _Batch(tables, n, ring=False)
    kinds = go_kinds(tables) + [_kind(tables, "water"), _kind(tables, "stone")]
    tasks = good_tasks(tables)
    cells = _interior(W, H, ring=False)
    for i, (p, d) in enumerate(starts):
        m = int(0.08 * W * H)
        for _ in range(m):
            if rng.rand() < 0.33:
                x, y = edge[rng.randint(len(edge))]
            else:
                x, y = cells[rng.randint(len(cells))]
            B.grid[i, x, y] = kinds[rng.randint(len(kinds))]
        B.pos[i], B.dir[i] = p, d
        kind = go_kinds(tables)[rng.randint(len(go_kinds(tables)))]
        B.task[i] = _go_task(tables, kind, rng) if rng.rand() < 0.7 else rng.choice(tasks)
        B.target[i] = kind
    return B.done("ringless")


def _front(tables, x, y, d):
    fx, fy = x + MOVES[d][0], y + MOVES[d][1]
    return (fx, fy) if 0 <= fx < tables.W and 0 <= fy < tables.H else None


def leaf_states(tables, case, n, seed):
    """n states whose teacher leaf is `case` (LEAF_CASES), on a sparse random board with a ring:
      use          task get[X] / makeat[X] while facing X: the go leaf is done, USE;
      stop         task get[X] with X in the inventory: nothing left to do, STOP;
      facing       task go[X] while facing X (satisfied, STOP); find_closest(X) has length 0;
      short        X 1-3 steps away;
      long         the far end of a serpentine maze;
      unreachable  X exists, walled off."""
    rng = np.random.RandomState(seed)
    W, H = tables.W, tables.H
    B = _Batch(tables, n)
    cells = _interior(W, H)
    grab = [_kind(tables, k) for k in ("wood", "iron", "grass")]
    shops = [_kind(tables, "workshop%d" % w) for w in range(3)]
    wall = _kind(tables, "boundary")
    for i in range(n):
        kind = (grab + shops)[rng.randint(6)] if case in ("use", "facing", "short", "unreachable") else \
            grab[rng.randint(3)]
        if case in ("long", "unreachable") and (case == "long" or i % 2):
            _maze(B, i, rng, kind, case == "long", rng.randint(8))
        else:
            c = _items(tables, rng, W, 0.1)
            c = {k: v for k, v in c.items() if k != kind}
            rest = _scatter(B, i, rng, cells, c)
            ax, ay = rng.randint(2, W - 2), rng.randint(2, H - 2)
            B.pos[i] = (ax, ay)
            d = rng.randint(4)
            B.dir[i] = d
            B.grid[i, ax, ay] = 0
            if case in ("use", "facing"):
                fx, fy = _front(tables, ax, ay, d)
                B.grid[i, fx, fy] = kind
            elif case == "short":                       # a clear 7x7 box around the agent
                B.grid[i, max(1, ax - 3):min(W - 1, ax + 4), max(1, ay - 3):min(H - 1, ay + 4)] = 0
                while True:
                    ox, oy = rng.randint(-3, 4), rng.randint(-3, 4)
                    if (1 <= abs(ox) + abs(oy) <= 3 and (ox, oy) != MOVES[d]
                            and 1 <= ax + ox < W - 1 and 1 <= ay + oy < H - 1):
                        break
                B.grid[i, ax + ox, ay + oy] = kind
            elif case == "unreachable":                 # every X cell boxed in
                for (x, y) in rest[:rng.randint(1, 4)]:
                    if 2 <= x < W - 2 and 2 <= y < H - 2 and max(abs(x - ax), abs(y - ay)) > 1:
                        B.grid[i, x - 1:x + 2, y - 1:y + 2] = wall
                        B.grid[i, x, y] = kind
                if not (B.grid[i] == kind).any():
                    B.grid[i, W - 3:W, H - 3:H] = wall
                    B.grid[i, W - 2, H - 2] = kind
            elif case == "stop":                        # somewhere, not in front of the agent
                fx, fy = _front(tables, ax, ay, d)
                x, y = rng.randint(1, W - 1), rng.randint(1, H - 1)
                if (x, y) not in ((ax, ay), (fx, fy)):
                    B.grid[i, x, y] = kind
        if case in ("use", "stop", "short", "long", "unreachable"):
            names = ["get[%s]", "makeat[%s]"] if case in ("use", "short", "unreachable") else ["get[%s]"]
            goals = [g % tables.cookbook.index.get(kind) for g in names]
            goals = [g for g in goals if g in tables.task_manager.tasks_by_goal]
            B.task[i] = task_id(tables, goals[rng.randint(len(goals))])
        else:
            B.task[i] = task_id(tables, "go[%s]" % tables.cookbook.index.get(kind))
        if case == "stop":
            B.inv[i, kind] = rng.choice(INV_COUNTS[1:])
        if case in ("long", "unreachable") and B.dir[i] == 0 and (case == "long" or i % 2):
            B.dir[i] = rng.randint(4)
        B.target[i] = kind
        B.case[i] = case
    return B.done("leaf")


def paired_leaf_batch(tables, reps, seed):
    """Envs 2i and 2i+1 run in one warp of the two-envs-per-warp teacher: this batch covers every
    ordered pair of LEAF_CASES `reps` times.  Returns the states with ``case`` per env."""
    pairs = list(itertools.product(LEAF_CASES, LEAF_CASES)) * reps
    need = {c: 2 * len(pairs) for c in LEAF_CASES}
    pool = {c: leaf_states(tables, c, need[c] // len(LEAF_CASES), seed + 101 * j)
            for j, c in enumerate(LEAF_CASES)}
    take = {c: 0 for c in LEAF_CASES}
    idx = []
    for a, b in pairs:
        for c in (a, b):
            idx.append((c, take[c]))
            take[c] += 1
    return concat([{k: v[[j]] for k, v in pool[c].items()} for c, j in idx])


def inventory_states(tables, n, seed):
    """The random mix with counts from INV_COUNTS on every kind; every tenth env holds 255 of each of
    the last three kinds of the cookbook."""
    S = random_states(tables, n, seed)
    rng = np.random.RandomState(seed + 1)
    K = tables.K
    inv = rng.choice(INV_COUNTS, size=(n, K)).astype(np.int32)
    inv *= rng.rand(n, K) < 0.6
    inv[:len(INV_COUNTS)] = np.array(INV_COUNTS)[:, None]
    inv[::10, K - 3:] = 255
    inv[:, 0] = 0
    S["inv"] = inv
    S["family"][:] = "inventory"
    return S


def concat(parts):
    return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}


def take(S, idx):
    return {k: v[idx] for k, v in S.items()}


# envs per family and grid size (leaf: repetitions of the 36 pairs; ringless: envs besides the edge
# cells): the 64x64 mazes are long (thousands of steps), so fewer
FAMILY_N = {16: dict(random=300, maze=64, open=256, leaf=1, inventory=200, ringless=200),
            32: dict(random=200, maze=48, open=192, leaf=1, inventory=120, ringless=120),
            64: dict(random=100, maze=24, open=128, leaf=1, inventory=60, ringless=60)}


@functools.lru_cache(maxsize=None)
def family(size, book, name, seed=0):
    """One family of states for the tables (size, book), seeded; cached for the test session."""
    tables = stress_tables(size, book)
    n = FAMILY_N[size][name]
    s = 1000 * size + 17 * seed + (7 if book == "custom" else 0)
    if name == "random":
        return random_states(tables, n, s + 1)
    if name == "maze":
        return maze_states(tables, n, s + 2)
    if name == "open":
        return open_states(tables, n, s + 3)
    if name == "ringless":
        return ringless_states(tables, s + 4, n_near=n)
    if name == "leaf":
        return paired_leaf_batch(tables, n, s + 5)
    if name == "inventory":
        return inventory_states(tables, n, s + 6)
    raise KeyError(name)


def all_families(size, book, seed=0):
    return concat([family(size, book, f, seed) for f in FAMILIES])


# ------------------------------------------------------------------------------------------------
# per-goal distances and first actions through the oracle (for the tie and edge checks)

def goal_distances(oracle, S, kinds):
    """For every env i and every cell of kinds[i]: the oracle's path length to that cell alone (the
    other cells of the kind turned into boundary, so occupancy is unchanged).  Returns a list of
    arrays of (x, y, length) per env."""
    H = oracle.H
    wall = oracle.tables.cookbook.index["boundary"]
    rows, owner, cell = [], [], []
    for i in range(len(S["grid"])):
        g = S["grid"][i]
        cs = np.flatnonzero(g == kinds[i])
        for c in cs:
            h = g.copy()
            h[cs] = wall
            h[c] = kinds[i]
            rows.append(h)
            owner.append(i)
            cell.append(c)
    out = [np.zeros((0, 3), np.int64) for _ in range(len(S["grid"]))]
    if not rows:
        return out
    owner = np.array(owner)
    _, length, _, _ = oracle.find_closest(np.stack(rows), S["pos"][owner], S["dir"][owner], kinds[owner], seq_cap=0)
    cell = np.array(cell)
    for i in np.unique(owner):
        m = owner == i
        out[i] = np.stack([cell[m] // H, cell[m] % H, length[m]], axis=1)
    return out


def first_action_ties(oracle, S, kinds):
    """Number of first actions (0-3) that start a shortest path to the nearest cell of kinds[i]."""
    n = len(S["grid"])
    _, length, st, _ = oracle.find_closest(S["grid"], S["pos"], S["dir"], kinds, seq_cap=0)
    good = np.zeros(n, np.int64)
    for a in range(4):
        g, _, p, d, _ = oracle.step(S["grid"], S["inv"], S["pos"], S["dir"], np.full(n, a))
        _, l2, _, _ = oracle.find_closest(g, p, d, kinds, seq_cap=0)
        good += (length > 0) & (l2 >= 0) & (l2 + 1 == length)
    return good, length, st


def tie_counts(size, book, name):
    """(envs with two or more goal cells at the minimum distance, envs with two or more first
    actions on a shortest path, at 64x64 goal ties inside one lane / across a lane boundary)."""
    S = family(size, book, name)
    o = stress_oracle(size, book)
    kinds = np.where(S["target"] > 0, S["target"], _kind(o.tables, "wood")).astype(np.int32)
    per = goal_distances(o, S, kinds)
    goal_ties = slot_ties = lane_ties = 0
    for d in per:
        ok = d[d[:, 2] >= 0]
        if len(ok) == 0:
            continue
        best = ok[ok[:, 2] == ok[:, 2].min()]
        if len(best) > 1:
            goal_ties += 1
            xs = set(best[:, 0].tolist())
            slot_ties += any(x % 2 == 0 and x + 1 in xs for x in xs)
            lane_ties += any(x % 2 == 1 and x + 1 in xs for x in xs)
    good, _, _ = first_action_ties(o, S, kinds)
    return goal_ties, int((good > 1).sum()), slot_ties, lane_ties


# ------------------------------------------------------------------------------------------------
# the families reach their edges

@pytest.mark.parametrize("book", BOOKS)
@pytest.mark.parametrize("size", SIZES)
def test_families_are_valid_states(size, book):
    """Every state fits the agent record and stands on a free cell; tasks are in the tables."""
    from psketch_b200 import _lib
    tables = stress_tables(size, book)
    assert tables.n_features == (404 if book == "stock" else 385)
    for f in FAMILIES:
        S = family(size, book, f)
        _lib.check_agent_inputs(tables, inv=S["inv"], pos=S["pos"], dirs=S["dir"], task=S["task"])
        g = S["grid"].reshape(-1, tables.W, tables.H)
        assert (g[np.arange(len(g)), S["pos"][:, 0], S["pos"][:, 1]] == 0).all(), f
        assert S["grid"].max() < tables.K and (S["task"] > 0).all(), f


@pytest.mark.parametrize("book", BOOKS)
@pytest.mark.parametrize("size", SIZES)
def test_mazes_are_long(size, book):
    """Reachable mazes give teacher distances above 255 on 32x32 and above 1,000 on 64x64; the
    walled-off ones give STOP with no path."""
    S = family(size, book, "maze")
    o = stress_oracle(size, book)
    act, dist, st = o.expert(S["grid"], S["inv"], S["pos"], S["dir"], S["task"])
    reach = S["case"] == "long"
    # go[X] tasks with the agent already facing X cannot happen: the goal sits in a far corner
    assert (dist[reach] > 0).all() and (act[reach] < 4).all()
    assert (dist[~reach] == -1).all() and (act[~reach] == 5).all() and (st[~reach] == 1).all()
    floor = {16: 60, 32: 255, 64: 1000}[size]
    assert dist.max() > floor and np.median(dist[reach]) > floor, (dist.max(), floor)
    print("maze %dx%d %s: teacher distances %d..%d" % (size, size, book, dist[reach].min(), dist.max()))


@pytest.mark.parametrize("book", BOOKS)
@pytest.mark.parametrize("size", SIZES)
def test_ties_occur(size, book):
    """Several goals at the minimum distance and several first actions on a shortest path occur in
    every family with free space; on 64x64 the open room has goal ties inside one lane (rows 2l and
    2l+1) and across a lane boundary (rows 2l+1 and 2l+2).  Counts are printed per family."""
    counts = {f: tie_counts(size, book, f) for f in ("random", "open", "ringless", "leaf", "maze")}
    for f, (g, a, s, l) in counts.items():
        print("%dx%d %s %-8s goal ties %4d  first-action ties %4d  slot ties %3d  lane ties %3d"
              % (size, size, book, f, g, a, s, l))
    for f in ("random", "open", "ringless"):
        assert counts[f][0] > 0 and counts[f][1] > 0, f
    g, a, s, l = counts["open"]
    assert g >= FAMILY_N[size]["open"] // 8 and a >= FAMILY_N[size]["open"] // 4
    assert s > 0 and l > 0


@pytest.mark.parametrize("size", SIZES)
def test_ringless_covers_every_edge_cell(size):
    """The agent stands on every edge cell with every facing and on cells 1-4 from each edge; items
    lie on the edges; there is no ring."""
    tables = stress_tables(size)
    W, H = tables.W, tables.H
    S = family(size, "stock", "ringless")
    edge, near = ringless_positions(W, H)
    seen = set(zip(S["pos"][:, 0].tolist(), S["pos"][:, 1].tolist(), S["dir"].tolist()))
    assert all((x, y, d) in seen for x, y in edge for d in range(4))
    depth = np.minimum.reduce([S["pos"][:, 0], S["pos"][:, 1], W - 1 - S["pos"][:, 0], H - 1 - S["pos"][:, 1]])
    assert set(depth.tolist()) == {0, 1, 2, 3, 4}
    g = S["grid"].reshape(-1, W, H)
    wall = _kind(tables, "boundary")
    assert not (g == wall).any()
    rim = np.concatenate([g[:, 0, :], g[:, -1, :], g[:, :, 0], g[:, :, -1]], axis=1)
    for k in go_kinds(tables):
        assert (rim == k).any(axis=1).sum() > len(g) // 4, k


def leaf_label(tables, oracle, S):
    """The teacher's leaf case of each env, from the oracle alone (None where it is none of them)."""
    n = len(S["grid"])
    act, dist, st = oracle.expert(S["grid"], S["inv"], S["pos"], S["dir"], S["task"])
    sat = oracle.satisfies(S["grid"], S["inv"], S["pos"], S["dir"], S["task"])
    _, flen, _, _ = oracle.find_closest(S["grid"], S["pos"], S["dir"], S["target"], seq_cap=0)
    lab = np.array([None] * n, dtype=object)
    lab[(act == 4) & (dist == -1)] = "use"
    lab[(act == 5) & (sat == 1) & (flen != 0)] = "stop"
    lab[(act == 5) & (sat == 1) & (flen == 0)] = "facing"
    lab[(act < 4) & (dist >= 1) & (dist <= 3)] = "short"
    lab[(act < 4) & (dist > 2 * tables.W)] = "long"
    lab[(act == 5) & (sat != 1) & (dist == -1) & (st == 1) & (flen == -1)
        & (S["grid"] == S["target"][:, None]).any(axis=1)] = "unreachable"
    return lab


@pytest.mark.parametrize("book", BOOKS)
@pytest.mark.parametrize("size", SIZES)
def test_paired_batches_cover_every_leaf_pair(size, book):
    """Each env's case is what the oracle answers, and envs (2i, 2i+1) cover all 36 ordered pairs."""
    tables, o = stress_tables(size, book), stress_oracle(size, book)
    S = family(size, book, "leaf")
    lab = leaf_label(tables, o, S)
    assert list(lab) == list(S["case"]), [(i, a, b) for i, (a, b) in enumerate(zip(lab, S["case"])) if a != b][:5]
    pairs = set(zip(lab[0::2], lab[1::2]))
    assert pairs == set(itertools.product(LEAF_CASES, LEAF_CASES))


@pytest.mark.parametrize("book", BOOKS)
@pytest.mark.parametrize("size", SIZES)
def test_inventory_counts_reach_255_on_every_kind(size, book):
    tables, o = stress_tables(size, book), stress_oracle(size, book)
    S = family(size, book, "inventory")
    K = tables.K
    for k in range(1, K):
        assert set(INV_COUNTS) <= set(S["inv"][:, k].tolist()), k
    f = o.features(S["grid"], S["inv"], S["pos"], S["dir"])
    assert np.array_equal(f[:, 18 * K:19 * K], S["inv"].astype(np.float32))
