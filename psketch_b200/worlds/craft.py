"""Drop-in mirror of the reference's ``worlds/craft.py`` object API, backed by the CUDA kernels.

Same names, argument meaning and error behaviour as the reference so that its trainers, students
and teachers run unchanged (SURVEY.md §8(b)):

    world = CraftWorld(config)                    worlds/craft.py:58-109
    state = world.init_state(grid, pos, dir=0)    worlds/craft.py:258-259
    reward, state2 = state.step(action)           worlds/craft.py:332-424   (state is not mutated)
    state.features()  -> float64[n_features]      worlds/craft.py:296-330
    state.satisfies(task)                         worlds/craft.py:285-294
    state.pos / .dir / .inventory / .grid / .world / .scenario

States are persistent host-side records (64 + 32 bytes); all arithmetic happens on the GPU.
The trainers call ``states[i].step(a)`` one env at a time, so ``step`` only *records* the
transition; the first read of any derived value flushes every pending transition of the world
in ONE batched launch sequence (step -> features -> teacher -> satisfies) and caches the results
on the state objects, exactly like the reference caches ``_cached_features``.
"""
import os

import numpy as np

from .. import _lib
from ..tables import (COORD_CHANGE, Cookbook, CraftTables, TaskManager, WORLD_CONFIGS, DOWN, UP,
                      LEFT, RIGHT, STOP, N_ACTIONS)


class _Struct(object):
    """Attribute bag compatible with misc.util.Struct for the fields the trainers read."""

    def __init__(self, **kw):
        for k, v in kw.items():
            setattr(self, k, _Struct(**v) if isinstance(v, dict) else v)


def _cfg_get(config, path, default=None):
    cur = config
    for name in path.split("."):
        if cur is None or not hasattr(cur, name):
            return default
        cur = getattr(cur, name)
    return cur


def _given_file(path, packaged_default):
    """A path from the config: the file itself when it exists; None (= the tables embedded in
    psketch_b200.tables, which ARE the reference's resources/craft files) only when the config names
    the reference's stock file and the process does not run from a reference checkout; a path the
    user typed that does not exist raises like the reference's open() (worlds/cookbook.py:9)."""
    if not path:
        return None
    if os.path.exists(path):
        return path
    if os.path.normpath(path) == os.path.normpath(packaged_default):
        return None
    raise FileNotFoundError(path)


class CraftWorld(object):
    def __init__(self, config=None, tables=None, device=None):
        recipes = _cfg_get(config, "recipes")
        cookbook = Cookbook(_given_file(recipes, "resources/craft/recipes.yaml"))
        world_name = _cfg_get(config, "world.config", "craft_medium")
        world_file = os.path.join("configs/worlds", "%s.yaml" % world_name)
        if os.path.exists(world_file):
            import yaml
            with open(world_file) as f:
                world_cfg = yaml.safe_load(f)
        else:
            world_cfg = dict(WORLD_CONFIGS[world_name])
        for k, v in world_cfg.items():          # worlds/craft.py:64-67
            setattr(self, k, v)
        hints = _cfg_get(config, "trainer.hints")
        tm = TaskManager(_given_file(hints, "resources/craft/hints.hierarchy.yaml"))
        self.tables = tables if tables is not None else CraftTables(cookbook, tm, world_cfg)
        self.cookbook = self.tables.cookbook
        self.task_manager = self.tables.task_manager
        self.n_features = self.tables.n_features
        self.n_actions = N_ACTIONS
        if config is not None and _cfg_get(config, "student.model") is not None:
            config.student.model.input_size = self.n_features      # worlds/craft.py:69
            config.student.model.n_actions = self.n_actions        # worlds/craft.py:76
        names = ("DOWN", "UP", "LEFT", "RIGHT", "USE", "STOP")
        self.actions = _Struct(**{n: {"index": i, "coord_change": COORD_CHANGE[i]}
                                  for i, n in enumerate(names)})
        self.action_space = [getattr(self.actions, n) for n in names]
        env = self.cookbook.environment
        self.non_grabbable_indices = env
        self.grabbable_indices = [i for i in range(self.cookbook.n_kinds) if i not in env]
        self.workshop_indices = list(self.tables.workshop_kinds)
        self.water_index = self.cookbook.index["water"]
        self.stone_index = self.cookbook.index["stone"]
        self.random = _cfg_get(config, "random")
        self._scenario_seed = _cfg_get(config, "seed", 123)
        self._device = device
        self._backend = None
        self._pending = []          # states whose transition has not been computed yet
        self._fresh = []            # initial states whose derived values are not cached yet
        self._grid_cache = {}
        self._task_ids = {}         # (goal_name, goal_arg) -> task id

    # -- reference API -----------------------------------------------------------------------
    def make_scenario(self, grid, pos, dir=0):
        return CraftScenario(grid, pos, self, init_dir=dir)

    def init_state(self, grid, pos, dir=0):
        return self.make_scenario(grid, pos, dir=dir).init()

    def sample_scenario(self, ingredients=None, make_island=False, make_cave=False):
        """``make_data.sample_scenario(world, ingredients, config)`` (make_data.py:105-144; the method
        of the same name in worlds/craft.py:111-166 is dead code inside a string literal): boundary
        ring, N_PRIMITIVES of every primitive, the workshops and a start cell, each placed so that
        the free cells stay connected.  Returns ``(grid one-hot float64[W, H, K], init_pos)`` like the
        reference.  Drawn by the Philox sampler kernel (psk_craft_sample_scenarios), 256 scenarios per
        launch, handed out one by one; distribution checked against the reference's sampler
        (tests/test_scenario_gpu.py), not its numpy random stream (SURVEY §8 R1)."""
        if make_island or make_cave:
            raise NotImplementedError("the reference's island / cave branch is broken (make_data.py:120) "
                                      "and never taken")
        pool = getattr(self, "_scenario_pool", None)
        if not pool:
            from .. import data
            seed = int(getattr(self, "_scenario_seed", 123))
            offset = int(getattr(self, "_scenario_offset", 0))
            grid, pos, fails = data.sample_scenarios(self.tables, 256, seed, offset, device=self._device)
            if fails:
                raise _lib.PskError("scenario sampler ran out of draws")
            self._scenario_offset = offset + 256
            C = self.tables.W * self.tables.H
            g, p = grid[:, :C].cpu().numpy(), pos.cpu().numpy()
            pool = self._scenario_pool = [(g[i], tuple(int(v) for v in p[i])) for i in range(len(g))][::-1]
        cells, init_pos = pool.pop()
        ids = cells.reshape(self.WIDTH, self.HEIGHT)
        onehot = np.zeros((self.WIDTH, self.HEIGHT, self.cookbook.n_kinds))
        xs, ys = np.nonzero(ids)
        onehot[xs, ys, ids[xs, ys]] = 1
        return onehot, init_pos

    def render(self, state):
        inv = {self.cookbook.index.get(i): int(v) for i, v in enumerate(state.inventory) if v > 0}
        print("\nInventory:", inv)
        rows = []
        arrows = {LEFT: "<", RIGHT: ">", UP: "^", DOWN: "v"}
        cells = state.cells.reshape(self.WIDTH, self.HEIGHT)
        for y in range(self.HEIGHT):
            row = ""
            for x in range(self.WIDTH):
                if (x, y) == state.pos:
                    row += arrows[state.dir] + " "
                elif cells[x, y] == 0:
                    row += ". "
                else:
                    row += "%-2s" % self.cookbook.index.get(int(cells[x, y]))[:2]
            rows.append(row)
        rows = rows[::-1]
        print("\n".join(rows))
        return rows

    # -- batching machinery ------------------------------------------------------------------
    def cells_of(self, grid):
        """one-hot float grid [W,H,K] (dataset item) or kind-id grid -> u8[W*H] kind ids."""
        g = np.asarray(grid)
        if g.ndim == 3:
            key = (g.__array_interface__["data"][0], g.shape)
            hit = self._grid_cache.get(key)
            if hit is not None and hit[0] is grid:
                return hit[1]
            assert (g.sum(axis=2) <= 1).all(), "impossible world configuration"   # craft.py:371
            ids = (g.argmax(axis=2) * (g.sum(axis=2) > 0)).astype(np.uint8).reshape(-1)
            if len(self._grid_cache) > 4096:
                self._grid_cache.clear()
            self._grid_cache[key] = (grid, ids)
            return ids
        return g.astype(np.uint8).reshape(-1)

    def backend(self):
        if self._backend is None:
            self._backend = _Backend(self)
        return self._backend

    def flush(self):
        """Computes every pending transition (and the derived values of the new states)."""
        if self._pending:
            pend, self._pending = self._pending, []
            self.backend().evaluate(pend)


class CraftScenario(object):
    def __init__(self, grid, init_pos, world, init_dir=0):
        self.init_grid = grid
        self.init_pos = init_pos
        self.init_dir = init_dir
        self.world = world

    def init(self):
        w = self.world
        agent = np.zeros(_lib.AGENT_BYTES, np.uint8)
        agent[_lib.AG_X], agent[_lib.AG_Y] = int(self.init_pos[0]), int(self.init_pos[1])
        agent[_lib.AG_DIR] = int(self.init_dir)
        onehot = self.init_grid if np.ndim(self.init_grid) == 3 else None
        state = CraftState(self, w.cells_of(self.init_grid), agent, grid_onehot=onehot)
        w._fresh.append(state)
        if len(w._fresh) > 65536:
            del w._fresh[:32768]
        return state


class CraftState(object):
    """Persistent state record.  ``_cells``/``_agent`` are None while the transition that produces
    this state is still pending (``_parent``, ``_action``)."""

    def __init__(self, scenario, cells, agent, grid_onehot=None, parent=None, action=None):
        self.scenario = scenario
        self.world = scenario.world
        self._cells = cells
        self._agent = agent
        self._grid = grid_onehot
        self._parent = parent
        self._action = action
        self._cached_features = None
        self._task_hint = parent._task_hint if parent is not None else 0
        self._expert = {}           # task id -> action
        self._sat = {}              # task id -> 0 / 1 / 2
        self._all = None            # (expert u8[T, m], sat u8[T, m], column): every task, see _run
        self._evaluated = False     # features / teacher / satisfies cached for the hinted task

    # -- materialisation ---------------------------------------------------------------------
    def _need(self):
        if self._cells is None:
            self.world.flush()
        if self._cells is None:      # created outside the queue (should not happen)
            self.world.backend().evaluate([self])

    @property
    def cells(self):
        self._need()
        return self._cells

    @property
    def pos(self):
        self._need()
        return (int(self._agent[_lib.AG_X]), int(self._agent[_lib.AG_Y]))

    @property
    def dir(self):
        self._need()
        return int(self._agent[_lib.AG_DIR])

    @property
    def inventory(self):
        self._need()
        return self._agent[:self.world.cookbook.n_kinds].astype(np.float64)

    @inventory.setter
    def inventory(self, value):
        self._need()
        value = np.asarray(value)
        _lib.check_agent_inputs(self.world.tables, inv=value.reshape(1, -1))
        self._agent = self._agent.copy()
        self._agent[:self.world.cookbook.n_kinds] = value.astype(np.uint8)
        self._invalidate()

    @property
    def grid(self):
        """one-hot float64 [W,H,K] view of the grid, as the reference stores it."""
        if self._grid is None:
            w = self.world
            cells = self.cells.reshape(w.WIDTH, w.HEIGHT)
            g = np.zeros((w.WIDTH, w.HEIGHT, w.cookbook.n_kinds))
            xs, ys = np.nonzero(cells)
            g[xs, ys, cells[xs, ys]] = 1
            self._grid = g
        return self._grid

    def _invalidate(self):
        self._cached_features = None
        self._expert, self._sat, self._all, self._evaluated = {}, {}, None, False

    def _task_id(self, task):
        w = self.world
        key = (task.goal_name, task.goal_arg)
        tid = w._task_ids.get(key)
        if tid is None:
            t = w.task_manager.tasks_by_goal.get("%s[%s]" % key)
            if t is None:
                raise KeyError("unknown task %r" % (task,))
            tid = w._task_ids[key] = t.task_id
        return tid

    def _evaluate(self, task_id=None):
        self._need()
        if task_id is not None and task_id != self._task_hint:
            self._task_hint = task_id
            self._evaluated = False
        if not self._evaluated:
            w = self.world
            # evaluate together with every other initial state that is still waiting
            batch = [self] + [s for s in w._fresh if s is not self and not s._evaluated]
            w._fresh = []
            w.backend().evaluate(batch, step=False)

    def _lookup(self, cache, which, tid):
        """Teacher action / satisfies code for task ``tid``: from the per-task cache, from the
        all-task table computed while the state's task was unknown, else by evaluating now.
        Remembers the task so that the states stepped from this one are evaluated for it."""
        v = cache.get(tid)
        if v is None:
            if self._all is not None:
                v = cache[tid] = int(self._all[which][tid - 1, self._all[2]])
                self._task_hint = tid
            else:
                self._evaluate(tid)
                v = cache[tid]
        return v

    # -- reference API -----------------------------------------------------------------------
    def step(self, action):
        action = int(action)
        if action < 0 or action >= N_ACTIONS:
            raise Exception("Unexpected action: %s" % action)      # worlds/craft.py:415-416
        child = CraftState(self.scenario, None, None, parent=self, action=action)
        self.world._pending.append(child)
        return 0, child

    def features(self):
        if self._cached_features is None:
            self._evaluate()
        return self._cached_features

    def satisfies(self, task):
        v = self._lookup(self._sat, 1, self._task_id(task))
        return None if v == 2 else bool(v)

    def expert_action(self, task):
        a = self._lookup(self._expert, 0, self._task_id(task))
        if a == 255:
            raise AssertionError("subtask is neither 'use' nor 'go'")   # demonstration.py:18
        return a

    def neighbors(self, pos, dir=None):
        x, y = pos
        w = self.world
        out = []
        if x > 0 and (dir is None or dir == LEFT):
            out.append((x - 1, y))
        if y > 0 and (dir is None or dir == DOWN):
            out.append((x, y - 1))
        if x < w.WIDTH - 1 and (dir is None or dir == RIGHT):
            out.append((x + 1, y))
        if y < w.HEIGHT - 1 and (dir is None or dir == UP):
            out.append((x, y + 1))
        return out

    def next_to(self, i_kind):
        x, y = self.pos
        c = self.cells.reshape(self.world.WIDTH, self.world.HEIGHT)
        return bool((c[max(x - 1, 0):x + 2, max(y - 1, 0):y + 2] == i_kind).any())

    def hit_wall(self):
        return not self.neighbors(self.pos, self.dir)

    def render(self):
        return self.world.render(self)

    def make_navigation_grid(self):
        return (self.cells.reshape(self.world.WIDTH, self.world.HEIGHT) != 0).astype(np.float64)

    def find_resource_positions(self, goal_arg):
        thing = self.world.cookbook.index[goal_arg]
        c = self.cells.reshape(self.world.WIDTH, self.world.HEIGHT)
        return list(zip(*np.nonzero(c == thing)))


class _Backend(object):
    """Device scratch + launch sequence for a list of states (any size; typically the batch)."""

    def __init__(self, world):
        import torch
        if not torch.cuda.is_available():
            raise _lib.PskError("the Craft façade needs a CUDA device (there is no CPU fallback)")
        self.torch = torch
        self.world = world
        self.lib = _lib.load()
        self.ct = _lib.make_tables(world.tables)
        self.device = torch.device(world._device or "cuda:%d" % torch.cuda.current_device())
        self.cap = 0
        self.C = world.tables.W * world.tables.H
        self.cs = ((self.C + 63) // 64) * 64
        self.nf = world.tables.n_features
        self.K = world.tables.K
        self.err = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.h_err = torch.zeros(1, dtype=torch.int32).pin_memory()
        self.T = world.tables.n_tasks - 1                      # task ids 1..T
        self.task_ids = torch.arange(1, self.T + 1, dtype=torch.uint8, device=self.device)

    def _reserve(self, n):
        if n <= self.cap:
            return
        torch = self.torch
        cap = max(64, 1 << (n - 1).bit_length())
        # one pinned blob and one device blob per direction: grid rows | agent records | four byte
        # rows (action, task, teacher action, satisfies), laid out per call for the batch at hand
        # so that a timestep is ONE host->device copy and two device->host copies
        per_env = self.cs + _lib.AGENT_BYTES + 4
        self.h_blob = torch.zeros(cap * per_env, dtype=torch.uint8).pin_memory()
        self.d_blob = torch.zeros(cap * per_env, dtype=torch.uint8, device=self.device)
        self.h_feat = torch.zeros(cap * self.nf, dtype=torch.float32).pin_memory()
        self.d_feat = torch.zeros(cap * self.nf, dtype=torch.float32, device=self.device)
        self.h_np, self.h_feat_np = self.h_blob.numpy(), self.h_feat.numpy()
        self.cap = cap

    def find_closest(self, cells, agent, kind, seq_cap=96):
        """BaseTeacher.find_closest_resources (teachers/base.py:27-34) for one state: (goal u8[2],
        path length or -1, action sequence u8[seq_cap] padded with 255) from psk_craft_find_closest."""
        import ctypes
        torch = self.torch
        grid = np.zeros((1, self.cs), np.uint8)
        grid[0, :self.C] = cells
        agent = np.array(agent, np.uint8).reshape(1, _lib.AGENT_BYTES)
        with torch.cuda.device(self.device):
            stream = _lib.raw_stream(torch, self.device)
            d_grid = torch.from_numpy(grid).to(self.device)
            d_agent = torch.from_numpy(agent).to(self.device)
            d_kind = torch.full((1,), int(kind), dtype=torch.uint8, device=self.device)
            d_goal = torch.empty((1, 2), dtype=torch.uint8, device=self.device)
            d_len = torch.empty(1, dtype=torch.int16, device=self.device)
            d_seq = torch.empty((1, seq_cap), dtype=torch.uint8, device=self.device)
            st = _lib.CraftStateC(d_grid.data_ptr(), d_agent.data_ptr(), 1, self.cs, 0)
            p = lambda t: ctypes.c_void_p(t.data_ptr())
            rc = self.lib.psk_craft_find_closest(ctypes.byref(self.ct), st, p(d_kind), p(d_goal),
                                                 p(d_len), p(d_seq), seq_cap, stream)
            _lib.check(rc, "psk_craft_find_closest")
            return d_goal.cpu().numpy()[0], int(d_len.cpu().numpy()[0]), d_seq.cpu().numpy()[0]

    def evaluate(self, states, step=True):
        """step=True: ``states`` are pending children (parent + action); computes their state.
        Always computes features, teacher action and satisfies for each state's hinted task."""
        import ctypes
        torch = self.torch
        if step:
            # parents may themselves be pending only if they are in the same queue *earlier*:
            # resolve generations in order
            order, rest = [], states
            while rest:
                ready = [s for s in rest if s._parent._cells is not None]
                if not ready:
                    raise _lib.PskError("dangling pending state")
                self._run(ready, True)
                rest = [s for s in rest if s._cells is None]
                order += ready
            return
        self._run(states, False)

    def _run(self, states, step):
        import contextlib
        import ctypes
        torch = self.torch
        n = len(states)
        self._reserve(n)
        C, cs, AB, nf = self.C, self.cs, _lib.AGENT_BYTES, self.nf
        n64 = (n + 63) & ~63
        off_a = n64 * cs
        off_s = off_a + n64 * AB
        end_in, end = off_s + 2 * n64, off_s + 4 * n64
        hb = self.h_np
        hg = hb[:n * cs].reshape(n, cs)
        ha = hb[off_a:off_a + n * AB].reshape(n, AB)
        hs = hb[off_s:end].reshape(4, n64)
        # gather with a handful of numpy calls for the whole batch (the per-state Python work of
        # this function is what bounds the object API, not the GPU)
        src = [s._parent for s in states] if step else states
        parent_cells = np.concatenate([q._cells for q in src]).reshape(n, C)
        hg[:, :C] = parent_cells
        if cs > C:
            hg[:, C:] = 0
        ha[:] = np.concatenate([q._agent for q in src]).reshape(n, AB)
        hs[0, :n] = [s._action for s in states] if step else STOP
        hs[1, :n] = [s._task_hint for s in states]
        same_device = torch.cuda.current_device() == self.device.index
        with (contextlib.nullcontext() if same_device else torch.cuda.device(self.device)):
            cur = torch.cuda.current_stream(self.device)
            stream = ctypes.c_void_p(cur.cuda_stream)
            self.d_blob[:end_in].copy_(self.h_blob[:end_in], non_blocking=True)
            base = self.d_blob.data_ptr()
            row = [ctypes.c_void_p(base + off_s + k * n64) for k in range(4)]
            st = _lib.CraftStateC(base, base + off_a, n, cs, 0)
            tb = ctypes.byref(self.ct)
            feat = ctypes.c_void_p(self.d_feat.data_ptr())
            p = lambda t: ctypes.c_void_p(t.data_ptr())
            if step:
                _lib.check(self.lib.psk_craft_step(tb, st, row[0], None, None, p(self.err), stream),
                           "psk_craft_step")
            _lib.check(self.lib.psk_craft_features(tb, st, feat, 0, stream), "psk_craft_features")
            _lib.check(self.lib.psk_craft_expert(tb, st, row[1], row[2], None, None, stream),
                       "psk_craft_expert")
            _lib.check(self.lib.psk_craft_satisfies(tb, st, row[1], row[3], stream),
                       "psk_craft_satisfies")
            # States whose task is not known yet (initial states; every state of an evaluation
            # rollout, where the teacher is never asked): teacher action and satisfies for EVERY
            # task, on T replicas of those states, so that the per-env teacher(task, state) /
            # satisfies(task) calls that follow are cache hits instead of one launch each.
            hintless = [i for i, s in enumerate(states) if not s._task_hint]
            all_tasks = None
            if hintless:
                m, T = len(hintless), self.T
                g = self.d_blob[:n * cs].view(n, cs)
                a = self.d_blob[off_a:off_a + n * AB].view(n, AB)
                if m < n:
                    idx = torch.as_tensor(hintless, dtype=torch.int64).to(self.device)
                    g, a = g.index_select(0, idx), a.index_select(0, idx)
                g, a = g.repeat(T, 1), a.repeat(T, 1)
                tasks = self.task_ids.repeat_interleave(m)
                all_tasks = torch.empty((2, T * m), dtype=torch.uint8, device=self.device)
                st_all = _lib.CraftStateC(g.data_ptr(), a.data_ptr(), T * m, cs, 0)
                _lib.check(self.lib.psk_craft_expert(tb, st_all, p(tasks), p(all_tasks[0]), None,
                                                     None, stream), "psk_craft_expert")
                _lib.check(self.lib.psk_craft_satisfies(tb, st_all, p(tasks), p(all_tasks[1]),
                                                        stream), "psk_craft_satisfies")
            lo = 0 if step else off_s + 2 * n64
            self.h_blob[lo:end].copy_(self.d_blob[lo:end], non_blocking=True)
            self.h_feat[:n * nf].copy_(self.d_feat[:n * nf], non_blocking=True)
            self.h_err.copy_(self.err, non_blocking=True)
            cur.synchronize()
            flags = int(self.h_err.item())
            if flags:
                # what the reference does for these conditions: float64 inventories keep counting
                # (ours are u8), a bad action raises (already rejected in CraftState.step)
                self.err.zero_()
                if flags & _lib.FLAG_INV_OVERFLOW:
                    raise OverflowError("inventory count above 255 (u8 storage; the reference's "
                                        "float64 inventory has no such limit)")
                if flags & _lib.FLAG_BAD_ACTION:
                    raise Exception("Unexpected action")              # worlds/craft.py:415-416
            if all_tasks is not None:
                all_tasks = all_tasks.cpu().numpy().reshape(2, self.T, len(hintless))
                for col, i in enumerate(hintless):
                    states[i]._all = (all_tasks[0], all_tasks[1], col)
        feats = self.h_feat_np[:n * nf].reshape(n, nf).astype(np.float64)   # one row view per state
        expert, sat = hs[2, :n].tolist(), hs[3, :n].tolist()
        if step:
            cells, agents = hg[:, :C].copy(), ha.copy()
            unchanged = (cells == parent_cells).all(axis=1).tolist()
        for i, s in enumerate(states):
            if step:
                parent = s._parent
                if unchanged[i]:                 # share the grid (and its one-hot view) with the parent
                    s._cells, s._grid = parent._cells, parent._grid
                else:
                    s._cells = cells[i]
                s._agent = agents[i]
                s._parent = None
            s._cached_features = feats[i]
            hint = s._task_hint
            if hint:
                s._expert[hint] = expert[i]
                s._sat[hint] = sat[i]
            s._evaluated = True
