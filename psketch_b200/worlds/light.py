"""Light world (rooms, doors, keys) — host-side scenario construction restated from
worlds/light.py:21-161 (same numpy RandomState call sequence, so the scenarios are the
reference's), with step / features / satisfies / teacher running on the GPU (psk_light.h).

    world = LightWorld()                               worlds/light.py:14-19
    scen = world.sample_scenario_with_goal("URU")      worlds/light.py:21-161
    state = scen.init()                                worlds/light.py:175-180
    reward, state2 = state.step(a); state.features(); state.satisfies(None, None)

``VecLight`` is the batched form (N envs, shared scenario table).
"""
import ctypes

import numpy as np

from .. import _lib

DOWN, UP, LEFT, RIGHT, USE = 0, 1, 2, 3, 4
ROOM_W = ROOM_H = 6
MAX_BOARD, MAX_DOORS, MAX_KEYS = 32, 8, 8
# resources/light/recipes.yaml "primitives": the goal strings, in index order (ids from 1)
LIGHT_GOALS = ("LL", "LU", "LD", "RR", "RU", "RD", "UL", "UR", "UU", "DL", "DR", "DD",
               "URU", "DRU", "LLD", "RDD", "LUR")


class LightScenarioC(ctypes.Structure):
    """Mirror of ``psk_light_scenario`` (include/psk_light.h), 192 bytes."""
    _fields_ = [("walls", ctypes.c_uint32 * 32), ("doors", ctypes.c_uint8 * 16),
                ("keys", ctypes.c_uint8 * 32), ("n_doors", ctypes.c_uint8),
                ("n_keys", ctypes.c_uint8), ("board_w", ctypes.c_uint8), ("board_h", ctypes.c_uint8),
                ("goal_rx", ctypes.c_uint8), ("goal_ry", ctypes.c_uint8), ("init_x", ctypes.c_uint8),
                ("init_y", ctypes.c_uint8), ("reserved", ctypes.c_uint8 * 8)]


def _walk(goal):
    x = y = 0
    for c in goal:
        if c == "L":
            x -= 1
        elif c == "R":
            x += 1
        elif c == "U":
            y -= 1
        elif c == "D":
            y += 1
        yield x, y


class LightWorld(object):
    def __init__(self, config=None):
        self.n_actions = 5
        self.n_features = 12
        self.goals = list(LIGHT_GOALS)
        self.random = np.random.RandomState(0)          # worlds/light.py:19

    def goal_name(self, goal):
        return goal if isinstance(goal, str) else self.goals[int(goal) - 1]

    def sample_scenario_with_goal(self, goal):
        goal = self.goal_name(goal)
        rnd = self.random
        l = r = u = d = 0
        for x, y in _walk(goal):
            l, r, u, d = min(l, x), max(r, x), min(u, y), max(d, y)
        l -= rnd.randint(2)
        r += rnd.randint(2)
        u -= rnd.randint(2)
        d += rnd.randint(2)
        rooms_x, rooms_y = r - l + 1, d - u + 1
        init_x, init_y = -l, -u
        board_w, board_h = ROOM_W * rooms_x + 1, ROOM_H * rooms_y + 1
        walls = np.zeros((board_w, board_h))
        walls[0::ROOM_W, :] = 1
        walls[:, 0::ROOM_H] = 1
        doors, keys = [], {}
        px = py = 0
        for x, y in _walk(goal):                        # doors along the goal path
            dx, dy = x - px, y - py
            cx = ROOM_W * (init_x + px) + ROOM_W // 2
            cy = ROOM_H * (init_y + py) + ROOM_H // 2
            wx, wy = cx + ROOM_W // 2 * dx, cy + ROOM_H // 2 * dy
            kx = cx + rnd.randint(ROOM_W // 2 + 1) - 1
            ky = cy + rnd.randint(ROOM_H // 2 + 1) - 1
            walls[wx, wy] = 0
            doors.append((wx, wy))
            if rnd.rand() < 0.5:
                keys[(kx, ky)] = (wx, wy)
            px, py = x, y
        for _ in range(min(rooms_x, rooms_y)):          # extra doors
            if rooms_x == 1 or rooms_y == 1:
                continue
            px = rnd.randint(rooms_x - 1)
            py = rnd.randint(rooms_y - 1)
            dx, dy = (1, 0) if rnd.randint(2) else (0, 1)
            cx = ROOM_W * px + ROOM_W // 2
            cy = ROOM_H * py + ROOM_H // 2
            wx, wy = cx + ROOM_W // 2 * dx, cy + ROOM_H // 2 * dy
            if (wx, wy) in doors:
                continue
            kx = cx + rnd.randint(ROOM_W // 2 + 1) - 1
            ky = cy + rnd.randint(ROOM_H // 2 + 1) - 1
            walls[wx, wy] = 0
            doors.append((wx, wy))
            if rnd.rand() < 0.5:
                keys[(kx, ky)] = (wx, wy)
        gx, gy = list(_walk(goal))[-1]
        return LightScenario(walls, doors, keys, (init_x, init_y), (init_x + gx, init_y + gy), self)


class LightScenario(object):
    def __init__(self, walls, doors, keys, init_room, goal_room, world):
        self.walls, self.doors, self.keys = walls, doors, keys
        self.init_room, self.goal_room, self.world = init_room, goal_room, world
        self._vec = None

    def to_c(self):
        bw, bh = self.walls.shape
        if bw > MAX_BOARD - 1 or bh > MAX_BOARD - 1 or len(self.doors) > MAX_DOORS or len(self.keys) > MAX_KEYS:
            raise ValueError("scenario exceeds the compiled Light limits")
        c = LightScenarioC()
        full = np.ones((MAX_BOARD, MAX_BOARD), np.uint8)
        full[:bw, :bh] = self.walls != 0
        rows = (full.astype(np.uint64) << np.arange(MAX_BOARD, dtype=np.uint64)[None, :]).sum(axis=1)
        for x in range(MAX_BOARD):
            c.walls[x] = int(rows[x])
        for i, (x, y) in enumerate(self.doors):
            c.doors[2 * i], c.doors[2 * i + 1] = x, y
        for i, ((kx, ky), (dx, dy)) in enumerate(self.keys.items()):
            c.keys[4 * i:4 * i + 4] = [kx, ky, dx, dy]
        c.n_doors, c.n_keys, c.board_w, c.board_h = len(self.doors), len(self.keys), bw, bh
        c.goal_rx, c.goal_ry = self.goal_room
        c.init_x = ROOM_W * self.init_room[0] + ROOM_W // 2
        c.init_y = ROOM_H * self.init_room[1] + ROOM_H // 2
        return c

    def init(self):
        ix = ROOM_W * self.init_room[0] + ROOM_W // 2
        iy = ROOM_H * self.init_room[1] + ROOM_H // 2
        return LightState(self.walls, self.doors, self.keys, (ix, iy), self)

    def vec(self):
        if self._vec is None:
            self._vec = VecLight([self], [0])
        return self._vec


class LightState(object):
    """Persistent single-env state (reference object API); every call is one batch-of-1 launch."""

    def __init__(self, walls, doors, keys, pos, scenario):
        self.walls, self.doors, self.keys, self.pos, self.scenario = walls, doors, keys, pos, scenario
        self._cached_features = None

    def _load(self):
        v = self.scenario.vec()
        mask = 0
        for i, k in enumerate(self.scenario.keys):
            if k in self.keys:
                mask |= 1 << i
        v.set_state(np.asarray([[self.pos[0], self.pos[1], mask, 0]], np.uint8))
        return v

    def features(self):
        if self._cached_features is None:
            self._cached_features = self._load().features().cpu().numpy()[0].astype(np.float64)
        return self._cached_features

    def satisfies(self, goal_name, goal_arg):
        return bool(self._load().satisfies().cpu().numpy()[0])

    def step(self, action):
        v = self._load()
        v.step(np.asarray([action], np.uint8))
        v.check_errors()
        st = v.state.cpu().numpy()[0]
        keys = {k: d for i, (k, d) in enumerate(self.scenario.keys.items()) if (st[2] >> i) & 1}
        return 0, LightState(self.walls, self.doors, keys, (int(st[0]), int(st[1])), self.scenario)

    def expert_action(self):
        a, d = self._load().expert()
        return int(a.cpu().numpy()[0]), int(d.cpu().numpy()[0])


class VecLight(object):
    """N Light envs over a shared table of scenarios; state u8[N,4] = x, y, key mask, 0."""

    def __init__(self, scenarios, scen_idx, device=None):
        import torch
        recs = [s.to_c() for s in scenarios]
        self._board = np.asarray([[c.board_w, c.board_h] for c in recs], np.int64).reshape(-1, 2)
        self._n_keys = np.asarray([c.n_keys for c in recs], np.int64)
        _lib.check_light_inputs(self._board, self._n_keys, scen_idx)
        if not torch.cuda.is_available():
            raise _lib.PskError("VecLight needs a CUDA device (there is no CPU fallback)")
        self.torch = torch
        self.lib = _lib.load_light()
        self.device = torch.device(device or "cuda:%d" % torch.cuda.current_device())
        arr = (LightScenarioC * len(scenarios))(*recs)
        raw = np.frombuffer(bytes(arr), dtype=np.uint8).reshape(len(scenarios), ctypes.sizeof(LightScenarioC))
        self.scen = torch.from_numpy(raw.copy()).to(self.device)
        self.max_keys = max([len(s.keys) for s in scenarios] + [0])
        self.scen_idx = scen_idx
        self.n = len(self.scen_idx)
        self.state = torch.zeros((self.n, 4), dtype=torch.uint8, device=self.device)
        self.err = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.reset()

    def _p(self, t):
        return ctypes.c_void_p(t.data_ptr()) if t is not None else None

    def _stream(self):
        return _lib.raw_stream(self.torch, self.device)

    def _u8(self, x):
        if x is None:
            return None
        if not self.torch.is_tensor(x):
            x = self.torch.as_tensor(np.asarray(x, np.uint8))
        return x.to(device=self.device, dtype=self.torch.uint8).contiguous()

    @property
    def scen_idx(self):
        return self._scen_idx

    @scen_idx.setter
    def scen_idx(self, idx):
        """Scenario of every env; an index out of range raises ValueError (the kernels trust it)."""
        host = idx.cpu().numpy() if self.torch.is_tensor(idx) else np.asarray(idx)
        _lib.check_light_inputs(self._board, self._n_keys, host)
        self._scen_idx_host = host.astype(np.int32).reshape(-1)
        self._scen_idx = self.torch.as_tensor(self._scen_idx_host).to(self.device)

    def set_state(self, st):
        """u8[N, 4] = x, y, key mask, steps of the episode.  ValueError, before anything is copied, for
        a position off the env's board, mask bits at or above its scenario's n_keys or a step byte
        >= 255 (the teacher table has no entry for such a state)."""
        st = np.asarray(st)
        _lib.check_light_inputs(self._board, self._n_keys, self._scen_idx_host, st)
        self.state.copy_(self.torch.as_tensor(st.astype(np.uint8)).to(self.device))

    def reset(self, mask=None):
        mask = self._u8(mask)
        with self.torch.cuda.device(self.device):
            rc = self.lib.psk_light_reset(self._p(self.scen), self._p(self.scen_idx), self._p(self.state),
                                          self._p(mask), self.n, self._stream())
        _lib.check(rc, "psk_light_reset")

    def step(self, actions, active=None):
        actions, active = self._u8(actions), self._u8(active)
        with self.torch.cuda.device(self.device):
            rc = self.lib.psk_light_step(self._p(self.scen), self._p(self.scen_idx), self._p(self.state),
                                         self._p(actions), self._p(active), None, self._p(self.err),
                                         self.n, self._stream())
        _lib.check(rc, "psk_light_step")

    def features(self, out=None):
        if out is None:
            out = self.torch.empty((self.n, 12), dtype=self.torch.float32, device=self.device)
        with self.torch.cuda.device(self.device):
            rc = self.lib.psk_light_features(self._p(self.scen), self._p(self.scen_idx), self._p(self.state),
                                             self._p(out), self.n, self._stream())
        _lib.check(rc, "psk_light_features")
        return out

    def satisfies(self):
        out = self.torch.empty(self.n, dtype=self.torch.uint8, device=self.device)
        with self.torch.cuda.device(self.device):
            rc = self.lib.psk_light_satisfies(self._p(self.scen), self._p(self.scen_idx), self._p(self.state),
                                              self._p(out), self.n, self._stream())
        _lib.check(rc, "psk_light_satisfies")
        return out

    def teacher_table(self):
        """u16[n_scen, 2^max_keys, 32, 32]: fewest actions to the goal room per (key subset, x, y),
        built on first use by psk_light_teacher_build (one CTA per scenario)."""
        if getattr(self, "_table", None) is None:
            n_scen = self.scen.shape[0]
            nbytes = self.lib.psk_light_teacher_table_bytes(n_scen, self.max_keys)
            self._table = self.torch.empty(nbytes // 2, dtype=self.torch.int16, device=self.device)
            with self.torch.cuda.device(self.device):
                rc = self.lib.psk_light_teacher_build(self._p(self.scen), n_scen, self.max_keys,
                                                      self._p(self._table), self._stream())
            _lib.check(rc, "psk_light_teacher_build")
        return self._table

    def expert(self, search=False):
        """(action u8[N], dist i16[N]); action 254 = already in the goal room, 255 = unreachable.
        Default: lookup in the per-scenario table; ``search=True``: one backward flood per env
        (psk_light_expert, the round-1 kernel, kept as an independent second implementation)."""
        act = self.torch.empty(self.n, dtype=self.torch.uint8, device=self.device)
        dist = self.torch.empty(self.n, dtype=self.torch.int16, device=self.device)
        with self.torch.cuda.device(self.device):
            if search:
                rc = self.lib.psk_light_expert(self._p(self.scen), self._p(self.scen_idx), self._p(self.state),
                                               self._p(act), self._p(dist), self.max_keys, self.n,
                                               self._stream())
            else:
                rc = self.lib.psk_light_expert_table(self._p(self.scen), self._p(self.scen_idx),
                                                     self._p(self.state), self._p(self.teacher_table()),
                                                     self.max_keys, self._p(act), self._p(dist), self.n,
                                                     self._stream())
        _lib.check(rc, "psk_light_expert")
        return act, dist

    def tick(self, actions=None, features_out=None, want_features=True, out=None, max_timesteps=100):
        """One rollout tick (psk_light_tick): teacher action, 12 features, then done / success /
        auto-reset or step — one launch.  Returns dict(expert, done, success, features)."""
        torch = self.torch
        actions = self._u8(actions)
        if out is None:
            out = {}
        for k in ("expert", "done", "success"):
            if k not in out:
                out[k] = torch.empty(self.n, dtype=torch.uint8, device=self.device)
        if want_features and features_out is None:
            features_out = torch.empty((self.n, 12), dtype=torch.float32, device=self.device)
        out["features"] = features_out
        if getattr(self, "stats", None) is None:
            self.stats = torch.zeros(4, dtype=torch.int64, device=self.device)
        table = self.teacher_table()
        with torch.cuda.device(self.device):
            rc = self.lib.psk_light_tick(self._p(self.scen), self._p(self.scen_idx), self._p(self.state),
                                         self._p(table), self.max_keys, self._p(actions),
                                         self._p(features_out), self._p(out["expert"]), self._p(out["done"]),
                                         self._p(out["success"]), self._p(self.stats), int(max_timesteps),
                                         self.n, self._stream())
        _lib.check(rc, "psk_light_tick")
        return out

    def rollout(self, ticks, actions=None, features_out=None, out=None, max_timesteps=100):
        """``ticks`` rollout ticks in ONE launch (psk_light_rollout).  actions: u8[ticks, N] or None
        (follow the teacher); features_out: f32[R, N, 12] ring or None (tick t writes frame t % R).
        Returns dict(expert u8[ticks, N], done, success)."""
        torch = self.torch
        actions = self._u8(actions)
        if out is None:
            out = {}
        for k in ("expert", "done", "success"):
            if k not in out or out[k].shape[0] != ticks:
                out[k] = torch.empty((ticks, self.n), dtype=torch.uint8, device=self.device)
        ring = 0
        if features_out is not None:
            assert features_out.dim() == 3 and features_out.is_contiguous() and features_out.dtype == torch.float32
            ring = features_out.shape[0]
        if getattr(self, "stats", None) is None:
            self.stats = torch.zeros(4, dtype=torch.int64, device=self.device)
        table = self.teacher_table()
        with torch.cuda.device(self.device):
            rc = self.lib.psk_light_rollout(self._p(self.scen), self._p(self.scen_idx), self._p(self.state),
                                            self._p(table), self.max_keys, int(ticks), self._p(actions),
                                            self._p(features_out), ring, self._p(out["expert"]),
                                            self._p(out["done"]), self._p(out["success"]), self._p(self.stats),
                                            int(max_timesteps), self.n, self._stream())
        _lib.check(rc, "psk_light_rollout")
        return out

    def check_errors(self):
        flags = int(self.err.item())
        if flags:
            self.err.zero_()
            raise Exception("Unexpected action")
