"""VecCraft — the batched Craft environment + teacher, state resident in HBM.

Host-side mirror of the reference's per-object API for N environments at once:

    reference (one env)                               VecCraft (N envs, one launch)
    world.init_state(grid, pos, dir)    craft.py:258  VecCraft.from_instances(...) / reset()
    state.step(a) -> (0, state')        craft.py:332  step(actions)
    state.features()                    craft.py:296  features()
    state.satisfies(task)               craft.py:285  satisfies()
    teacher(task, state)         demonstration.py:9   expert()
    teacher.find_closest_resources      base.py:27    find_closest(kind)
    do_rollout loop body            imitation.py:42   tick()

PyTorch owns the device memory and the stream; all arithmetic happens in libpsk_b200.so
(psketch_b200/csrc/psk_craft.cu) through the C ABI of include/psk_craft.h.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .tables import CraftTables


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


class VecCraft(object):
    def __init__(self, tables, n, device=None, max_timesteps=40):
        if not torch.cuda.is_available():
            raise _lib.PskError("VecCraft needs a CUDA device (there is no CPU fallback)")
        self.lib = _lib.load()
        self.tables = tables if tables is not None else CraftTables()
        self.ct = _lib.make_tables(self.tables)
        if not self.lib.psk_craft_supported(ctypes.byref(self.ct)):
            raise _lib.PskError("world geometry %dx%d window %dx%d with %d kinds is outside what libpsk_b200 "
                                "runs: 1 <= WIDTH, HEIGHT <= 64, odd WINDOW_WIDTH / WINDOW_HEIGHT from 1 to 9, "
                                "at most 24 kinds"
                                % (self.tables.W, self.tables.H, self.tables.win_w, self.tables.win_h,
                                   self.tables.K))
        self.device = torch.device(device if device is not None else
                                   "cuda:%d" % torch.cuda.current_device())
        self.n = int(n)
        self.W, self.H, self.K = self.tables.W, self.tables.H, self.tables.K
        self.C = self.W * self.H
        self.cell_stride = ((self.C + 63) // 64) * 64
        self.n_features = self.tables.n_features
        self.max_timesteps = _lib.check_max_timesteps(max_timesteps)
        dev = self.device
        self.grid = torch.zeros((self.n, self.cell_stride), dtype=torch.uint8, device=dev)
        self.agent = torch.zeros((self.n, _lib.AGENT_BYTES), dtype=torch.uint8, device=dev)
        self.scen_grid = None
        self.scen_idx = None
        self.init_agent = None
        self.err_flags = torch.zeros(1, dtype=torch.int32, device=dev)
        self.stats = torch.zeros(4, dtype=torch.int64, device=dev)
        self._reward = None

    # ------------------------------------------------------------------ construction
    @classmethod
    def from_instances(cls, tables, scen_grids, scen_idx, init_pos, task, init_dir=None,
                       max_timesteps=40, device=None):
        """scen_grids u8[S, W*H] kind ids (cell (x,y) at x*H+y); scen_idx int[N]; init_pos
        int[N,2]; task int[N] (task id = 1-based position in the hint file)."""
        tables = tables if tables is not None else CraftTables()
        _lib.check_agent_inputs(tables, pos=init_pos, dirs=init_dir, task=task, scen_idx=scen_idx,
                                n_scen=len(scen_grids))
        scen_grids = np.asarray(scen_grids, np.uint8)
        scen_idx = np.asarray(scen_idx, np.int32)
        n = len(scen_idx)
        env = cls(tables, n, device=device, max_timesteps=max_timesteps)
        S, C = scen_grids.shape
        assert C == env.C, "grid has %d cells, world needs %d" % (C, env.C)
        sg = np.zeros((S, env.cell_stride), np.uint8)
        sg[:, :C] = scen_grids
        ia = np.zeros((n, _lib.AGENT_BYTES), np.uint8)
        init_pos = np.asarray(init_pos)
        ia[:, _lib.AG_X] = init_pos[:, 0]
        ia[:, _lib.AG_Y] = init_pos[:, 1]
        ia[:, _lib.AG_DIR] = 0 if init_dir is None else np.asarray(init_dir)
        ia[:, _lib.AG_TASK] = np.asarray(task)
        ia[:, _lib.AG_TIMER] = max_timesteps
        env.scen_grid = torch.from_numpy(sg).to(env.device)
        env.scen_idx = torch.from_numpy(scen_idx).to(env.device)
        env.init_agent = torch.from_numpy(ia).to(env.device)
        env.reset()
        return env

    @classmethod
    def from_states(cls, tables, grid, inv, pos, dirs, task=None, max_timesteps=40, device=None):
        """Arbitrary states (e.g. exported from the reference): every env is its own scenario."""
        tables = tables if tables is not None else CraftTables()
        _lib.check_agent_inputs(tables, inv=inv, pos=pos, dirs=dirs, task=task)
        grid = np.asarray(grid, np.uint8)
        n = len(grid)
        env = cls(tables, n, device=device, max_timesteps=max_timesteps)
        g = np.zeros((n, env.cell_stride), np.uint8)
        g[:, :env.C] = grid
        ag = np.zeros((n, _lib.AGENT_BYTES), np.uint8)
        inv = np.asarray(inv)
        ag[:, :inv.shape[1]] = inv
        pos = np.asarray(pos)
        ag[:, _lib.AG_X] = pos[:, 0]
        ag[:, _lib.AG_Y] = pos[:, 1]
        ag[:, _lib.AG_DIR] = np.asarray(dirs)
        ag[:, _lib.AG_TASK] = 0 if task is None else np.asarray(task)
        ag[:, _lib.AG_TIMER] = max_timesteps
        env.scen_grid = torch.from_numpy(g).to(env.device)
        env.scen_idx = torch.arange(n, dtype=torch.int32, device=env.device)
        env.init_agent = torch.from_numpy(ag).to(env.device)
        env.reset()
        return env

    # ------------------------------------------------------------------ C structs
    def _state(self):
        return _lib.CraftStateC(self.grid.data_ptr(), self.agent.data_ptr(), self.n,
                                self.cell_stride, 0)

    def _episodes(self):
        return _lib.CraftEpisodesC(self.scen_grid.data_ptr(), self.scen_idx.data_ptr(),
                                   self.init_agent.data_ptr())

    def _stream(self):
        return _lib.raw_stream(torch, self.device)

    def _u8(self, x):
        if x is None:
            return None
        if not torch.is_tensor(x):
            x = torch.as_tensor(np.asarray(x, np.uint8))
        return x.to(device=self.device, dtype=torch.uint8).contiguous()

    # ------------------------------------------------------------------ ops
    def reset(self, mask=None):
        mask = self._u8(mask)
        with torch.cuda.device(self.device):
            rc = self.lib.psk_craft_reset(self._state(), self._episodes(), _ptr(mask), self._stream())
        _lib.check(rc, "psk_craft_reset")

    def step(self, actions, active=None):
        """CraftState.step for every env, in place; returns the (all-zero) reward f32[N]."""
        actions, active = self._u8(actions), self._u8(active)
        if self._reward is None:
            self._reward = torch.empty(self.n, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.psk_craft_step(ctypes.byref(self.ct), self._state(), _ptr(actions),
                                         _ptr(active), _ptr(self._reward), _ptr(self.err_flags),
                                         self._stream())
        _lib.check(rc, "psk_craft_step")
        return self._reward

    def features(self, out=None, impl=0):
        if out is None:
            out = torch.empty((self.n, self.n_features), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.psk_craft_features(ctypes.byref(self.ct), self._state(), _ptr(out),
                                             int(impl), self._stream())
        _lib.check(rc, "psk_craft_features")
        return out

    def features_u8(self, out=None):
        """The feature rows as bytes, u8[N, n_features] (psk_craft_features_u8): every feature is an
        exact integer <= 255, so ``out.float()`` equals ``features()``."""
        if out is None:
            out = torch.empty((self.n, self.n_features), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.psk_craft_features_u8(ctypes.byref(self.ct), self._state(), _ptr(out),
                                                self._stream())
        _lib.check(rc, "psk_craft_features_u8")
        return out

    def satisfies(self, task=None):
        """u8[N]: 1 True, 0 False, 2 None (goal names other than get/make/go)."""
        task = self._u8(task)
        out = torch.empty(self.n, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.psk_craft_satisfies(ctypes.byref(self.ct), self._state(), _ptr(task),
                                              _ptr(out), self._stream())
        _lib.check(rc, "psk_craft_satisfies")
        return out

    def expert(self, task=None, want_dist=False, out=None):
        task = self._u8(task)
        if out is None:
            out = torch.empty(self.n, dtype=torch.uint8, device=self.device)
        dist = torch.empty(self.n, dtype=torch.int16, device=self.device) if want_dist else None
        with torch.cuda.device(self.device):
            rc = self.lib.psk_craft_expert(ctypes.byref(self.ct), self._state(), _ptr(task),
                                           _ptr(out), _ptr(dist), _ptr(self.err_flags),
                                           self._stream())
        _lib.check(rc, "psk_craft_expert")
        return (out, dist) if want_dist else out

    def find_closest(self, kind, seq_cap=0):
        """goal u8[N,2], length i16[N], seq u8[N,seq_cap] or None."""
        kind = self._u8(kind)
        goal = torch.empty((self.n, 2), dtype=torch.uint8, device=self.device)
        length = torch.empty(self.n, dtype=torch.int16, device=self.device)
        seq = (torch.empty((self.n, seq_cap), dtype=torch.uint8, device=self.device)
               if seq_cap else None)
        with torch.cuda.device(self.device):
            rc = self.lib.psk_craft_find_closest(ctypes.byref(self.ct), self._state(), _ptr(kind),
                                                 _ptr(goal), _ptr(length), _ptr(seq),
                                                 int(seq_cap), self._stream())
        _lib.check(rc, "psk_craft_find_closest")
        return goal, length, seq

    def tick(self, actions=None, features_out=None, want_features=True, fused=True, out=None,
             advance_first=False):
        """One rollout tick (see psk_craft_tick).  Returns dict(expert, done, success, features).
        ``advance_first``: "step, then observe" — ``actions`` (None = no step) are applied first and
        expert / features describe the state AFTER the step (PSK_TICK_ADVANCE_FIRST): the order a
        policy in the loop needs, one launch per timestep.  A ``features_out`` tensor of dtype uint8
        selects the compact byte frame (psk_craft_tick_u8)."""
        actions = self._u8(actions)
        if out is None:
            out = {}
        for k in ("expert", "done", "success"):
            if k not in out:
                out[k] = torch.empty(self.n, dtype=torch.uint8, device=self.device)
        if want_features and features_out is None:
            features_out = torch.empty((self.n, self.n_features), dtype=torch.float32,
                                       device=self.device)
        out["features"] = features_out
        order = 2 if advance_first else (1 if fused else 0)
        with torch.cuda.device(self.device):
            if features_out is not None and features_out.dtype == torch.uint8:
                rc = self.lib.psk_craft_tick_u8(ctypes.byref(self.ct), self._state(), self._episodes(),
                                                _ptr(actions), _ptr(features_out), _ptr(out["expert"]),
                                                _ptr(out["done"]), _ptr(out["success"]), _ptr(self.stats),
                                                _ptr(self.err_flags), order or 1, self._stream())
            else:
                rc = self.lib.psk_craft_tick(ctypes.byref(self.ct), self._state(), self._episodes(),
                                             _ptr(actions), _ptr(features_out), _ptr(out["expert"]),
                                             _ptr(out["done"]), _ptr(out["success"]),
                                             _ptr(self.stats), _ptr(self.err_flags), order, self._stream())
        _lib.check(rc, "psk_craft_tick")
        return out

    def step_observe(self, actions=None, features_out=None, out=None):
        """One launch of PSK_TICK_STEP_FIRST: ``actions`` (None = no step) go through CraftState.step
        alone — no timer, no done, no auto-reset, STOP is the idle action — then the teacher's action
        and the features of the NEW states.  The language trainers' decoding step
        (trainers/primitive_language.py:47-70).  A ``features_out`` tensor of dtype uint8 selects the
        byte frame.  Returns dict(expert u8[N], features)."""
        actions = self._u8(actions)
        if out is None:
            out = {}
        if "expert" not in out:
            out["expert"] = torch.empty(self.n, dtype=torch.uint8, device=self.device)
        if features_out is None:
            features_out = torch.empty((self.n, self.n_features), dtype=torch.float32, device=self.device)
        out["features"] = features_out
        entry = self.lib.psk_craft_tick_u8 if features_out.dtype == torch.uint8 else self.lib.psk_craft_tick
        with torch.cuda.device(self.device):
            rc = entry(ctypes.byref(self.ct), self._state(), self._episodes(), _ptr(actions),
                       _ptr(features_out), _ptr(out["expert"]), None, None, None, _ptr(self.err_flags),
                       _lib.TICK_STEP_FIRST, self._stream())
        _lib.check(rc, "psk_craft_tick")
        return out

    def rollout(self, ticks, actions=None, features_out=None, out=None, want_flags=True):
        """``ticks`` rollout ticks in one launch (psk_craft_rollout).  actions: u8[ticks, N] or None
        (follow the teacher); features_out: f32[R, N, n_features] ring or None.  Returns
        dict(expert u8[ticks, N], done, success)."""
        actions = self._u8(actions)
        if out is None:
            out = {}
        keys = ("expert", "done", "success") if want_flags else ("expert",)
        for k in keys:
            if k not in out or out[k].shape[0] != ticks:
                out[k] = torch.empty((ticks, self.n), dtype=torch.uint8, device=self.device)
        ring = 0
        if features_out is not None:
            assert features_out.dim() == 3 and features_out.is_contiguous()
            ring = features_out.shape[0]
        entry = (self.lib.psk_craft_rollout_u8 if features_out is not None and features_out.dtype == torch.uint8
                 else self.lib.psk_craft_rollout)            # byte frames: u8[R, N, n_features]
        with torch.cuda.device(self.device):
            rc = entry(ctypes.byref(self.ct), self._state(), self._episodes(),
                                            int(ticks), _ptr(actions), _ptr(features_out), ring,
                                            _ptr(out["expert"]), _ptr(out.get("done")),
                                            _ptr(out.get("success")), _ptr(self.stats),
                                            _ptr(self.err_flags), self._stream())
        _lib.check(rc, "psk_craft_rollout")
        return out

    def random_actions(self, t=0, seed=123, out=None, device_clock=False, ticks=None):
        """u8[N] uniform actions from Philox(seed, counter=(env, t)) — off-policy rollouts; with
        ``ticks`` u8[ticks, N], row k from clock t + k (the ``actions`` block of ``rollout``).
        device_clock=True adds the env-step counter (stats[2]) to t on the device, so a captured
        CUDA graph draws fresh actions on every replay."""
        shape = (self.n,) if ticks is None else (int(ticks), self.n)
        if out is None:
            out = torch.empty(shape, dtype=torch.uint8, device=self.device)
        clock = ctypes.c_void_p(self.stats.data_ptr() + 16) if device_clock else None
        with torch.cuda.device(self.device):
            rc = self.lib.psk_random_actions_block(_ptr(out), self.n, 1 if ticks is None else int(ticks), 6,
                                                   ctypes.c_uint64(seed), ctypes.c_uint64(t), clock,
                                                   self._stream())
        _lib.check(rc, "psk_random_actions_block")
        return out

    # ------------------------------------------------------------------ views / checks
    @property
    def pos(self):
        return self.agent[:, _lib.AG_X:_lib.AG_Y + 1]

    @property
    def dir(self):
        return self.agent[:, _lib.AG_DIR]

    @property
    def task(self):
        return self.agent[:, _lib.AG_TASK]

    @property
    def timer(self):
        return self.agent[:, _lib.AG_TIMER]

    @property
    def inventory(self):
        return self.agent[:, :self.K]

    @property
    def cells(self):
        return self.grid[:, :self.C]

    def snapshot(self):
        return self.grid.clone(), self.agent.clone()

    def restore(self, snap):
        self.grid.copy_(snap[0])
        self.agent.copy_(snap[1])

    def check_errors(self):
        """Raises what the reference would have raised for conditions seen by the kernels."""
        flags = int(self.err_flags.item())
        if not flags:
            return
        self.err_flags.zero_()
        if flags & _lib.FLAG_CHAIN_TIMEOUT:   # before anything else: the outputs of that call are suspect
            raise _lib.PskError("tile chain timeout: a previous fused launch on these envs never finished "
                                "(aborted launch?); the kernel went on instead of hanging")
        if flags & _lib.FLAG_BAD_LEAF:        # the teacher speaks before the step (imitation.py:53,72)
            raise AssertionError("teacher: subtask is neither 'use' nor 'go', or every subtask of an "
                                 "unsatisfied task is satisfied")  # demonstration.py:18, base.py:23-24
        if flags & _lib.FLAG_BAD_ACTION:
            raise Exception("Unexpected action")              # worlds/craft.py:415-416
        if flags & _lib.FLAG_INV_OVERFLOW:
            raise OverflowError("inventory count above 255")
        raise _lib.PskError("kernel error flags 0x%x" % flags)
