"""HostCraft — the batched tick for callers whose environments live in HOST memory.

This is the end-to-end entry point for a CPU-resident caller (the reference keeps every
CraftState on the CPU): numpy arrays in pinned memory go through ``psk_craft_host_tick``
(include/psk_craft.h), which pipelines H2D copies, the fused tick kernel and D2H copies over
several CUDA streams.  No torch tensors cross this boundary.
"""
import ctypes
import os

import numpy as np

from . import _lib
from .tables import CraftTables


def _np_ptr(a):
    return ctypes.c_void_p(a.ctypes.data) if a is not None else None


class PinnedArray(object):
    """numpy view over cudaHostAlloc'ed memory (freed when the object dies)."""

    def __init__(self, lib, shape, dtype):
        self.lib = lib
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        self.ptr = lib.psk_host_alloc(max(self.nbytes, 1))
        if not self.ptr:
            raise _lib.PskError("psk_host_alloc(%d) failed" % self.nbytes)
        buf = (ctypes.c_uint8 * max(self.nbytes, 1)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def __del__(self):
        try:
            if self.ptr:
                self.lib.psk_host_free(ctypes.c_void_p(self.ptr))
                self.ptr = None
        except Exception:
            pass


class HostCraft(object):
    def __init__(self, tables, scen_grids, scen_idx, init_pos, task, init_dir=None,
                 max_timesteps=40, chunk_envs=16384, host_threads=None):
        """host_threads: threads that widen the u8 wire frame (``features="f32_wire_u8"``), this one
        included; default min(8, cores / 2) divided among the ranks torchrun started on this box."""
        self.tables = tables if tables is not None else CraftTables()
        _lib.check_agent_inputs(self.tables, pos=init_pos, dirs=init_dir, task=task, scen_idx=scen_idx,
                                n_scen=len(scen_grids))
        self.lib = _lib.load()
        self.ct = _lib.make_tables(self.tables)
        t = self.tables
        scen_grids = np.asarray(scen_grids, np.uint8)
        scen_idx = np.ascontiguousarray(scen_idx, np.int32)
        self.n = n = len(scen_idx)
        self.C = t.W * t.H
        self.cell_stride = cs = ((self.C + 63) // 64) * 64
        self.n_features = t.n_features
        sg = np.zeros((len(scen_grids), cs), np.uint8)
        sg[:, :self.C] = scen_grids
        ia = np.zeros((n, _lib.AGENT_BYTES), np.uint8)
        init_pos = np.asarray(init_pos)
        ia[:, _lib.AG_X], ia[:, _lib.AG_Y] = init_pos[:, 0], init_pos[:, 1]
        ia[:, _lib.AG_DIR] = 0 if init_dir is None else np.asarray(init_dir)
        ia[:, _lib.AG_TASK] = np.asarray(task)
        ia[:, _lib.AG_TIMER] = _lib.check_max_timesteps(max_timesteps)
        ctx = ctypes.c_void_p()
        _lib.check(self.lib.psk_craft_host_create(ctypes.byref(self.ct), n, chunk_envs,
                                                  ctypes.byref(ctx)), "psk_craft_host_create")
        self.ctx = ctx
        ce = min(int(chunk_envs) if chunk_envs and chunk_envs > 0 else 16384, n)
        self.chunk_envs = (ce + 127) // 128 * 128       # as psk_craft_host_create rounds it
        self.last_wire_direct = 0
        if host_threads is None:
            local = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
            host_threads = max(1, min(8, (os.cpu_count() or 2) // 2 // local))
        _lib.check(self.lib.psk_craft_host_set_threads(self.ctx, int(host_threads)), "psk_craft_host_set_threads")
        _lib.check(self.lib.psk_craft_host_set_episodes(self.ctx, _np_ptr(sg), len(sg),
                                                        _np_ptr(scen_idx), _np_ptr(ia), n),
                   "psk_craft_host_set_episodes")
        # pinned host-side state and outputs
        self._pins = {k: PinnedArray(self.lib, shape, dt) for k, (shape, dt) in dict(
            grid=((n, cs), np.uint8), agent=((n, _lib.AGENT_BYTES), np.uint8),
            features=((n, self.n_features), np.float32), expert=((n,), np.uint8),
            done=((n,), np.uint8), success=((n,), np.uint8), action=((n,), np.uint8)).items()}
        self.grid = self._pins["grid"].array
        self.agent = self._pins["agent"].array
        self.features = self._pins["features"].array
        self.expert = self._pins["expert"].array
        self.done = self._pins["done"].array
        self.success = self._pins["success"].array
        self.action = self._pins["action"].array
        self.grid[:] = sg[scen_idx]
        self.agent[:] = ia
        self.stats = np.zeros(4, np.uint64)
        self.err = np.zeros(1, np.int32)
        self.resident = False
        self._features_u8 = None
        self.last_h2d = self.last_d2h = 0
        self._ptrs = {}

    def _raise_flags(self):
        """What the reference would have raised (worlds/craft.py:415-416, demonstration.py:18)."""
        flags = int(self.err[0])
        if not flags:
            return
        self.err[0] = 0
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

    def tick(self, actions=None, want_features=True):
        """State round trip per call (psk_craft_host_tick): grid / agent go up, come back advanced."""
        if self.resident:
            raise _lib.PskError("state is resident on the device: use tick_resident() or download()")
        if actions is not None:
            self.action[:] = actions
        rc = self.lib.psk_craft_host_tick(
            self.ctx, _np_ptr(self.grid), _np_ptr(self.agent),
            _np_ptr(self.action) if actions is not None else None,
            _np_ptr(self.features) if want_features else None, _np_ptr(self.expert),
            _np_ptr(self.done), _np_ptr(self.success), self.n, _np_ptr(self.stats),
            _np_ptr(self.err))
        _lib.check(rc, "psk_craft_host_tick")
        self.last_h2d = self.h2d_bytes + (self.n if actions is not None else 0)
        self.last_d2h = self.d2h_bytes - (0 if want_features else self.n * self.n_features * 4)
        self._raise_flags()
        return self.expert

    # ---- resident mode: the environments stay in HBM between ticks
    def reset_resident(self):
        """Every env at its episode start, on the device (world.init_state for the batch)."""
        _lib.check(self.lib.psk_craft_host_reset(self.ctx, self.n), "psk_craft_host_reset")
        self.resident = True

    def upload(self):
        """Host state (self.grid / self.agent) -> device; switches to resident mode."""
        _lib.check(self.lib.psk_craft_host_put_state(self.ctx, _np_ptr(self.grid),
                                                     _np_ptr(self.agent), self.n),
                   "psk_craft_host_put_state")
        self.resident = True

    def download(self, keep_resident=True):
        """Device state -> self.grid / self.agent (e.g. for state.pos / state.inventory)."""
        _lib.check(self.lib.psk_craft_host_get_state(self.ctx, _np_ptr(self.grid),
                                                     _np_ptr(self.agent), self.n),
                   "psk_craft_host_get_state")
        self.resident = keep_resident

    @property
    def features_u8(self):
        if self._features_u8 is None:
            self._pins["features_u8"] = PinnedArray(self.lib, (self.n, self.n_features), np.uint8)
            self._features_u8 = self._pins["features_u8"].array
        return self._features_u8

    def _p(self, a):
        """c_void_p of a numpy array; the arrays handed over call after call are looked up once
        (``ndarray.ctypes`` builds a new helper object on every access: ~1.5 us per pointer)."""
        if a is None:
            return None
        hit = self._ptrs.get(id(a))
        if hit is None or hit[0] is not a:
            if len(self._ptrs) > 32:
                self._ptrs.clear()
            hit = self._ptrs[id(a)] = (a, ctypes.c_void_p(a.ctypes.data))
        return hit[1]

    def tick_resident(self, actions=None, features="f32", advance_first=False):
        """psk_craft_host_tick_resident: only actions go up; features (``"f32"`` -> self.features,
        ``"u8"`` -> self.features_u8, ``"f32_wire_u8"`` -> self.features again, but PCIe carries the
        byte frame and host threads widen it; None), teacher actions and flags come down.
        ``advance_first``: step with ``actions`` (None = no step), THEN observe — the order of a host
        policy in the loop: ``a = policy(env.features); env.tick_resident(a, advance_first=True)``."""
        if not self.resident:
            self.upload()
        if actions is not None:
            self.action[:] = actions
        direct = self.wire_direct if features == "f32_wire_u8" else 0
        fmt = {None: _lib.FEATURES_NONE, "f32": _lib.FEATURES_F32, "u8": _lib.FEATURES_U8,
               "f32_wire_u8": _lib.FEATURES_F32_WIRE_U8}[features]
        buf = {None: None, "f32": self.features, "f32_wire_u8": self.features}.get(features)
        if features == "u8":
            buf = self.features_u8
        p = self._p
        rc = self.lib.psk_craft_host_tick_resident(
            self.ctx, p(self.action) if actions is not None else None, p(buf), fmt,
            1 if advance_first else 0, p(self.expert), p(self.done), p(self.success), self.n,
            p(self.stats), p(self.err))
        _lib.check(rc, "psk_craft_host_tick_resident")
        self.last_h2d = self.n if actions is not None else 0
        wire = 0 if buf is None else buf.nbytes
        if features == "f32_wire_u8":       # bytes for the leading chunks, f32 for the last `direct` ones
            chunks = -(-self.n // self.chunk_envs)
            direct = min(direct, chunks) if buf.ctypes.data == self._pins["features"].ptr else 0
            n_f32 = 0 if direct == 0 else self.n - (chunks - direct) * self.chunk_envs
            wire = (self.n - n_f32) * self.n_features + n_f32 * self.n_features * 4
            self.last_wire_direct = direct
        self.last_d2h = self.n * 3 + wire + 36
        self._raise_flags()
        return self.expert

    @property
    def wire_direct(self):
        """Chunks of the next ``f32_wire_u8`` call that cross PCIe as f32 instead of bytes (the split
        follows the measured PCIe and widening rates unless ``set_wire_direct`` fixed it)."""
        return int(self.lib.psk_craft_host_wire_direct(self.ctx))

    def set_wire_direct(self, chunks=-1):
        """Fix the number of trailing f32 chunks of ``f32_wire_u8`` calls; -1 = adaptive (default)."""
        _lib.check(self.lib.psk_craft_host_set_wire_direct(self.ctx, int(chunks)), "psk_craft_host_set_wire_direct")

    def set_zerocopy_max(self, max_envs=2048):
        """Calls of at most ``max_envs`` envs whose buffers are all pinned run as ONE launch that reads
        and writes host memory itself (0 = always the copy-engine route)."""
        _lib.check(self.lib.psk_craft_host_set_zerocopy_max(self.ctx, int(max_envs)), "psk_craft_host_set_zerocopy_max")

    @property
    def h2d_bytes(self):
        return self.n * (self.cell_stride + _lib.AGENT_BYTES)

    @property
    def d2h_bytes(self):
        return self.n * (self.n_features * 4 + 3 + self.cell_stride + _lib.AGENT_BYTES)

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.psk_craft_host_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
