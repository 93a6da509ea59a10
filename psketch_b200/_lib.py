"""ctypes binding of libpsk_b200.so (include/psk_craft.h).  There is no CPU fallback: if the
shared library is missing or a CUDA device is absent, the ops raise."""
import ctypes
import os

import numpy as np

from . import tables as _tables

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpsk_b200.so")

PSK_OK, PSK_ERR_UNSUPPORTED, PSK_ERR_BADARG, PSK_ERR_CUDA = 0, 1, 2, 3
FLAG_BAD_ACTION, FLAG_INV_OVERFLOW, FLAG_BAD_LEAF, FLAG_OFF_GRID, FLAG_CHAIN_TIMEOUT = 1, 2, 4, 8, 16
AGENT_BYTES = 32
AG_X, AG_Y, AG_DIR, AG_TASK, AG_TIMER = 24, 25, 26, 27, 28
MAX_INV = 24

CRAFT_EXPORTS = (
    "psk_version", "psk_craft_n_features", "psk_craft_supported", "psk_craft_step",
    "psk_craft_features", "psk_craft_satisfies", "psk_craft_expert", "psk_craft_find_closest",
    "psk_craft_reset", "psk_craft_tick", "psk_host_alloc", "psk_host_free",
    "psk_craft_host_create", "psk_craft_host_destroy", "psk_craft_host_set_episodes",
    "psk_craft_host_tick", "psk_craft_sample_scenarios", "psk_craft_sample_positions",
    "psk_random_actions", "psk_craft_rollout", "psk_set_tuning", "psk_get_tuning",
    "psk_craft_features_u8", "psk_craft_host_reset", "psk_craft_host_put_state",
    "psk_craft_host_get_state", "psk_craft_host_tick_resident", "psk_random_actions_block",
    "psk_craft_tick_u8", "psk_craft_rollout_u8", "psk_craft_host_threads", "psk_craft_host_set_threads",
    "psk_host_widen_u8_f32", "psk_debug_chain_skip_ticket", "psk_craft_host_wire_direct",
    "psk_craft_host_set_wire_direct", "psk_craft_host_set_zerocopy_max",
    "psk_debug_wire_split_next",
)
FEATURES_NONE, FEATURES_F32, FEATURES_U8, FEATURES_F32_WIRE_U8 = 0, 1, 2, 3
TICK_PIPELINE, TICK_FUSED, TICK_ADVANCE_FIRST, TICK_STEP_FIRST = 0, 1, 2, 3   # psk_craft_tick orders


class CraftTablesC(ctypes.Structure):
    """Mirror of ``psk_craft_tables`` (include/psk_craft.h)."""
    _fields_ = [
        ("width", ctypes.c_int32), ("height", ctypes.c_int32), ("n_kinds", ctypes.c_int32),
        ("window_w", ctypes.c_int32), ("window_h", ctypes.c_int32),
        ("n_recipes", ctypes.c_int32), ("n_tasks", ctypes.c_int32),
        ("water_kind", ctypes.c_int32), ("stone_kind", ctypes.c_int32),
        ("bridge_kind", ctypes.c_int32), ("axe_kind", ctypes.c_int32),
        ("reserved", ctypes.c_int32),
        ("kind_class", ctypes.c_uint8 * 32),
        ("recipes", ctypes.c_uint8 * (16 * 8)),
        ("task_len", ctypes.c_uint8 * 32),
        ("task_nodes", ctypes.c_uint8 * (32 * 16 * 4)),
        ("ws_recipes", ctypes.c_uint16 * 32),
    ]


class CraftStateC(ctypes.Structure):
    _fields_ = [("grid", ctypes.c_void_p), ("agent", ctypes.c_void_p), ("n", ctypes.c_int64),
                ("cell_stride", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class CraftEpisodesC(ctypes.Structure):
    _fields_ = [("scen_grid", ctypes.c_void_p), ("scen_idx", ctypes.c_void_p),
                ("init_agent", ctypes.c_void_p)]


class PskError(RuntimeError):
    pass


_lib = None


def load():
    """Loads the shared library (building nothing: ``__graft_entry__.build()`` does that)."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("PSK_LIB") or LIB_PATH        # PSK_LIB: experiment builds for same-box A/B runs
    if not os.path.exists(path):
        raise PskError("%s not found — run `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(there is no CPU fallback)" % path)
    lib = ctypes.CDLL(path)
    lib.psk_version.restype = ctypes.c_char_p
    vp, i32 = ctypes.c_void_p, ctypes.c_int32
    tp = ctypes.POINTER(CraftTablesC)
    lib.psk_craft_n_features.argtypes = [tp]
    lib.psk_craft_supported.argtypes = [tp]
    lib.psk_craft_step.argtypes = [tp, CraftStateC, vp, vp, vp, vp, vp]
    lib.psk_craft_features.argtypes = [tp, CraftStateC, vp, i32, vp]
    lib.psk_craft_satisfies.argtypes = [tp, CraftStateC, vp, vp, vp]
    lib.psk_craft_expert.argtypes = [tp, CraftStateC, vp, vp, vp, vp, vp]
    lib.psk_craft_find_closest.argtypes = [tp, CraftStateC, vp, vp, vp, vp, i32, vp]
    lib.psk_craft_reset.argtypes = [CraftStateC, CraftEpisodesC, vp, vp]
    lib.psk_craft_tick.argtypes = [tp, CraftStateC, CraftEpisodesC, vp, vp, vp, vp, vp, vp, vp,
                                   i32, vp]
    i64 = ctypes.c_int64
    lib.psk_craft_rollout.argtypes = [tp, CraftStateC, CraftEpisodesC, i32, vp, vp, i32, vp, vp, vp, vp, vp, vp]
    lib.psk_craft_rollout_u8.argtypes = [tp, CraftStateC, CraftEpisodesC, i32, vp, vp, i32, vp, vp, vp, vp, vp, vp]
    lib.psk_craft_tick_u8.argtypes = [tp, CraftStateC, CraftEpisodesC, vp, vp, vp, vp, vp, vp, vp, i32, vp]
    lib.psk_host_alloc.argtypes = [ctypes.c_size_t]
    lib.psk_host_alloc.restype = ctypes.c_void_p
    lib.psk_host_free.argtypes = [vp]
    lib.psk_host_free.restype = None
    lib.psk_craft_host_create.argtypes = [tp, i64, i64, ctypes.POINTER(vp)]
    lib.psk_craft_host_destroy.argtypes = [vp]
    lib.psk_craft_host_destroy.restype = None
    lib.psk_craft_host_set_episodes.argtypes = [vp, vp, i64, vp, vp, i64]
    lib.psk_craft_host_tick.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i64, vp, vp]
    u64 = ctypes.c_uint64
    lib.psk_craft_sample_scenarios.argtypes = [tp, vp, vp, vp, i32, i32, u64, u64, i64, i32, vp, vp]
    lib.psk_craft_sample_positions.argtypes = [tp, vp, vp, i32, vp, u64, u64, i64, i32, vp, vp]
    lib.psk_random_actions.argtypes = [vp, i64, i32, u64, u64, vp, vp]
    lib.psk_random_actions_block.argtypes = [vp, i64, i32, i32, u64, u64, vp, vp]
    lib.psk_craft_features_u8.argtypes = [tp, CraftStateC, vp, vp]
    lib.psk_craft_host_reset.argtypes = [vp, i64]
    lib.psk_craft_host_put_state.argtypes = [vp, vp, vp, i64]
    lib.psk_craft_host_get_state.argtypes = [vp, vp, vp, i64]
    lib.psk_craft_host_tick_resident.argtypes = [vp, vp, vp, i32, i32, vp, vp, vp, i64, vp, vp]
    lib.psk_debug_chain_skip_ticket.argtypes = [CraftStateC, i64, vp]
    lib.psk_craft_host_threads.argtypes = [vp]
    lib.psk_craft_host_set_threads.argtypes = [vp, i32]
    lib.psk_craft_host_wire_direct.argtypes = [vp]
    lib.psk_craft_host_set_wire_direct.argtypes = [vp, i32]
    lib.psk_craft_host_set_zerocopy_max.argtypes = [vp, i64]
    lib.psk_debug_wire_split_next.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double,
                                              ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
    lib.psk_host_widen_u8_f32.argtypes = [vp, vp, ctypes.c_size_t, ctypes.c_int]
    lib.psk_set_tuning.argtypes = [ctypes.c_char_p, i32]
    lib.psk_get_tuning.argtypes = [ctypes.c_char_p, ctypes.POINTER(i32)]
    for name in CRAFT_EXPORTS[1:]:
        if name not in ("psk_host_alloc", "psk_host_free", "psk_craft_host_destroy"):
            getattr(lib, name).restype = ctypes.c_int
    _lib = lib
    return lib


LIGHT_EXPORTS = ("psk_light_reset", "psk_light_step", "psk_light_features", "psk_light_satisfies",
                 "psk_light_expert", "psk_light_teacher_build", "psk_light_expert_table", "psk_light_tick",
                 "psk_light_rollout")
_light_bound = False


def load_light():
    """Binds the psk_light.h entry points (same shared library)."""
    global _light_bound
    lib = load()
    if not _light_bound:
        vp, i64 = ctypes.c_void_p, ctypes.c_int64
        lib.psk_light_reset.argtypes = [vp, vp, vp, vp, i64, vp]
        lib.psk_light_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, vp]
        lib.psk_light_features.argtypes = [vp, vp, vp, vp, i64, vp]
        lib.psk_light_satisfies.argtypes = [vp, vp, vp, vp, i64, vp]
        lib.psk_light_expert.argtypes = [vp, vp, vp, vp, vp, ctypes.c_int32, i64, vp]
        i32 = ctypes.c_int32
        lib.psk_light_teacher_table_bytes.argtypes = [i64, i32]
        lib.psk_light_teacher_table_bytes.restype = ctypes.c_int64
        lib.psk_light_teacher_build.argtypes = [vp, i64, i32, vp, vp]
        lib.psk_light_expert_table.argtypes = [vp, vp, vp, vp, i32, vp, vp, i64, vp]
        lib.psk_light_tick.argtypes = [vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp, i32, i64, vp]
        lib.psk_light_rollout.argtypes = [vp, vp, vp, vp, i32, i32, vp, vp, i32, vp, vp, vp, vp, i32, i64, vp]
        for name in LIGHT_EXPORTS:
            getattr(lib, name).restype = ctypes.c_int
        _light_bound = True
    return lib


def set_tuning(**knobs):
    """psk_set_tuning for every keyword (value None or -1 = automatic); returns the old values."""
    lib = load()
    old = {}
    for key, value in knobs.items():
        cur = ctypes.c_int32()
        check(lib.psk_get_tuning(key.encode(), ctypes.byref(cur)), "psk_get_tuning(%s)" % key)
        old[key] = cur.value
        check(lib.psk_set_tuning(key.encode(), -1 if value is None else int(value)),
              "psk_set_tuning(%s)" % key)
    return old


def raw_stream(torch, device):
    """cudaStream_t of torch's current stream on ``device`` as a c_void_p — the fast path
    (torch._C._cuda_getCurrentRawStream, no Stream object) where this torch has it."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    get = getattr(torch._C, "_cuda_getCurrentRawStream", None)
    if get is not None:
        return ctypes.c_void_p(get(idx))
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def check_max_timesteps(max_timesteps):
    """The episode timer is one byte of the agent record (include/psk_craft.h: PSK_AG_TIMER); the
    reference's is an unbounded Python int (trainers/imitation.py:30)."""
    t = int(max_timesteps)
    if not 0 < t <= 255:
        raise ValueError("max_timesteps must be in 1..255 (u8 timer in the agent record), got %r"
                         % (max_timesteps,))
    return t


def check_agent_inputs(tables, inv=None, pos=None, dirs=None, task=None, scen_idx=None, n_scen=None):
    """Rejects caller state that does not fit the agent record (include/psk_craft.h) before anything
    is allocated: numpy would wrap a count or a position of 300 into the u8 record as 44, and the
    kernels trust positions and scenario indices as row offsets (they never raise PSK_FLAG_OFF_GRID),
    so an off-grid position or a scenario index out of range would read outside the env's rows."""
    def bad(name, a, lo, hi):
        a = np.asarray(a)
        if a.size == 0:
            return
        if a.dtype.kind not in "iub" and not np.array_equal(a, np.floor(a)):
            raise ValueError("%s must be whole numbers" % name)
        if a.min() < lo or a.max() > hi:
            raise ValueError("%s must be in %d..%d, got values in %s..%s" % (name, lo, hi, a.min(), a.max()))
    if inv is not None:
        inv = np.asarray(inv)
        if inv.ndim != 2 or inv.shape[1] > min(tables.K, MAX_INV):
            raise ValueError("inventory must be [n, <= %d], got shape %s" % (tables.K, inv.shape))
        bad("inventory counts", inv, 0, 255)
    if pos is not None:
        pos = np.asarray(pos)
        if pos.ndim != 2 or pos.shape[1] != 2:
            raise ValueError("positions must be [n, 2], got shape %s" % (pos.shape,))
        bad("x positions", pos[:, 0], 0, tables.W - 1)
        bad("y positions", pos[:, 1], 0, tables.H - 1)
    if dirs is not None:
        bad("facing directions", dirs, 0, 3)
    if task is not None:
        bad("task ids", task, 0, tables.n_tasks - 1)
    if scen_idx is not None:
        bad("scenario indices", scen_idx, 0, n_scen - 1)


def check_light_inputs(board, n_keys, scen_idx, state=None):
    """Rejects Light envs that the kernels (include/psk_light.h) would read outside their tables
    for, before anything reaches the device.  ``board`` i32[S, 2] = board_w, board_h and ``n_keys``
    i32[S] per scenario; ``scen_idx`` [n]; ``state`` [n, 4] = x, y, key mask, steps of the episode.
    A scenario index selects a record and a table block; a position off the board, or a mask with a
    bit for a key the scenario does not have, is no state of the scenario (the teacher table has no
    entry for it); the step counter must leave room for one more step below 255."""
    board = np.asarray(board).reshape(-1, 2)
    n_keys = np.asarray(n_keys).reshape(-1)

    def whole(name, a):
        a = np.asarray(a)
        if a.size and a.dtype.kind not in "iub" and not np.array_equal(a, np.floor(a)):
            raise ValueError("%s must be whole numbers" % name)
        return a.astype(np.int64)
    si = whole("scenario indices", scen_idx).reshape(-1)
    if si.size and (si.min() < 0 or si.max() >= len(board)):
        raise ValueError("scenario indices must be in 0..%d, got values in %d..%d"
                         % (len(board) - 1, si.min(), si.max()))
    if state is None:
        return
    st = whole("Light states", state)
    if st.shape != (len(si), 4):
        raise ValueError("Light state must be [%d, 4], got shape %s" % (len(si), st.shape))
    if st.size and (st.min() < 0 or st.max() > 255):
        raise ValueError("Light state bytes must be in 0..255, got values in %d..%d" % (st.min(), st.max()))
    bad = np.flatnonzero((st[:, 0] >= board[si, 0]) | (st[:, 1] >= board[si, 1]))
    if bad.size:
        e = bad[0]
        raise ValueError("env %d: position (%d, %d) is off its %d x %d board"
                         % (e, st[e, 0], st[e, 1], board[si[e], 0], board[si[e], 1]))
    bad = np.flatnonzero(st[:, 2] >> n_keys[si])
    if bad.size:
        e = bad[0]
        raise ValueError("env %d: key mask %#x has bits at or above its scenario's %d keys"
                         % (e, st[e, 2], n_keys[si[e]]))
    bad = np.flatnonzero(st[:, 3] >= 255)
    if bad.size:
        raise ValueError("env %d: step counter %d must be below 255" % (bad[0], st[bad[0], 3]))


def check(rc, what):
    if rc == PSK_OK:
        return
    msg = {PSK_ERR_UNSUPPORTED: "unsupported world geometry", PSK_ERR_BADARG: "bad argument",
           PSK_ERR_CUDA: "CUDA launch failed"}.get(rc, "error %d" % rc)
    raise PskError("%s: %s" % (what, msg))


def make_tables(t):
    """psketch_b200.tables.CraftTables -> CraftTablesC."""
    c = CraftTablesC()
    c.width, c.height, c.n_kinds = t.W, t.H, t.K
    c.window_w, c.window_h = t.win_w, t.win_h
    c.n_recipes, c.n_tasks = t.n_recipes, t.n_tasks
    c.water_kind, c.stone_kind = t.water_kind, t.stone_kind
    c.bridge_kind, c.axe_kind = t.bridge_kind, t.axe_kind
    ctypes.memmove(c.kind_class, np.ascontiguousarray(t.kind_class[:32]).ctypes.data, 32)
    ctypes.memmove(c.recipes, np.ascontiguousarray(t.recipes).ctypes.data, 16 * 8)
    ctypes.memmove(c.task_len, np.ascontiguousarray(t.task_len[:32]).ctypes.data, 32)
    ctypes.memmove(c.task_nodes, np.ascontiguousarray(t.task_nodes[:32]).ctypes.data, 32 * 16 * 4)
    assert _tables.MAX_TASKS == 32 and _tables.MAX_TASK_NODES == 16
    rec = np.asarray(t.recipes)
    for r in range(int(t.n_recipes)):                 # recipes[r] = out, workshop, n_in, ...
        c.ws_recipes[int(rec[r][1]) & 31] |= 1 << r
    return c
