"""ctypes front-end of sampler_oracle.c — TEST INFRASTRUCTURE ONLY."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "liborc_sampler.so")
_lib = None


def build(force=False):
    src = os.path.join(_HERE, "sampler_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        subprocess.check_call(["gcc", "-O2", "-fopenmp", "-fPIC", "-shared", "-o", _SO, src, "-lm"])
    return _SO


def _load():
    global _lib
    if _lib is None:
        lib = ctypes.CDLL(build())
        vp, i32, i64, u64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_uint64
        lib.orc_philox_block.argtypes = [vp, vp, vp]
        lib.orc_philox_block.restype = None
        lib.orc_below.argtypes = [ctypes.c_uint32, i32]
        lib.orc_below.restype = i32
        lib.orc_rule_violations.argtypes = [vp, i32, i32]
        lib.orc_rule_violations.restype = i32
        lib.orc_sample_scenarios.argtypes = [i32, i32, vp, i32, i32, u64, u64, i64, i32, vp, vp]
        lib.orc_sample_scenarios.restype = i64
        lib.orc_sample_positions.argtypes = [i32, i32, vp, vp, i32, u64, u64, i64, i32, vp]
        lib.orc_sample_positions.restype = i64
        lib.orc_random_actions.argtypes = [vp, i64, i32, i32, u64, u64]
        lib.orc_random_actions.restype = None
        _lib = lib
    return _lib


def _p(a):
    return ctypes.c_void_p(a.ctypes.data)


def cell_stride(W, H):
    return ((W * H + 63) // 64) * 64


def philox_block(ctr, key):
    """The raw Philox4x32-10 block: four counter words, two key words -> four output words."""
    c = np.ascontiguousarray(ctr, np.uint32)
    k = np.ascontiguousarray(key, np.uint32)
    out = np.zeros(4, np.uint32)
    _load().orc_philox_block(_p(c), _p(k), _p(out))
    return out


def below(word, n):
    return int(_load().orc_below(int(word), int(n)))


def rule_violations(occupied):
    """Acceptance rule of a grid occupied[W, H] (bool): 0 if it holds, bit 0 = (i) the free cells
    are not all connected, bit 1 = (ii) an occupied interior cell has no free neighbour."""
    occ = np.ascontiguousarray(occupied, np.uint8)
    W, H = occ.shape
    return int(_load().orc_rule_violations(_p(occ), W, H))


def sample_scenarios(W, H, place_kinds, boundary_kind, seed, offset, n):
    """(grid u8[n, cell_stride], init_pos u8[n, 2], n_failed) as psk_craft_sample_scenarios."""
    cs = cell_stride(W, H)
    pk = np.ascontiguousarray(place_kinds, np.uint8)
    grid = np.empty((n, cs), np.uint8)
    pos = np.empty((n, 2), np.uint8)
    fails = _load().orc_sample_scenarios(W, H, _p(pk), len(pk), int(boundary_kind), ctypes.c_uint64(seed),
                                         ctypes.c_uint64(offset), n, cs, _p(grid), _p(pos))
    return grid, pos, int(fails)


def sample_positions(W, H, scen_grid, group_scen, per_group, seed, offset=0):
    """(u8[n_groups, per_group, 2], n_failed) as psk_craft_sample_positions."""
    sg = np.ascontiguousarray(scen_grid, np.uint8)
    gs = np.ascontiguousarray(group_scen, np.int32)
    out = np.empty((len(gs), per_group, 2), np.uint8)
    fails = _load().orc_sample_positions(W, H, _p(sg), _p(gs), per_group, ctypes.c_uint64(seed),
                                         ctypes.c_uint64(offset), len(gs), sg.shape[1], _p(out))
    return out, int(fails)


def random_actions(n, ticks, n_actions, seed, t):
    """u8[ticks, n] as psk_random_actions_block; ``t`` includes the device clock (mod 2^64)."""
    out = np.empty((ticks, n), np.uint8)
    _load().orc_random_actions(_p(out), n, ticks, n_actions, ctypes.c_uint64(seed),
                               ctypes.c_uint64(int(t) % (1 << 64)))
    return out


def sample_for(tables, n, seed, offset=0, place_kinds=None):
    """sample_scenarios with the geometry, boundary kind and default placement of CraftTables."""
    from psketch_b200.data import default_placement
    pk = default_placement(tables) if place_kinds is None else place_kinds
    return sample_scenarios(tables.W, tables.H, pk, tables.cookbook.index["boundary"], seed, offset, n)
