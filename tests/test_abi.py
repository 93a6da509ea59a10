"""CPU-only checks of the drop-in boundary: the C-ABI library builds for sm_100a, loads, and
exports every symbol that include/*.h declares; the host tables match the reference's ids."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib_path():
    import __graft_entry__ as g
    return g.build()


def _declared(header):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(psk_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(lib_path):
    lib = ctypes.CDLL(lib_path)
    headers = [h for h in os.listdir(os.path.join(ROOT, "include")) if h.endswith(".h")]
    assert "psk_craft.h" in headers
    n = 0
    for h in headers:
        for sym in _declared(h):
            assert hasattr(lib, sym), "%s declared in %s but not exported" % (sym, h)
            n += 1
    assert n >= 10
    lib.psk_version.restype = ctypes.c_char_p
    assert b"sm_100a" in lib.psk_version()


def test_library_has_sm100a_sass_with_tma(lib_path):
    out = subprocess.run(["cuobjdump", "-sass", lib_path], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert "UBLKCP" in out          # TMA bulk store of feature tiles
    assert ".256" in out            # 256-bit agent-record loads/stores


def test_struct_sizes_match_header():
    from psketch_b200 import _lib
    assert ctypes.sizeof(_lib.CraftTablesC) == 12 * 4 + 32 + 128 + 32 + 2048 + 64
    assert ctypes.sizeof(_lib.CraftStateC) == 32
    assert ctypes.sizeof(_lib.CraftEpisodesC) == 24


def test_ops_fail_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from psketch_b200 import _lib
    from psketch_b200.vec import VecCraft
    with pytest.raises(_lib.PskError):
        VecCraft(None, 4)


def test_tables_match_reference_ids(medium_tables):
    """Kind ids / classes (SURVEY §8, Appendix A.1-A.2) and task ids (Appendix B)."""
    cb = medium_tables.cookbook
    names = ["boundary", "workshop0", "workshop1", "workshop2", "water", "stone", "iron", "grass",
             "wood", "gold", "gem", "plank", "stick", "axe", "rope", "bed", "shears", "cloth",
             "bridge", "ladder"]
    assert [cb.index[n] for n in names] == list(range(1, 21))
    assert cb.n_kinds == 21 and medium_tables.n_features == 404
    assert cb.index["none"] is None
    assert medium_tables.kind_class[:21].tolist() == [0, 1, 2, 2, 2, 3, 4] + [5] * 14
    rec = medium_tables.recipes[:9]
    assert rec[:, 0].tolist() == [12, 14, 15, 13, 16, 17, 18, 19, 20]
    assert rec[:, 1].tolist() == [2, 2, 2, 3, 3, 3, 4, 4, 4]
    tm = medium_tables.task_manager
    assert tm["get[wood]"].task_id == 13 and tm["make[shears]"].task_id == 26
    assert tm["make[bed]"].encoding == [19, 25] and tm["get[iron]"].encoding == [17, 12]
    assert len(tm.vocab) - 1 == 27
    # make[bed] flattens to 14 pre-order nodes
    assert medium_tables.task_len[24] == 14


def test_rollout_kernel_register_budget(lib_path):
    """The multi-tick kernel is built for 896 threads per SM: 7 CTAs of 64 env threads + 2 feature
    warps, or 9 CTAs of 32 + 2 (the shape used from 65,536 envs up: 2,048 CTAs on 1,332 slots).
    One CTA less per SM costs 20 % (17.5 -> 21 us per tick when a change pushed it to 80 registers)."""
    out = subprocess.run(["cuobjdump", "-res-usage", lib_path], capture_output=True, text=True).stdout
    lines = out.splitlines()
    for shape, threads, ctas in (("Li64ELi2E", 128, 7), ("Li32ELi2E", 96, 9)):
        regs = []
        for i, line in enumerate(lines):
            if "craft_rollout_kernelILi8ELi8ELi3E" + shape in line and i + 1 < len(lines):
                m = re.search(r"REG:(\d+)", lines[i + 1])
                if m:
                    regs.append(int(m.group(1)))
        assert regs, "rollout kernel %s not found in the library" % shape
        # registers are allocated per warp in units of 8 per thread
        assert ctas * threads * ((max(regs) + 7) // 8 * 8) <= 65536, (shape, regs)


def _build_c_host(tmp_path):
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "host_rollout")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-O2", "-I", os.path.join(root, "include"),
                           "-I", os.path.join(cuda, "include"), os.path.join(root, "examples", "host_rollout.c"),
                           "-L", os.path.join(root, "psketch_b200"), "-lpsk_b200",
                           "-L", os.path.join(cuda, "lib64"), "-lcudart",
                           "-Wl,-rpath," + os.path.join(root, "psketch_b200"), "-o", exe])
    return exe


def test_headers_are_plain_c_and_a_c_host_links(tmp_path):
    """The boundary is a C ABI: both headers compile as strict C99 (-Wall -Werror), and a host written
    in plain C (examples/host_rollout.c: no Python, no torch) builds and links against the library."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "inc.c"
    src.write_text('#include "psk_craft.h"\n#include "psk_light.h"\nint main(void) { return PSK_OK; }\n')
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-fsyntax-only",
                           "-I", os.path.join(root, "include"), str(src)])
    assert os.path.exists(_build_c_host(tmp_path))


@pytest.mark.gpu
def test_c_host_runs_rollouts(tmp_path):
    """The plain-C host on the GPU: teacher-driven rollouts of get[wood] on its hand-built scenario.
    The teacher's plan is RIGHT, RIGHT, USE, STOP (4 ticks per episode), so 24 ticks of 4,096 envs
    are 24,576 episodes, all successful."""
    import subprocess
    out = subprocess.check_output([_build_c_host(tmp_path), "4096", "24"], text=True)
    assert "sm_100a" in out
    assert "episodes=24576 successes=24576 env_steps=98304 err=0" in out, out
    assert out.strip().endswith("teacher: 3 3 4 5 3 3 4 5"), out


def test_wire_split_rule_converges_and_holds():
    """The split-frame rule of PSK_FEATURES_F32_WIRE_U8 (psk_debug_wire_split_next; no CUDA call): on a
    simulated box where a byte chunk costs p on the wire (an f32 chunk 4 p) and w on the host threads, the
    number of chunks sent as f32 settles within a few calls just below 0.8 C (w - p) / (w + 3 p), stays
    there under 5 % timing noise (moves of at most one chunk), returns to 0 when the host is the faster
    side, and never leaves [0, C - 1]."""
    import ctypes
    from psketch_b200 import _lib
    lib = _lib.load()
    rng = np.random.RandomState(3)

    def simulate(C, p, w, calls=40, d=0, noise=0.0):
        ps, ws = ctypes.c_double(0.0), ctypes.c_double(0.0)
        hist = []
        for _ in range(calls):
            jp, jw = 1 + noise * rng.uniform(-1, 1), 1 + noise * rng.uniform(-1, 1)
            t_pcie = (C + 3 * d) * p * jp + 30.0                  # + start-up latency
            t_widen = (C - d) * max(w, p) * jw + 30.0             # threads cannot finish before the bytes land
            d = lib.psk_debug_wire_split_next(C, d, t_pcie, t_widen, ctypes.byref(ps), ctypes.byref(ws))
            assert 0 <= d <= C - 1
            hist.append(d)
        return hist

    for C, p, w in [(16, 29.6, 75.0), (16, 29.6, 34.0), (16, 29.6, 20.0), (5, 10.0, 80.0), (64, 8.0, 12.0),
                    (16, 60.0, 61.0), (2, 10.0, 100.0)]:
        ideal = min(max(0.0, 0.8 * C * (w - p) / (w + 3 * p)), C - 1)       # the rule aims below the balance
        hist = simulate(C, p, w)
        assert len(set(hist[6:])) == 1, (C, p, w, hist)                     # settled, no oscillation
        assert ideal - 1.6 <= hist[-1] <= ideal + 0.6, (C, p, w, hist, ideal)
        noisy = simulate(C, p, w, calls=200, noise=0.05)
        assert max(noisy[10:]) - min(noisy[10:]) <= 1 + (C >= 64), (C, p, w, noisy)
        assert ideal - 1.6 <= np.mean(noisy[10:]) <= ideal + 1.0, (C, p, w, noisy, ideal)
    # the host became the faster side (e.g. the caller gave the library more threads): back to bytes only
    assert simulate(16, 29.6, 20.0, d=7)[-1] == 0
    # degenerate calls leave the split alone
    ps, ws = ctypes.c_double(0.0), ctypes.c_double(0.0)
    assert lib.psk_debug_wire_split_next(1, 0, 50.0, 50.0, ctypes.byref(ps), ctypes.byref(ws)) == 0
    assert lib.psk_debug_wire_split_next(0, 0, 0.0, 0.0, ctypes.byref(ps), ctypes.byref(ws)) == 0
    assert lib.psk_debug_wire_split_next(4, 9, 50.0, 50.0, ctypes.byref(ps), ctypes.byref(ws)) == 3
    assert lib.psk_debug_wire_split_next(4, 2, 0.0, 50.0, ctypes.byref(ps), ctypes.byref(ws)) == 2


def test_host_widening_of_byte_frames():
    """psk_host_widen_u8_f32 (the host half of PSK_FEATURES_F32_WIRE_U8): dst[i] == src[i] for every
    length and alignment, single-threaded and through the thread pool.  No CUDA call: runs here."""
    from psketch_b200 import _lib
    lib = _lib.load()
    rng = np.random.RandomState(5)
    src = rng.randint(0, 256, size=(1 << 22) + 77).astype(np.uint8)
    dst = np.empty(len(src) + 16, np.float32)
    for n, so, do, threads in ((0, 0, 0, 1), (1, 3, 1, 1), (31, 1, 3, 1), (404, 0, 0, 1), (4099, 5, 7, 2),
                               ((1 << 20) + 13, 1, 1, 4), (len(src) - 9, 9, 5, 3), (len(src), 0, 0, 8)):
        dst[:] = -1.0
        rc = lib.psk_host_widen_u8_f32(ctypes.c_void_p(src.ctypes.data + so), ctypes.c_void_p(dst.ctypes.data + 4 * do),
                                       n, threads)
        assert rc == 0
        assert np.array_equal(dst[do:do + n], src[so:so + n].astype(np.float32)), (n, so, do, threads)
        assert (dst[:do] == -1).all() and (dst[do + n:] == -1).all(), (n, so, do, threads)
    assert lib.psk_host_widen_u8_f32(None, None, 5, 1) != 0
    for _ in range(20):         # pools are created and joined without leaking or hanging
        assert lib.psk_host_widen_u8_f32(ctypes.c_void_p(src.ctypes.data), ctypes.c_void_p(dst.ctypes.data),
                                         1 << 21, 4) == 0
    assert np.array_equal(dst[:1 << 21], src[:1 << 21].astype(np.float32))
