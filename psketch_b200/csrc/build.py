"""Builds libpsk_b200.so (sm_100a only) in-tree with nvcc.  Used by __graft_entry__.build()."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
LIB = os.path.join(PKG, "libpsk_b200.so")
SOURCES = ["psk_craft.cu", "psk_craft_generic.cu", "psk_scenario.cu", "psk_light.cu", "psk_host.cu", "psk_hostcpu.cpp"]
HEADERS = ["psk_common.cuh", "psk_hostcpu.h", os.path.join("..", "..", "include", "psk_craft.h"),
           os.path.join("..", "..", "include", "psk_light.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17", "--expt-relaxed-constexpr",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2",
]
LINK_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "shared", "-lpthread"]
OBJ_DIR = os.path.join(HERE, "build")          # git-ignored; objects are rebuilt per source file


def nvcc_path():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return "nvcc"


def _obj(src):
    return os.path.splitext(src)[0] + ".o"


def needs_build():
    if not os.path.exists(LIB):
        return True
    mt = os.path.getmtime(LIB)
    for f in SOURCES + HEADERS + ["build.py"]:
        p = os.path.join(HERE, f)
        if os.path.exists(p) and os.path.getmtime(p) > mt:
            return True
    return False


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    mt = os.path.getmtime(target)
    return any(os.path.exists(d) and os.path.getmtime(d) > mt for d in deps)


def build(force=False, verbose=False, out=None, extra=()):
    """Compiles every source to its own object (in parallel, only the stale ones) and links the
    shared library.  ``out`` / ``extra``: experiment builds (another file name, extra -D flags) for
    A/B runs — those always recompile everything into their own object directory."""
    if not force and not needs_build() and out is None:
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    target = out or LIB
    obj_dir = OBJ_DIR if out is None else OBJ_DIR + "_" + os.path.basename(out).replace(".", "_")
    os.makedirs(obj_dir, exist_ok=True)
    common = [os.path.join(HERE, h) for h in HEADERS] + [os.path.join(HERE, "build.py")]
    jobs = []
    for src in SOURCES:
        sp = os.path.join(HERE, src)
        if not os.path.exists(sp):
            continue
        obj = os.path.join(obj_dir, _obj(src))
        if force or out is not None or _stale(obj, [sp] + common):
            cmd = ([nvcc_path()] + NVCC_FLAGS + list(extra) + (["-Xptxas", "-v"] if verbose else []) +
                   ["-c", "-o", obj, sp])
            jobs.append(cmd)
    with ThreadPoolExecutor(max_workers=max(1, len(jobs))) as pool:
        for rc in pool.map(lambda c: subprocess.call(c, cwd=HERE), jobs):
            if rc:
                raise subprocess.CalledProcessError(rc, "nvcc -c")
    objs = [os.path.join(obj_dir, _obj(s)) for s in SOURCES
            if os.path.exists(os.path.join(HERE, s))]
    subprocess.check_call([nvcc_path()] + LINK_FLAGS + ["-o", target] + objs, cwd=HERE)
    return target


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
