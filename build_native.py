"""Builds libdmc_b200.so (hand-written sm_100a kernels + C ABI) in-tree with nvcc.

    python build_native.py [--force]

(kept outside the package so that building never imports the package, which loads the library)

Flags that matter for bit parity: -fmad=false (no FMA contraction) and no --use_fast_math (IEEE division and
square root).  -lineinfo keeps the ncu source page mapped to these files.
"""
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
HERE = os.path.join(ROOT, "depthmapcompression_b200")
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libdmc_b200.so")
SOURCES = ["dmc_kernels_8u.cu", "dmc_bwrf8u_h2.cu", "dmc_bwrf8u_c3_h2.cu", "dmc_joint_bwrf.cu", "dmc_front8u.cu", "dmc_kernels_32f.cu", "dmc_prepare.cu", "dmc_brf.cu", "dmc_bwrf32f_tiled.cu", "dmc_jpeg.cu", "dmc_jpeg_color.cu", "dmc_jpeg_enc.cu", "dmc_jpeg_color_enc.cu", "dmc_metrics.cu", "dmc_hostlink.cu", "dmc_render.cu", "dmc_capi.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=false", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "--shared", "-Xptxas", "-v", "--threads", "0"]


def _nvcc():
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


OBJDIR = os.path.join(HERE, "_obj")           # per-source objects (git- and gpurun-ignored): only changed sources recompile


def _headers():
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC) if not f.endswith(".cu")] + [os.path.join(ROOT, "include", "dmc_c.h"), os.path.abspath(__file__)]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def needs_build():
    return _stale(LIB, [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(ROOT, "include", "dmc_c.h")])


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    ccbin = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else None
    base = [_nvcc()] + [f for f in NVCC_FLAGS if f != "--shared"] + (["-ccbin", ccbin] if ccbin else [])
    os.makedirs(OBJDIR, exist_ok=True)
    hdrs = _headers()
    logs = {}

    def compile_one(src):
        obj = os.path.join(OBJDIR, src[:-3] + ".o")
        if not force and not _stale(obj, [os.path.join(CSRC, src)] + hdrs):
            return obj
        cmd = base + ["-c", "-o", obj, os.path.join(CSRC, src)]
        res = subprocess.run(cmd, capture_output=True, text=True)
        logs[src] = " ".join(cmd) + "\n" + res.stdout + res.stderr
        if res.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (src, (res.stdout + res.stderr)[-4000:]))
        return obj

    with ThreadPoolExecutor(min(len(SOURCES), os.cpu_count() or 4)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [_nvcc(), "--shared", "-gencode", "arch=compute_100a,code=sm_100a"] + (["-ccbin", ccbin] if ccbin else []) + ["-o", LIB] + objs
    res = subprocess.run(cmd, capture_output=True, text=True)
    log = "".join(logs[k] for k in sorted(logs)) + " ".join(cmd) + "\n" + res.stdout + res.stderr
    with open(os.path.join(HERE, "build.log"), "a" if not force else "w") as f:
        f.write(log)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + log[-4000:])
    if verbose:
        print(log)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
    print("built", LIB)
