"""Build recipe of the CUDA library (nvcc, sm_100a only, in-tree output)."""
from __future__ import annotations

import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB = os.path.join(_HERE, "libtscm_b200.so")
SOURCES = ["tscm_b200.cu", "tscm_remap.cu", "tscm_posegraph.cu", "tscm_monoinit.cu"]
# per-source flags: the mono cold start mirrors scalar IEEE statements (no FMA contraction)
SOURCE_FLAGS = {"tscm_monoinit.cu": ["-fmad=false"]}
HEADERS = ["tscm_kernels.cuh", "tscm_eval5.cuh", "tscm_solve.cuh", "tscm_solve_cluster.cuh", "tscm_math.cuh", "tscm_p2p.cuh", "tscm_remap.cuh", "tscm_posegraph.cuh", "tscm_covariance.cuh", "tscm_internal.h", "tscm_schur_pairs.cuh", "tscm_pair_lists.h", os.path.join("..", "..", "include", "tscm.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build_cuda(force: bool = False, verbose: bool = False, defines=(), out: str | None = None) -> str:
    """Compile csrc/*.cu into tscm_calib_b200/libtscm_b200.so for sm_100a.
    defines / out: A/B builds of tuning macros into another path (tools/ab_build.py)."""
    lib = out or LIB
    if not force and not defines and not needs_build():
        return lib
    env = dict(os.environ)
    # nvcc must use the distribution g++ (the image's $CXX lacks some specs)
    env.pop("CXX", None)
    env.pop("CC", None)
    objdir = os.path.join(_HERE, "_obj" + ("_" + os.path.basename(lib) if out else ""))
    os.makedirs(objdir, exist_ok=True)

    def run(cmd):
        res = subprocess.run(cmd, capture_output=True, text=True, env=env)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
        if verbose:
            print(res.stderr)

    common = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-D" + d for d in defines]
    objs, procs = [], []
    for src in SOURCES:                      # one translation unit each, compiled side by side
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(obj)
        spath = os.path.join(CSRC, src)
        if (not force and not defines and os.path.exists(obj)
                and all(os.path.getmtime(obj) >= os.path.getmtime(d)
                        for d in [spath] + [os.path.join(CSRC, h) for h in HEADERS])):
            continue
        cmd = common + SOURCE_FLAGS.get(src, []) + ["-c", "-o", obj, spath]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env)))
    for cmd, pr in procs:
        o, e = pr.communicate()
        if pr.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + o + e)
        if verbose:
            print(e)
    run([_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", lib] + objs + ["-ldl"])
    return lib


HOST = os.path.join(_HERE, "host")
HOST_DEMO = os.path.join(HOST, "host_demo")
HOST_SOURCES = ["host_demo.cpp", "multi_calib_b200.cpp", "ts_camera.cpp"]
HOST_HEADERS = ["multi_calib_b200.h", "ts_camera.h", "cv_compat.h"]


def build_host(force: bool = False) -> str:
    """Compile the C++ drop-in adapters (TripleSphereCamera / MultiCalib shaped) and their
    demo driver against libtscm_b200.so."""
    build_cuda()
    deps = [os.path.join(HOST, f) for f in HOST_SOURCES + HOST_HEADERS] + [LIB]
    if not force and os.path.exists(HOST_DEMO) and \
            all(os.path.getmtime(d) <= os.path.getmtime(HOST_DEMO) for d in deps):
        return HOST_DEMO
    cmd = ["g++", "-O2", "-std=c++17", "-Wall", "-o", HOST_DEMO] + \
          [os.path.join(HOST, f) for f in HOST_SOURCES] + \
          ["-L" + _HERE, "-ltscm_b200", "-Wl,-rpath,$ORIGIN/.."]
    env = dict(os.environ)
    env.pop("CXX", None)
    res = subprocess.run(cmd, capture_output=True, text=True, env=env)
    if res.returncode != 0:
        raise RuntimeError("host adapter build failed:\n" + res.stdout + res.stderr)
    return HOST_DEMO
