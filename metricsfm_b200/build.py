"""In-tree build of the native library (nvcc, sm_100a only).  `python -m metricsfm_b200.build [--force]`."""
from __future__ import annotations

import os
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
HOST_DIR = os.path.join(PKG_DIR, "host")
INC = os.path.join(PKG_DIR, "..", "include")
LIB_PATH = os.path.join(CSRC, "libmsfm_match.so")
OBJ_DIR = os.path.join(CSRC, "_obj")
PUBLIC_HEADERS = [os.path.join(INC, h) for h in ("msfm_match.h", "msfm_sched.h", "msfm_multi.h")]
# translation units of libmsfm_match.so: (source, headers it depends on, compiled by nvcc as CUDA?)
UNITS = [
    (os.path.join(CSRC, "msfm_api.cu"),
     [os.path.join(CSRC, h) for h in ("match_kernel.cuh", "aux_kernels.cuh", "geo_kernels.cuh", "sm100_ptx.cuh", "msfm_internal.h")]),
    (os.path.join(CSRC, "msfm_multi.cc"), [os.path.join(CSRC, "msfm_internal.h")]),   # multi-GPU engine (host code + CUDA runtime API)
    (os.path.join(HOST_DIR, "msfm_sched.cc"), []),                                    # pair scheduler (pure host)
]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
    "-ccbin", "/usr/bin/g++",
]


def _newer(target: str, deps) -> bool:
    return os.path.exists(target) and all(os.path.getmtime(d) <= os.path.getmtime(target) for d in deps if os.path.exists(d))


def build_native(force: bool = False, verbose: bool = False) -> str:
    """Compile the translation units of csrc/libmsfm_match.so for sm_100a (each object is rebuilt only when its own
    sources changed) and link them.  Returns the library path."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    extra = os.environ.get("MSFM_NVCC_EXTRA", "").split()  # kernel experiments, e.g. -DMSFM_EXPERIMENTS
    os.makedirs(OBJ_DIR, exist_ok=True)
    me = os.path.abspath(__file__)
    objs, relink = [], force or not os.path.exists(LIB_PATH)
    for src, hdrs in UNITS:
        obj = os.path.join(OBJ_DIR, os.path.splitext(os.path.basename(src))[0] + ".o")
        objs.append(obj)
        if not force and _newer(obj, [src, me] + hdrs + PUBLIC_HEADERS):
            continue
        cmd = [nvcc] + NVCC_FLAGS + extra + ["-x", "cu", "-c", "-o", obj, src]
        proc = subprocess.run(cmd, capture_output=True, text=True)
        if verbose or proc.returncode != 0:
            sys.stderr.write(proc.stdout + proc.stderr)
        if proc.returncode != 0:
            raise RuntimeError(f"nvcc failed compiling {os.path.basename(src)}")
        if src.endswith("msfm_api.cu"):
            with open(os.path.join(CSRC, "ptxas_info.txt"), "w") as f:
                f.write(proc.stderr)
        relink = True
    if relink or not _newer(LIB_PATH, objs):
        proc = subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin", "/usr/bin/g++", "-o", LIB_PATH] + objs + ["-ldl", "-lpthread"],
                              capture_output=True, text=True)
        if proc.returncode != 0:
            sys.stderr.write(proc.stdout + proc.stderr)
            raise RuntimeError("linking libmsfm_match.so failed")
    return LIB_PATH


SHIM_BIN = os.path.join(HOST_DIR, "shim_selftest")
GUIDED_BIN = os.path.join(HOST_DIR, "guided_selftest")  # MatchGraphB200::MatchPairsGuided driver
HOMOGRAPHY_BIN = os.path.join(HOST_DIR, "homography_selftest")  # MatchGraphB200::MatchPairsGuidedHomography driver


def build_host_shim(force: bool = False) -> str:
    """Compile the C++ mirror of the reference's matcher interface + its self-test drivers against the C ABI library.
    Returns the path of the main self-test (the guided-matching drivers are GUIDED_BIN and HOMOGRAPHY_BIN)."""
    for exe in (SHIM_BIN, GUIDED_BIN, HOMOGRAPHY_BIN):
        srcs = [exe + ".cc", os.path.join(HOST_DIR, "feature_matching_b200.cc")]
        deps = srcs + [os.path.join(HOST_DIR, f) for f in ("feature_matching_b200.h", "cv_standin.h")] + [LIB_PATH]
        if not force and os.path.exists(exe) and all(os.path.getmtime(d) <= os.path.getmtime(exe) for d in deps):
            continue
        cmd = ["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-o", exe] + srcs + ["-L" + CSRC, "-lmsfm_match", "-Wl,-rpath,$ORIGIN/../csrc"]
        subprocess.check_call(cmd)
    return SHIM_BIN


STORE_LIB = os.path.join(HOST_DIR, "libmsfm_store.so")
GRAPH_LIB = os.path.join(HOST_DIR, "libmsfm_graph.so")
SCHED_LIB = os.path.join(HOST_DIR, "libmsfm_sched.so")


def build_host_libs(force: bool = False):
    """libmsfm_store.so (the reference's on-disk formats, host only) and libmsfm_graph.so (the fine-matching-graph
    driver = store + GPU matcher)."""
    inc = os.path.join(PKG_DIR, "..", "include")
    store_src = os.path.join(HOST_DIR, "msfm_store.cc")
    graph_src = os.path.join(HOST_DIR, "msfm_graph.cc")
    common = ["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-fPIC", "-shared"]
    if force or not _newer(STORE_LIB, [store_src, os.path.join(inc, "msfm_store.h"), os.path.abspath(__file__)]):
        subprocess.check_call(common + ["-o", STORE_LIB, store_src])
    if force or not _newer(GRAPH_LIB, [graph_src, store_src, LIB_PATH, os.path.join(inc, "msfm_graph.h"), os.path.abspath(__file__)]):
        subprocess.check_call(common + ["-o", GRAPH_LIB, graph_src, store_src, "-L" + CSRC, "-lmsfm_match", "-Wl,-rpath,$ORIGIN/../csrc"])
    sched_src = os.path.join(HOST_DIR, "msfm_sched.cc")
    if force or not _newer(SCHED_LIB, [sched_src, os.path.join(inc, "msfm_sched.h"), os.path.join(inc, "msfm_match.h"), os.path.abspath(__file__)]):
        subprocess.check_call(common + ["-o", SCHED_LIB, sched_src])   # host-only copy of the pair scheduler (CPU tests, launchers)
    return STORE_LIB, GRAPH_LIB, SCHED_LIB


if __name__ == "__main__":
    print(build_native(force="--force" in sys.argv, verbose=True))
    print(build_host_shim(force="--force" in sys.argv))
    print(*build_host_libs(force="--force" in sys.argv))
