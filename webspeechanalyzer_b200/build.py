"""Builds webspeechanalyzer_b200/libfa_b200.so (hand-written CUDA for sm_100a behind the C-ABI of include/fa_b200.h).

In-tree build with nvcc: the .so travels to the GPU box with the repo snapshot.  --fmad=false and
-ffp-contract=off are part of the arithmetic contract (DESIGN.md): every fused multiply-add in the
kernels is an explicit fmaf(), so the float32 / float64 DAGs match the CPU oracle bit for bit.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libfa_b200.so")
SYNTH_LIB = os.path.join(HERE, "libfa_synth.so")   # host-only workload generator (bench / tests), not part of the product
SOURCES = ["fa_spectrum.cu", "fa_peaks.cu", "fa_segment.cu", "fa_features.cu", "fa_utterance.cu", "fa_curves.cu", "fa_mlp.cu", "fa_train.cu", "fa_capi.cu"]
HEADERS = [os.path.join(CSRC, "fa_internal.cuh")] + [os.path.join(ROOT, "include", h)
                                                      for h in ("fa_b200.h", "fa_jsmath.h", "fa_tables.h", "fa_curves.h", "fa_train.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "--fmad=false", "-std=c++17",
         "-Xcompiler", "-fPIC,-ffp-contract=off,-fvisibility=hidden", "-diag-suppress", "39,222",
         "-I", os.path.join(ROOT, "include"), "-I", CSRC]


def build_synth(force: bool = False) -> str:
    src, hdr = os.path.join(CSRC, "fa_synth.cpp"), os.path.join(ROOT, "include", "fa_synth.h")
    if not force and os.path.exists(SYNTH_LIB) and os.path.getmtime(SYNTH_LIB) >= max(os.path.getmtime(src), os.path.getmtime(hdr)):
        return SYNTH_LIB
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-fopenmp", "-fvisibility=hidden", "-I",
                           os.path.join(ROOT, "include"), "-o", SYNTH_LIB + ".tmp", src])
    os.replace(SYNTH_LIB + ".tmp", SYNTH_LIB)
    return SYNTH_LIB


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    build_synth(force)
    if not force and not needs_build():
        return LIB
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for s in SOURCES:
        o = os.path.join(objdir, os.path.splitext(s)[0] + ".o")
        cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, s), "-o", o]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    for s, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError(f"nvcc failed on {s}")
    subprocess.check_call([NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB + ".tmp"] + objs +
                          ["-Xcompiler", "-fPIC", "-cudart", "static"])   # the arch on the link line keeps nvcc from adding an (empty) sm_52 stub
    os.replace(LIB + ".tmp", LIB)
    build_node_addon()
    return LIB


def build_node_addon() -> str:
    """The Node.js addon over the C-ABI (webspeechanalyzer_b200/node).  No Node here: compile-checked against the
    minimal N-API declarations in node/node_api_min.h; the napi_* symbols resolve when node loads the addon."""
    node = os.path.join(HERE, "node")
    out = os.path.join(node, "fa_b200.node")
    subprocess.check_call(["gcc", "-std=gnu11", "-O2", "-fPIC", "-shared", "-fvisibility=hidden", "-Wall", "-I",
                           os.path.join(ROOT, "include"), "-o", out, os.path.join(node, "fa_napi.c"), "-L", HERE,
                           "-lfa_b200", "-Wl,-rpath,$ORIGIN/.."])
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
