#!/usr/bin/env python
"""Build libvrpx.so (hand-written sm_100a CUDA behind the C ABI of include/vrpx.h) in-tree.

    python vrp-gym_b200/csrc/build.py [--force]

nvcc cross-compiles without a GPU; the .so lands in vrp-gym_b200/vrpx/ so that it travels to the GPU box
with the repo snapshot (it is git-ignored, not gpurun-ignored).
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(os.path.dirname(HERE), "vrpx", "libvrpx.so")
SOURCES = ["env.cu", "mt19937_legacy.cu", "encoder.cu", "gemm_tc4.cu", "gemm_tn_tc.cu", "ff_fused.cu", "attn_fused.cu", "rollout.cu", "rollout_steps.cu", "score_table_fused.cu", "decoder_bwd.cu", "encoder_bwd.cu", "attention_bwd.cu"]
HEADERS = ["common.cuh", "tc_common.cuh", "f16split.cuh", "env_rules.cuh", "gemm.cuh", "tile_gemm.cuh", "glimpse_mma.cuh", "rollout.cuh", os.path.join(ROOT, "include", "vrpx.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-Xcompiler", "-ffp-contract=off", "-I" + os.path.join(ROOT, "include"),
]


def _stale():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(HERE, s) for s in SOURCES] + [h if os.path.isabs(h) else os.path.join(HERE, h) for h in HEADERS]
    deps.append(os.path.abspath(__file__))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not _stale():
        return OUT
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for s in SOURCES:
        o = os.path.join(HERE, "build", s.replace(".cu", ".o"))
        objs.append(o)
        cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(HERE, s), "-o", o]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    cmd = [NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", OUT] + objs + ["-Xcompiler", "-fPIC"]
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
