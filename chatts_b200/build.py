"""Build libchatts_b200.so (hand-written sm_100a CUDA + the C-ABI) in-tree with nvcc.

    python -m chatts_b200.build          # incremental
    python -m chatts_b200.build --force

nvcc cross-compiles without a GPU; the .so lands in chatts_b200/lib/ (git-ignored, shipped to the GPU box).
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_build")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libchatts_b200.so")
SOURCES = ["ctx.cu", "gemm_tcgen05.cu", "ts_frontend.cu", "elementwise.cu", "attention.cu", "allreduce.cu", "decode_chain.cu",
           "train_elementwise.cu", "attention_bwd.cu", "sampling.cu", "decoder_step.cu", "attention_bwd_tc5.cu", "lora_wgrad_mma.cu", "gemm_decode_fused.cu", "allreduce_ll.cu", "ts_encoder_fused.cu", "gemm_w4.cu", "gemm_w4_mma.cu", "gemm_w4_persistent.cu"]
HEADERS = ["common.cuh", "tensormap.cuh", "trace.cuh", "ts_rows.cuh", os.path.join("..", "..", "include", "chatts_b200.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
         '-DCTS_BUILD_ARCH="sm_100a"', "-diag-suppress", "177"]


def _newer(src_list, target):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in src_list)


def build(force=False, verbose=True):
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(LIBDIR, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    jobs = []
    for s in srcs:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, s.replace(".cu", ".o"))
        if force or _newer([src] + hdrs, obj):
            jobs.append((src, obj))

    def run(job):
        src, obj = job
        cmd = [NVCC] + FLAGS + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return job, r

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        for (src, obj), r in ex.map(run, jobs):
            if verbose:
                print(f"[chatts_b200.build] nvcc {os.path.basename(src)} -> rc {r.returncode}")
            if r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
                raise RuntimeError(f"nvcc failed on {src}")
    objs = [os.path.join(OBJ, s.replace(".cu", ".o")) for s in srcs]
    if force or jobs or _newer(objs, LIB):
        cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
        if verbose:
            print(f"[chatts_b200.build] linked {LIB}")
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv)
