"""Builds ``pmgt_b200/libpmgt_b200.so`` in-tree with nvcc for sm_100a.

    python -m pmgt_b200.build [--force] [--verbose]

The library has no torch dependency (plain C ABI, include/pmgt_b200.h); nvcc
cross-compiles it without a GPU present.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ_DIR = os.path.join(HERE, "csrc", "_obj")
OUT = os.path.join(HERE, "libpmgt_b200.so")
SOURCES = ["api.cu", "sampler.cu", "graph_build.cu", "gemm_umma.cu", "gather_proj.cu", "linear_tile.cu", "ffn_block.cu", "rowwise.cu", "res_ln_wide.cu", "embed128.cu", "embed_multi.cu", "ln_bwd_stream.cu", "attention.cu", "attention_small.cu", "attention_mma.cu", "attention_mid.cu", "attention_reg.cu", "loss.cu", "peer_reduce.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "--use_fast_math", "-Xcompiler", "-fvisibility=default",
] + os.environ.get("PMGT_NVCC_FLAGS", "").split()  # e.g. -DPMGT_SPIN_WAIT for an A/B build on the GPU box


def _deps_mtime() -> float:
    paths = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh"))]
    paths.append(os.path.join(HERE, "..", "include", "pmgt_b200.h"))
    return max(os.path.getmtime(p) for p in paths)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and os.path.exists(OUT) and os.path.getmtime(OUT) >= _deps_mtime():
        return OUT
    os.makedirs(OBJ_DIR, exist_ok=True)
    extra = ["-Xptxas", "-v"] if verbose else []

    def compile_one(src):
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", OUT, *objs]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
