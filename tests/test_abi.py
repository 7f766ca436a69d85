"""CPU-only: the C-ABI shared library loads and exports every symbol include/pmgt_b200.h declares
(no compute calls without a GPU), and fails loudly -- not silently on the CPU -- when asked to compute."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


@pytest.fixture(scope="module")
def lib():
    from pmgt_b200 import _lib, build
    build.build()
    return _lib.lib()


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "pmgt_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(pmgt_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_are_exported(lib):
    from pmgt_b200 import _lib
    names = _declared_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/pmgt_b200.h but not exported"
    assert sorted(_lib.SIGNATURES) == names, "ctypes binding and header disagree"
    assert lib.pmgt_abi_version() == _lib.ABI_VERSION


def test_struct_layouts_match_the_header():
    """sizeof of each ctypes struct == what the C compiler computes for the header's struct."""
    import subprocess
    import tempfile
    from pmgt_b200 import _lib
    prog = r'''
#include <stdio.h>
#include "pmgt_b200.h"
int main(void){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(pmgt_gemm_args), sizeof(pmgt_embed_args), sizeof(pmgt_attn_args),
 sizeof(pmgt_resln_args), sizeof(pmgt_gsr_args), sizeof(pmgt_nfr_args), sizeof(pmgt_block_args), sizeof(pmgt_linear_tile_args),
 sizeof(pmgt_dw_tile_args), sizeof(pmgt_lnbwd_args), sizeof(pmgt_gather_proj_args)); return 0;}
'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(prog)
        exe = os.path.join(d, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        sizes = [int(x) for x in subprocess.check_output([exe]).split()]
    got = [ctypes.sizeof(s) for s in (_lib.GemmArgs, _lib.EmbedArgs, _lib.AttnArgs, _lib.ResLnArgs, _lib.GsrArgs, _lib.NfrArgs,
                                   _lib.BlockArgs, _lib.LinearTileArgs, _lib.DwTileArgs, _lib.LnBwdArgs, _lib.GatherProjArgs)]
    assert got == sizes, (got, sizes)


def test_argument_validation_without_a_gpu(lib):
    """Bad arguments are rejected with PMGT_ERR_INVALID and a message before any CUDA call."""
    from pmgt_b200 import _lib
    g = _lib.GemmArgs()
    g.M, g.N, g.K = 8, 12, 8  # N not a multiple of 8
    g.a = g.b = g.out = 16
    assert lib.pmgt_gemm_bf16(ctypes.byref(g), None) == -1
    assert b"multiple of 8" in lib.pmgt_last_error()
    assert lib.pmgt_sample_contexts(None, None, None, 0, None, 3, 5, 0, None, None, None, None) == -1


def test_attention_rejects_misaligned_buffers_without_a_gpu(lib):
    """qkvc / ctx / dctx / dqkvc must be 16-byte aligned: a misaligned one is named in the error, before any CUDA call.
    The pointers are fake, so this only runs where no device could be reached by a faulty check."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from pmgt_b200 import _lib
    a = _lib.AttnArgs()
    a.rows, a.L, a.H, a.heads, a.beta = 4, 33, 64, 1, 0.5
    a.qkvc, a.mask, a.ctx, a.dctx, a.dqkvc = 16, 16, 24, 16, 16
    a.dropout_p = 0.1
    assert lib.pmgt_attn_core_fwd(ctypes.byref(a), None) == -1
    assert b"pmgt_attn_core_fwd: ctx must be 16-byte aligned" in lib.pmgt_last_error()
    a.dctx = 24
    assert lib.pmgt_attn_core_bwd(ctypes.byref(a), None) == -1
    assert b"pmgt_attn_core_bwd: dctx must be 16-byte aligned" in lib.pmgt_last_error()
    a.dctx, a.dqkvc = 16, 24
    assert lib.pmgt_attn_core_bwd(ctypes.byref(a), None) == -1
    assert b"pmgt_attn_core_bwd: dqkvc must be 16-byte aligned" in lib.pmgt_last_error()


def test_no_cpu_fallback():
    """Without a CUDA device the product path raises instead of computing on the CPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from pmgt_b200 import PMGT, PMGTConfig, PMGTDataset, _lib, synthetic
    g = synthetic.make_item_graph((50, 120), seed=0)
    with pytest.raises(_lib.PMGTError):
        PMGTDataset(g).sample_batch([0, 1])
    net = PMGT(50, config=PMGTConfig(num_hidden_layers=1))
    x = {"node_ids": torch.randint(2, 52, (2, 6)), "attention_mask": torch.ones(2, 6)}
    with pytest.raises(_lib.PMGTError):
        net(x)
    with pytest.raises(_lib.PMGTError):
        g.device_handle(0)  # pmgt_graph_create -> PMGT_ERR_CUDA


def test_product_code_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "pmgt_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", txt, flags=re.M), f
                assert "/root/reference" not in txt, f
