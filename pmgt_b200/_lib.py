"""ctypes binding of ``libpmgt_b200.so`` (C ABI declared in ``include/pmgt_b200.h``).

There is no CPU fallback: if the shared library has not been built, importing a
compute entry point raises; if it is built but no CUDA device is present, the
library itself fails with ``PMGT_ERR_CUDA``.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpmgt_b200.so")
ABI_VERSION = 13

_lib = None

c_i64p = C.POINTER(C.c_int64)
c_i32p = C.POINTER(C.c_int32)
c_f32p = C.POINTER(C.c_float)
c_u16p = C.POINTER(C.c_uint16)
c_u8p = C.POINTER(C.c_uint8)
c_vp = C.c_void_p


class PMGTError(RuntimeError):
    pass


class GemmArgs(C.Structure):
    _fields_ = [
        ("M", C.c_int64), ("N", C.c_int64), ("K", C.c_int64),
        ("a", c_vp), ("lda", C.c_int64), ("a_mn", C.c_int), ("a_rows", c_vp), ("a_src_rows", C.c_int64),
        ("b", c_vp), ("ldb", C.c_int64), ("b_mn", C.c_int), ("b_rows", c_vp), ("b_src_rows", C.c_int64),
        ("out", c_vp), ("ldo", C.c_int64),
        ("bias", c_vp),
        ("addend", c_vp), ("ld_addend", C.c_int64),
        ("aux", c_vp), ("ld_aux", C.c_int64),
        ("alpha", C.c_float),
        ("epi", C.c_uint32),
        ("split_k", C.c_int),
    ]


class EmbedArgs(C.Structure):
    _fields_ = [
        ("rows", C.c_int64), ("L", C.c_int), ("H", C.c_int),
        ("ev", c_vp), ("et", c_vp),
        ("w_att", c_vp), ("b_att", c_vp), ("pos", c_vp), ("role", c_vp),
        ("ln_g", c_vp), ("ln_b", c_vp), ("ln_eps", C.c_float),
        ("dropout_p", C.c_float), ("dropout_seed", C.c_uint64), ("dropout_site", C.c_uint32),
        ("x_out", c_vp),
        ("dx", c_vp),
        ("dev", c_vp), ("det", c_vp),
        ("d_w_att", c_vp), ("d_b_att", c_vp), ("d_pos", c_vp), ("d_role", c_vp),
        ("d_ln_g", c_vp), ("d_ln_b", c_vp),
        ("d_bias_v", c_vp), ("d_bias_t", c_vp),
        ("dx_b", c_vp),
        ("row_idx", c_vp), ("dev_acc", c_vp), ("det_acc", c_vp), ("skip_row0", C.c_int),
    ]


MAX_MODALITIES = 4  # PMGT_MAX_MODALITIES
_PerMod = c_vp * MAX_MODALITIES


class EmbedMultiArgs(C.Structure):
    _fields_ = [
        ("rows", C.c_int64), ("L", C.c_int), ("H", C.c_int), ("n_mod", C.c_int),
        ("e", _PerMod),
        ("w_att", c_vp), ("b_att", c_vp), ("pos", c_vp), ("role", c_vp),
        ("ln_g", c_vp), ("ln_b", c_vp), ("ln_eps", C.c_float),
        ("dropout_p", C.c_float), ("dropout_seed", C.c_uint64), ("dropout_site", C.c_uint32),
        ("x_out", c_vp),
        ("dx", c_vp),
        ("de", _PerMod),
        ("d_w_att", c_vp), ("d_b_att", c_vp), ("d_pos", c_vp), ("d_role", c_vp),
        ("d_ln_g", c_vp), ("d_ln_b", c_vp),
        ("d_bias", _PerMod),
        ("dx_b", c_vp),
        ("row_idx", c_vp), ("de_acc", _PerMod), ("skip_row0", C.c_int),
    ]


class AttnArgs(C.Structure):
    _fields_ = [
        ("rows", C.c_int64), ("L", C.c_int), ("H", C.c_int), ("heads", C.c_int), ("beta", C.c_float),
        ("qkvc", c_vp), ("mask", c_vp),
        ("dropout_p", C.c_float), ("dropout_seed", C.c_uint64), ("dropout_site", C.c_uint32),
        ("ctx", c_vp),
        ("dctx", c_vp),
        ("dqkvc", c_vp),
        ("d_bias_qkvc", c_vp),
    ]


class ResLnArgs(C.Structure):
    _fields_ = [
        ("T", C.c_int64), ("H", C.c_int),
        ("o", c_vp), ("res", c_vp),
        ("ln_g", c_vp), ("ln_b", c_vp), ("ln_eps", C.c_float),
        ("dropout_p", C.c_float), ("dropout_seed", C.c_uint64), ("dropout_site", C.c_uint32),
        ("y", c_vp), ("y_f32", c_vp),
        ("dy", c_vp), ("dy_f32", c_vp),
        ("dz", c_vp), ("d_o", c_vp),
        ("d_g", c_vp), ("d_b", c_vp), ("d_bias", c_vp),
    ]


class LinearTileArgs(C.Structure):
    _fields_ = [
        ("T", C.c_int64), ("K", C.c_int), ("N", C.c_int),
        ("x", c_vp), ("ldx", C.c_int64),
        ("w", c_vp), ("ldw", C.c_int64), ("w_mn", C.c_int),
        ("epi", C.c_int),
        ("bias", c_vp),
        ("out", c_vp), ("ldo", C.c_int64),
        ("aux_out", c_vp), ("ld_aux_out", C.c_int64),
        ("e_in", c_vp), ("ld_e", C.c_int64),
        ("ln_g", c_vp), ("ln_b", c_vp), ("ln_eps", C.c_float),
        ("dropout_p", C.c_float), ("dropout_seed", C.c_uint64), ("dropout_site", C.c_uint32),
        ("out_f32", c_vp),
        ("dw_x", c_vp), ("ld_dw_x", C.c_int64),
        ("dw", c_vp), ("ld_dw", C.c_int64), ("dbias", c_vp),
    ]


class GatherProjArgs(C.Structure):
    _fields_ = [
        ("T", C.c_int64), ("K", C.c_int64),
        ("table", c_vp), ("ld", C.c_int64), ("table_rows", C.c_int64),
        ("rows", c_vp),
        ("w", c_vp), ("ldw", C.c_int64), ("bias", c_vp),
        ("out", c_vp), ("ldo", C.c_int64),
        ("dy", c_vp), ("ld_dy", C.c_int64),
        ("dw", c_vp), ("ld_dw", C.c_int64),
    ]


class DwTileArgs(C.Structure):
    _fields_ = [
        ("T", C.c_int64), ("N", C.c_int), ("K", C.c_int),
        ("dy", c_vp), ("ld_dy", C.c_int64),
        ("x", c_vp), ("ldx", C.c_int64),
        ("dw", c_vp), ("ld_dw", C.c_int64),
        ("dbias", c_vp),
    ]


class BlockArgs(C.Structure):
    _fields_ = [
        ("T", C.c_int64), ("ffn", C.c_int),
        ("in_", c_vp), ("ld_in", C.c_int64),
        ("res", c_vp), ("ld_res", C.c_int64),
        ("w1", c_vp), ("b1", c_vp), ("w2", c_vp), ("b2", c_vp),
        ("ln_g", c_vp), ("ln_b", c_vp), ("ln_eps", C.c_float),
        ("dropout_p", C.c_float), ("dropout_seed", C.c_uint64), ("dropout_site", C.c_uint32),
        ("out", c_vp), ("ld_out", C.c_int64),
        ("out_f32", c_vp),
        ("h", c_vp), ("gp", c_vp), ("xhat", c_vp), ("ld_save", C.c_int64),
        ("rstd", c_vp),
        ("dy", c_vp), ("ld_dy", C.c_int64),
        ("dy_b", c_vp), ("ld_dy_b", C.c_int64),
        ("dx", c_vp), ("ld_dx", C.c_int64),
        ("dz", c_vp), ("ld_dz", C.c_int64),
        ("dw1", c_vp), ("dw2", c_vp),
        ("db1", c_vp), ("db2", c_vp), ("d_ln_g", c_vp), ("d_ln_b", c_vp),
    ]


class LnBwdArgs(C.Structure):
    _fields_ = [
        ("T", C.c_int64), ("H", C.c_int),
        ("z", c_vp),
        ("dy_a", c_vp), ("dy_b", c_vp), ("dy_f32", c_vp),
        ("ln_g", c_vp), ("ln_eps", C.c_float),
        ("dropout_p", C.c_float), ("dropout_seed", C.c_uint64), ("dropout_site", C.c_uint32),
        ("dz", c_vp), ("d_o", c_vp),
        ("d_g", c_vp), ("d_b", c_vp),
    ]


class GsrArgs(C.Structure):
    _fields_ = [
        ("B", C.c_int64), ("SP", C.c_int64), ("H", C.c_int),
        ("tgt_h", c_vp), ("ld_t", C.c_int64), ("pair_h", c_vp), ("ld_p", C.c_int64),
        ("pair_off", c_vp), ("labels", c_vp),
        ("logits", c_vp), ("loss_out", c_vp),
        ("grad_out", c_vp), ("d_tgt", c_vp), ("d_pair", c_vp),
    ]


class NfrArgs(C.Structure):
    _fields_ = [
        ("Mm", C.c_int64), ("D", C.c_int64),
        ("proj", c_vp), ("ld_proj", C.c_int64),
        ("table", c_vp), ("ld_table", C.c_int64), ("target_ids", c_vp),
        ("weight", C.c_float),
        ("loss_out", c_vp),
        ("grad_out", c_vp), ("dproj", c_vp),
    ]


# name -> (restype, argtypes); also the list of symbols include/pmgt_b200.h declares
SIGNATURES = {
    "pmgt_abi_version": (C.c_int, []),
    "pmgt_set_pdl": (C.c_int, [C.c_int]),
    "pmgt_set_alternate_order": (C.c_int, [C.c_int]),
    "pmgt_last_error": (C.c_char_p, []),
    "pmgt_graph_create": (C.c_int, [C.POINTER(c_vp), C.c_int, C.c_int64, C.c_int64, c_i64p, c_i32p, c_f32p]),
    "pmgt_graph_create_device": (C.c_int, [C.POINTER(c_vp), C.c_int, C.c_int64, C.c_int64, c_vp, c_vp, c_vp, c_vp]),
    "pmgt_graph_destroy": (C.c_int, [c_vp]),
    "pmgt_graph_num_nodes": (C.c_int64, [c_vp]),
    "pmgt_graph_num_edges": (C.c_int64, [c_vp]),
    "pmgt_graph_indptr": (c_vp, [c_vp]),
    "pmgt_graph_indices": (c_vp, [c_vp]),
    "pmgt_graph_cdf": (c_vp, [c_vp]),
    "pmgt_sample_contexts": (C.c_int, [c_vp, c_vp, c_vp, C.c_int64, c_i32p, C.c_int, C.c_int, C.c_uint64,
                                       c_vp, c_vp, c_vp, c_vp]),
    "pmgt_sample_pairs": (C.c_int, [c_vp, c_vp, c_vp, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int,
                                    C.c_uint64, c_vp, c_vp, c_vp, c_vp]),
    "pmgt_gemm_bf16": (C.c_int, [C.POINTER(GemmArgs), c_vp]),
    "pmgt_gather_proj_supported": (C.c_int, [C.c_int64, C.c_int64]),
    "pmgt_gather_proj_fwd": (C.c_int, [C.POINTER(GatherProjArgs), c_vp]),
    "pmgt_gather_proj_dw": (C.c_int, [C.POINTER(GatherProjArgs), c_vp]),
    "pmgt_embed_fuse_fwd": (C.c_int, [C.POINTER(EmbedArgs), c_vp]),
    "pmgt_embed_fuse_bwd": (C.c_int, [C.POINTER(EmbedArgs), c_vp]),
    "pmgt_embed_multi_fwd": (C.c_int, [C.POINTER(EmbedMultiArgs), c_vp]),
    "pmgt_embed_multi_bwd": (C.c_int, [C.POINTER(EmbedMultiArgs), c_vp]),
    "pmgt_attn_core_fwd": (C.c_int, [C.POINTER(AttnArgs), c_vp]),
    "pmgt_attn_core_bwd": (C.c_int, [C.POINTER(AttnArgs), c_vp]),
    "pmgt_res_ln_fwd": (C.c_int, [C.POINTER(ResLnArgs), c_vp]),
    "pmgt_res_ln_bwd": (C.c_int, [C.POINTER(ResLnArgs), c_vp]),
    "pmgt_linear_tile_supported": (C.c_int, [C.c_int64, C.c_int64, C.c_int, C.c_int]),
    "pmgt_linear_tile": (C.c_int, [C.POINTER(LinearTileArgs), c_vp]),
    "pmgt_dw_tile_supported": (C.c_int, [C.c_int64, C.c_int64]),
    "pmgt_dw_tile": (C.c_int, [C.POINTER(DwTileArgs), c_vp]),
    "pmgt_dw_tile_batch": (C.c_int, [C.POINTER(DwTileArgs), C.c_int, c_vp]),
    "pmgt_block_fwd": (C.c_int, [C.POINTER(BlockArgs), c_vp]),
    "pmgt_block_bwd": (C.c_int, [C.POINTER(BlockArgs), c_vp]),
    "pmgt_block_set_trace": (C.c_int, [c_vp]),
    "pmgt_ln_bwd": (C.c_int, [C.POINTER(LnBwdArgs), c_vp]),
    "pmgt_colsum_bf16": (C.c_int, [c_vp, C.c_int64, C.c_int64, C.c_int64, c_vp, c_vp]),
    "pmgt_gsr_fwd": (C.c_int, [C.POINTER(GsrArgs), c_vp]),
    "pmgt_gsr_bwd": (C.c_int, [C.POINTER(GsrArgs), c_vp]),
    "pmgt_nfr_mse_fwd": (C.c_int, [C.POINTER(NfrArgs), c_vp]),
    "pmgt_nfr_mse_bwd": (C.c_int, [C.POINTER(NfrArgs), c_vp]),
    "pmgt_adamw_step": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, C.c_int64, C.c_float, C.c_float, C.c_float,
                                  C.c_float, C.c_float, C.c_int64, C.c_float, c_vp, c_vp]),
    "pmgt_cast_f32_bf16": (C.c_int, [c_vp, c_vp, C.c_int64, c_vp]),
    "pmgt_peer_reduce_f32": (C.c_int, [C.POINTER(C.c_uint64), C.c_int, C.c_int, C.c_int64, c_vp]),
    "pmgt_clip_coef": (C.c_int, [c_vp, C.c_float, C.c_float, c_vp, c_vp]),
    "pmgt_sumsq_f32": (C.c_int, [c_vp, C.c_int64, c_vp, c_vp]),
    "pmgt_gather_rows_bf16": (C.c_int, [c_vp, C.c_int64, c_vp, C.c_int64, C.c_int64, c_vp, C.c_int64, c_vp]),
    "pmgt_scatter_rows_bf16": (C.c_int, [c_vp, C.c_int64, c_vp, C.c_int64, C.c_int64, c_vp, C.c_int64, c_vp]),
}


def lib() -> C.CDLL:
    """Load the shared library (once).  Fails loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PMGTError(
                f"{LIB_PATH} is missing: build it with `python -m pmgt_b200.build` "
                "(nvcc, sm_100a).  pmgt_b200 has no CPU fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        if l.pmgt_abi_version() != ABI_VERSION:
            raise PMGTError(f"ABI mismatch: library {l.pmgt_abi_version()} vs binding {ABI_VERSION}; rebuild")
        _lib = l
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().pmgt_last_error()
        raise PMGTError(f"{what or 'libpmgt_b200'} failed (status {rc}): {msg.decode() if msg else ''}")


def ptr(t) -> int:
    """Device (or host) address of a torch tensor, 0 for None."""
    return 0 if t is None else t.data_ptr()


def cur_stream() -> int:
    """Raw cudaStream_t of torch's current stream on the current device (the fast private accessor when present:
    ``torch.cuda.current_stream()`` costs ~15 us per call, which adds up over ~100 launches a step)."""
    import torch

    try:
        return torch._C._cuda_getCurrentRawStream(torch.cuda.current_device())
    except AttributeError:
        return torch.cuda.current_stream().cuda_stream


# -- graph -------------------------------------------------------------------------
def graph_create(device_index: int, num_nodes: int, indptr: np.ndarray, indices: np.ndarray, cdf: np.ndarray):
    h = c_vp()
    indptr = np.ascontiguousarray(indptr, dtype=np.int64)
    indices = np.ascontiguousarray(indices, dtype=np.int32)
    cdf = np.ascontiguousarray(cdf, dtype=np.float32)
    rc = lib().pmgt_graph_create(
        C.byref(h), device_index, num_nodes, len(indices),
        indptr.ctypes.data_as(c_i64p), indices.ctypes.data_as(c_i32p), cdf.ctypes.data_as(c_f32p))
    check(rc, "pmgt_graph_create")
    return h


def graph_create_device(device_index: int, num_nodes: int, indptr_dev, indices_dev, weights_dev):
    """``pmgt_graph_create_device``: torch CUDA tensors (int64 / int32 / float64) -> opaque handle."""
    h = c_vp()
    rc = lib().pmgt_graph_create_device(C.byref(h), device_index, num_nodes, indices_dev.numel(), ptr(indptr_dev),
                                        ptr(indices_dev), ptr(weights_dev), cur_stream())
    check(rc, "pmgt_graph_create_device")
    return h


def graph_destroy(h) -> None:
    if _lib is not None and h:
        _lib.pmgt_graph_destroy(h)
