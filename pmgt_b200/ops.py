"""Thin torch-tensor wrappers over the C ABI (``include/pmgt_b200.h``).

Every function enqueues work on torch's current CUDA stream and returns
immediately; torch is used only for device memory and streams.  bf16 tensors
are passed as raw ``uint16`` storage.
"""
import ctypes as C

import torch

from . import _lib
from ._lib import (AttnArgs, DwTileArgs, EmbedArgs, EmbedMultiArgs, BlockArgs, GemmArgs, GsrArgs, LinearTileArgs, LnBwdArgs, NfrArgs, ResLnArgs, check,
                   cur_stream, ptr)

EPI_BIAS, EPI_GELU, EPI_GELU_BWD, EPI_ADDEND, EPI_OUT_F32, EPI_ATOMIC = 1, 2, 4, 8, 16, 32
BF16 = torch.bfloat16

# -- instrumentation ---------------------------------------------------------------------------
# LAUNCHES counts kernels launched by this library (bench.py's `gpu_launches`).  When PROFILE is
# a list, every C-ABI call is bracketed by CUDA events on the launching stream and recorded as
# (tag, start_event, end_event, algorithmic_bytes, flops); bench.py aggregates them after a sync.
LAUNCHES = [0]
PROFILE = None
# When TAPE is a list, every call is also appended to it as (tag, fn, args, launches, bytes, flops).  A recorded tape
# can be re-issued with `replay` as long as every buffer it names is still alive at the same address: this is how the
# encoder's fixed-shape launch sequence is issued after the first step (modeling_pmgt._EncoderPlan) -- a few
# microseconds of host time per launch instead of re-deriving ~170 argument blocks in Python every step.
TAPE = None


def _run(tag, fn, args, launches=1, nbytes=0, flops=0):
    LAUNCHES[0] += launches
    if TAPE is not None:
        TAPE.append((tag, fn, args, launches, nbytes, flops))
    if PROFILE is None:
        check(fn(*args), tag)
        return
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    check(fn(*args), tag)
    e1.record()
    PROFILE.append((tag, e0, e1, nbytes, flops))


def replay(tape):
    """Re-issue a recorded launch list on the stream it was recorded on."""
    if PROFILE is not None or TAPE is not None:
        for tag, fn, args, launches, nbytes, flops in tape:
            _run(tag, fn, args, launches, nbytes, flops)
        return
    n = 0
    for tag, fn, args, launches, _, _ in tape:
        rc = fn(*args)
        if rc:
            check(rc, tag)
        n += launches
    LAUNCHES[0] += n


def set_pdl(enabled: bool) -> bool:
    """Programmatic dependent launch of the encoder's kernel chain on/off; returns the previous setting."""
    return bool(_lib.lib().pmgt_set_pdl(int(bool(enabled))))


def set_alternate_order(enabled: bool) -> bool:
    """Alternating tile traversal order of consecutive encoder kernels (L2 reuse) on/off; returns the previous setting."""
    return bool(_lib.lib().pmgt_set_alternate_order(int(bool(enabled))))


def zero_(t):
    """``t.zero_()`` that a tape can replay (a torch memset on the current stream; not counted as one of our launches)."""
    def fn():
        t.zero_()
        return 0
    _run("memset", fn, (), 0, t.numel() * t.element_size(), 0)


def host_hook(fn, *args):
    """A host-side callback at this point of the launch sequence (replayed with the tape): e.g. the trainer starts the
    gradient allreduce of the encoder layers here, while the embedding backward is still to be enqueued."""
    def call():
        fn(*args)
        return 0
    _run("host_hook", call, (), 0, 0, 0)


def tape_seed_blocks(tape):
    """The argument blocks of a tape that carry a dropout seed (patched before every replay)."""
    out = []
    for _, _, args, _, _, _ in tape:
        if args and hasattr(args[0], "_obj") and hasattr(args[0]._obj, "dropout_seed"):
            out.append(args[0]._obj)
    return out


def profile_summary(records):
    """{tag: dict(ms, calls, bytes, flops)} from PROFILE records (call after torch.cuda.synchronize())."""
    out = {}
    for tag, e0, e1, nbytes, flops in records:
        d = out.setdefault(tag, dict(ms=0.0, calls=0, bytes=0, flops=0))
        d["ms"] += e0.elapsed_time(e1)
        d["calls"] += 1
        d["bytes"] += nbytes
        d["flops"] += flops
    return out


def _require_cuda(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise _lib.PMGTError(f"{name} must be a CUDA tensor: pmgt_b200 has no CPU fallback")


def _num_sms(dev) -> int:
    return torch.cuda.get_device_properties(dev).multi_processor_count


def gemm(a, b, out, *, M, N, K, lda, ldb, ldo, a_mn=False, b_mn=False, a_rows=None, a_src_rows=0, b_rows=None,
         b_src_rows=0, bias=None, addend=None, ld_addend=0, aux=None, ld_aux=0, alpha=1.0, epi=0, split_k=1,
         tag="gemm"):
    """``pmgt_gemm_bf16``: D[M,N] (+)= op(A) op(B); see the header for operand layouts."""
    _require_cuda(a, "a")
    g = GemmArgs(M, N, K, ptr(a), lda, int(a_mn), ptr(a_rows), a_src_rows, ptr(b), ldb, int(b_mn), ptr(b_rows),
                 b_src_rows, ptr(out), ldo, ptr(bias), ptr(addend), ld_addend, ptr(aux), ld_aux, alpha, epi, split_k)
    # algorithmic (compulsory) bytes: each operand element once, the output once, epilogue side inputs once
    osz = 4 if epi & (EPI_OUT_F32 | EPI_ATOMIC) else 2
    nbytes = 2 * M * K + 2 * N * K + osz * M * N
    if epi & EPI_ADDEND:
        nbytes += 2 * M * N
    if epi & (EPI_GELU | EPI_GELU_BWD):
        nbytes += 2 * M * N
    _run(tag, _lib.lib().pmgt_gemm_bf16, (C.byref(g), cur_stream()), 1, nbytes, 2 * M * N * K)


# gathered feature projections through the persistent wide-stage kernels (csrc/gather_proj.cu); False: pmgt_gemm_bf16
GATHER_PROJ = True
_GP_SUPPORTED = {}


def gather_proj_supported(N: int, K: int) -> bool:
    key = (int(N), int(K))
    if key not in _GP_SUPPORTED:
        _GP_SUPPORTED[key] = bool(_lib.lib().pmgt_gather_proj_supported(key[0], key[1]))
    return _GP_SUPPORTED[key]


def linear_fwd(x, w, bias, out, *, rows=None, src_rows=0, gelu_aux=None, tag=None):
    """out[T,N] = x[T,K] @ w[N,K]^T + bias   (x optionally gathered through ``rows``)."""
    N, K = w.shape
    T = out.shape[0]
    epi = EPI_BIAS if bias is not None else 0
    if gelu_aux is not None:
        epi |= EPI_GELU
    if rows is not None and gelu_aux is None and GATHER_PROJ and gather_proj_supported(N, K) and out.stride(0) % 16 == 0:
        g = _lib.GatherProjArgs(T, K, ptr(x), x.stride(0), src_rows, ptr(rows), ptr(w), w.stride(0), ptr(bias), ptr(out),
                                out.stride(0), None, 0, None, 0)
        _run(tag or "gemm_fwd_gather", _lib.lib().pmgt_gather_proj_fwd, (C.byref(g), cur_stream()), 1,
             2 * T * K + 2 * N * K + 2 * T * N, 2 * T * N * K)
        return
    gemm(x, w, out, M=T, N=N, K=K, lda=x.stride(0), ldb=w.stride(0), ldo=out.stride(0), a_rows=rows,
         a_src_rows=src_rows, bias=bias, aux=gelu_aux, ld_aux=(gelu_aux.stride(0) if gelu_aux is not None else 0), epi=epi,
         tag=tag or ("gemm_fwd_gather" if rows is not None else "gemm_fwd"))


def linear_dx(dy, w, out, *, addend=None, gelu_bwd_aux=None, tag="gemm_dx"):
    """out[T,K] = dy[T,N] @ w[N,K] (+ addend) (* gelu'(aux))."""
    N, K = w.shape
    T = dy.shape[0]
    epi = 0
    if addend is not None:
        epi |= EPI_ADDEND
    if gelu_bwd_aux is not None:
        epi |= EPI_GELU_BWD
    gemm(dy, w, out, M=T, N=K, K=N, lda=dy.stride(0), ldb=w.stride(0), ldo=out.stride(0), b_mn=True,
         addend=addend, ld_addend=(addend.stride(0) if addend is not None else 0),
         aux=gelu_bwd_aux, ld_aux=(gelu_bwd_aux.stride(0) if gelu_bwd_aux is not None else 0), epi=epi, tag=tag)


def linear_dw(dy, x, dw_f32, *, rows=None, src_rows=0, x_cols=None, tag=None):
    """dw[N,K] += dy[T,N]^T @ x[T,K]  (fp32 atomic accumulation, split over T).

    ``x`` may be a table whose rows are fetched through ``rows`` (T int64 ids)."""
    T, N = dy.shape
    K = x_cols if x_cols is not None else x.shape[1]
    if rows is not None and GATHER_PROJ and gather_proj_supported(N, K) and dy.stride(1) == 1:
        g = _lib.GatherProjArgs(T, K, ptr(x), x.stride(0), src_rows, ptr(rows), None, 0, None, None, 0, ptr(dy), dy.stride(0),
                                ptr(dw_f32), dw_f32.stride(0))
        _run(tag or "gemm_dw_gather", _lib.lib().pmgt_gather_proj_dw, (C.byref(g), cur_stream()), 1,
             2 * T * K + 2 * T * N + 4 * N * K, 2 * T * N * K)
        return
    tiles = ((N + 127) // 128) * ((K + 127) // 128)
    num_kb = (T + 63) // 64
    # two CTAs are resident per SM: the split count keeps tiles * split WITHIN one wave of 2 * SMs CTAs (rounding up put 300
    # CTAs on 296 slots: a second, nearly empty wave doubled the kernel's duration -- ncu grid 300, round 2)
    split = max(1, min(num_kb, (2 * _num_sms(dy.device)) // tiles))
    # short reductions (the NFR heads: a few thousand rows): every split flushes a whole fp32 tile through the L2 atomic
    # units, which then costs more than the products -- keep at least 8 k-blocks (512 rows) per CTA
    split = max(1, min(split, num_kb // 8))
    gemm(dy, x, dw_f32, M=N, N=K, K=T, lda=dy.stride(0), ldb=x.stride(0), ldo=dw_f32.stride(0), a_mn=True, b_mn=True,
         b_rows=rows, b_src_rows=src_rows, epi=EPI_ATOMIC, split_k=split,
         tag=tag or ("gemm_dw_gather" if rows is not None else "gemm_dw"))


# -- persistent token-tile kernels (fast path for H = I = 128) ------------------------------------
LT_BIAS, LT_GELU, LT_RES_LN, LT_PLAIN, LT_GELU_BWD = 0, 1, 2, 3, 4


def linear_tile_supported(K, N, w_mn, epi) -> bool:
    return bool(_lib.lib().pmgt_linear_tile_supported(K, N, int(w_mn), epi))


def dw_tile_supported(N, K) -> bool:
    return bool(_lib.lib().pmgt_dw_tile_supported(N, K))


def linear_tile(x, w, out, epi, *, w_mn=False, bias=None, aux_out=None, e_in=None, ln_g=None, ln_b=None, ln_eps=0.0,
                p=0.0, seed=0, site=0, out_f32=None, dw_x=None, dw=None, dbias=None, tag=None):
    """``pmgt_linear_tile``: out[T,N] = epi(x[T,K] @ w^T) (w_mn=False, w [N,K]) or epi(x[T,K] @ w) (w_mn=True, w [K,N])."""
    _require_cuda(x, "x")
    T, K = x.shape
    N = out.shape[1]
    a = LinearTileArgs()
    a.T, a.K, a.N = T, K, N
    a.x, a.ldx = ptr(x), x.stride(0)
    a.w, a.ldw, a.w_mn = ptr(w), w.stride(0), int(w_mn)
    a.epi = epi
    a.bias = ptr(bias)
    a.out, a.ldo = ptr(out), out.stride(0)
    a.aux_out, a.ld_aux_out = ptr(aux_out), (aux_out.stride(0) if aux_out is not None else 0)
    a.e_in, a.ld_e = ptr(e_in), (e_in.stride(0) if e_in is not None else 0)
    a.ln_g, a.ln_b, a.ln_eps = ptr(ln_g), ptr(ln_b), ln_eps
    a.dropout_p, a.dropout_seed, a.dropout_site = p, seed, site
    a.out_f32 = ptr(out_f32)
    a.dw_x, a.ld_dw_x = ptr(dw_x), (dw_x.stride(0) if dw_x is not None else 0)
    a.dw, a.ld_dw, a.dbias = ptr(dw), (dw.stride(0) if dw is not None else 0), ptr(dbias)
    nbytes = 2 * T * K + 2 * K * N + 2 * T * N
    flops = 2 * T * N * K
    if dw is not None:  # fused weight gradient: one more activation stream, one more GEMM
        nbytes += 2 * T * dw_x.shape[1] + 4 * K * dw_x.shape[1]
        flops += 2 * T * K * dw_x.shape[1]
    if aux_out is not None:
        nbytes += 2 * T * N
    if e_in is not None:
        nbytes += 2 * T * N
    if out_f32 is not None:
        nbytes += 4 * T * N
    _run(tag or "linear_tile", _lib.lib().pmgt_linear_tile, (C.byref(a), cur_stream()), 1, nbytes, flops)


class BlockSaved:
    """What ``block_fwd`` leaves for ``block_bwd``: xhat (normalised pre-affine LayerNorm value), rstd and
    -- FFN block -- h = gelu(h_pre) and gp = gelu'(h_pre)."""
    __slots__ = ("xhat", "rstd", "h", "gp")

    def __init__(self, T, ffn, p, device, new=None):
        mk = new if new is not None else (lambda *shape, dtype=torch.bfloat16: torch.empty(shape, dtype=dtype, device=device))
        self.xhat = mk(T, 128)
        self.rstd = mk(T, dtype=torch.float32)
        self.h = mk(T, 128) if ffn else None
        self.gp = mk(T, 128) if ffn else None

    def tensors(self):
        return tuple(t for t in (self.xhat, self.rstd, self.h, self.gp) if t is not None)


def block_args(x, w2, b2, ln_g, ln_b, eps, p, seed, site, w1=None, b1=None, res=None):
    """Argument block shared by ``block_fwd`` / ``block_bwd``.  ``w1`` given: the feed-forward block
    ``LayerNorm(dropout(gelu(x w1^T + b1) w2^T + b2) + x)``; otherwise the dense block
    ``LayerNorm(dropout(x w2^T + b2) + res)`` (H = I = 128)."""
    _require_cuda(x, "x")
    f = BlockArgs()
    f.T = x.shape[0]
    f.ffn = 1 if w1 is not None else 0
    f.in_, f.ld_in = ptr(x), x.stride(0)
    f.res, f.ld_res = ptr(res), (res.stride(0) if res is not None else 0)
    f.w1, f.b1, f.w2, f.b2 = ptr(w1), ptr(b1), ptr(w2), ptr(b2)
    f.ln_g, f.ln_b, f.ln_eps = ptr(ln_g), ptr(ln_b), eps
    f.dropout_p, f.dropout_seed, f.dropout_site = p, seed, site
    return f


def block_supported(H, I) -> bool:
    return H == 128 and I == 128


def _block_saved(f: BlockArgs, sv):
    f.xhat, f.rstd = ptr(sv.xhat), ptr(sv.rstd)
    f.h, f.gp, f.ld_save = ptr(sv.h), ptr(sv.gp), sv.xhat.stride(0)


def block_fwd(f: BlockArgs, out, out_f32=None, saved: BlockSaved = None):
    """One persistent tcgen05 kernel for the whole block; ``saved`` receives the activations ``block_bwd`` needs."""
    f.out, f.ld_out, f.out_f32 = ptr(out), out.stride(0), ptr(out_f32)
    if saved is not None:
        _block_saved(f, saved)
    else:
        f.xhat = f.rstd = f.h = f.gp = None
    T, ffn = f.T, f.ffn
    rows = (2 if ffn else 3) + (2 if out_f32 is not None else 0) + ((3 if ffn else 1) if saved is not None else 0)
    _run("ffn_fwd" if ffn else "dense_ln_fwd", _lib.lib().pmgt_block_fwd, (C.byref(f), cur_stream()), 1,
         2 * T * 128 * rows + 2 * 128 * 128 * (2 if ffn else 1), 2 * T * 128 * 128 * (2 if ffn else 1))


def block_bwd(f: BlockArgs, saved: BlockSaved, dy, dx, dw2, db2, d_ln_g, d_ln_b, dy_b=None, dw1=None, db1=None, dz=None):
    """d(in) and the parameter gradients of the block from (in, saved, dy [+ dy_b]); dense block: ``dz`` receives the
    residual-branch gradient."""
    _block_saved(f, saved)
    f.dy, f.ld_dy = ptr(dy), dy.stride(0)
    f.dy_b, f.ld_dy_b = ptr(dy_b), (dy_b.stride(0) if dy_b is not None else 0)
    f.dx, f.ld_dx = ptr(dx), dx.stride(0)
    f.dz, f.ld_dz = ptr(dz), (dz.stride(0) if dz is not None else 0)
    f.dw1, f.dw2, f.db1, f.db2, f.d_ln_g, f.d_ln_b = ptr(dw1), ptr(dw2), ptr(db1), ptr(db2), ptr(d_ln_g), ptr(d_ln_b)
    T, ffn = f.T, f.ffn
    rows = (6 if ffn else 5) + (1 if dy_b is not None else 0)
    _run("ffn_bwd" if ffn else "dense_ln_bwd", _lib.lib().pmgt_block_bwd, (C.byref(f), cur_stream()), 1,
         2 * T * 128 * rows + 6 * 128 * 128 * (2 if ffn else 1), 2 * T * 128 * 128 * (4 if ffn else 2))


def dw_tile(dy, x, dw_f32, dbias=None, tag="dw_tile"):
    """``pmgt_dw_tile``: dw[N,K] += dy[T,N]^T @ x[T,K]; dbias[N] += dy.sum(0)."""
    T, N = dy.shape
    K = x.shape[1]
    a = DwTileArgs()
    a.T, a.N, a.K = T, N, K
    a.dy, a.ld_dy = ptr(dy), dy.stride(0)
    a.x, a.ldx = ptr(x), x.stride(0)
    a.dw, a.ld_dw = ptr(dw_f32), dw_f32.stride(0)
    a.dbias = ptr(dbias)
    _run(tag, _lib.lib().pmgt_dw_tile, (C.byref(a), cur_stream()), 1, 2 * T * (N + K) + 4 * N * K, 2 * T * N * K)


def dw_tile_batch(problems, tag="dw_tile"):
    """``pmgt_dw_tile_batch``: ``problems`` = [(dy, x, dw_f32, dbias-or-None), ...] of one shape, one launch."""
    n = len(problems)
    arr = (DwTileArgs * n)()
    nbytes = flops = 0
    for a, (dy, x, dw_f32, dbias) in zip(arr, problems):
        T, N = dy.shape
        K = x.shape[1]
        a.T, a.N, a.K = T, N, K
        a.dy, a.ld_dy = ptr(dy), dy.stride(0)
        a.x, a.ldx = ptr(x), x.stride(0)
        a.dw, a.ld_dw = ptr(dw_f32), dw_f32.stride(0)
        a.dbias = ptr(dbias)
        nbytes += 2 * T * (N + K) + 4 * N * K
        flops += 2 * T * N * K
    _run(tag, _lib.lib().pmgt_dw_tile_batch, (arr, n, cur_stream()), 1, nbytes, flops)


def ln_bwd(T, H, z, ln_g, eps, p, seed, site, dz, d_o, d_g, d_b, dy_a=None, dy_b=None, dy_f32=None):
    a = LnBwdArgs()
    a.T, a.H = T, H
    a.z, a.dy_a, a.dy_b, a.dy_f32 = ptr(z), ptr(dy_a), ptr(dy_b), ptr(dy_f32)
    a.ln_g, a.ln_eps = ptr(ln_g), eps
    a.dropout_p, a.dropout_seed, a.dropout_site = p, seed, site
    a.dz, a.d_o, a.d_g, a.d_b = ptr(dz), ptr(d_o), ptr(d_g), ptr(d_b)
    n_in = 1 + (dy_a is not None) + (dy_b is not None) + 2 * (dy_f32 is not None)
    n_out = 1 + (d_o is not None and d_o is not dz)
    _run("ln_bwd", _lib.lib().pmgt_ln_bwd, (C.byref(a), cur_stream()), 1, 2 * T * H * (n_in + n_out))


def embed_args(rows, L, H, ev, et, w_att, b_att, pos, role, ln_g, ln_b, eps, p, seed, site, **kw):
    a = EmbedArgs()
    a.rows, a.L, a.H = rows, L, H
    a.ev, a.et = ptr(ev), ptr(et)
    a.w_att, a.b_att, a.pos, a.role, a.ln_g, a.ln_b = ptr(w_att), ptr(b_att), ptr(pos), ptr(role), ptr(ln_g), ptr(ln_b)
    a.ln_eps, a.dropout_p, a.dropout_seed, a.dropout_site = eps, p, seed, site
    for k, v in kw.items():
        setattr(a, k, v if isinstance(v, (int, bool)) else ptr(v))
    return a


def embed_fuse_fwd(a: EmbedArgs):
    T = a.rows * a.L
    _run("embed_fuse_fwd", _lib.lib().pmgt_embed_fuse_fwd, (C.byref(a), cur_stream()), 1, 6 * T * a.H)


def embed_fuse_bwd(a: EmbedArgs):
    T = a.rows * a.L
    _run("embed_fuse_bwd", _lib.lib().pmgt_embed_fuse_bwd, (C.byref(a), cur_stream()), 1, 10 * T * a.H)


_PER_MODALITY = ("de", "d_bias", "de_acc")


def embed_multi_args(rows, L, H, e, w_att, b_att, pos, role, ln_g, ln_b, eps, p, seed, site, **kw):
    """``pmgt_embed_multi_args`` for ``len(e)`` modalities; ``de`` / ``d_bias`` / ``de_acc`` take one tensor per
    modality, the other keywords are the fields of ``pmgt_embed_args``."""
    a = EmbedMultiArgs()
    if not 1 <= len(e) <= _lib.MAX_MODALITIES:
        raise _lib.PMGTError(f"embed_multi_args: {len(e)} modalities, supported 1..{_lib.MAX_MODALITIES}")
    a.rows, a.L, a.H, a.n_mod = rows, L, H, len(e)
    for m, t in enumerate(e):
        a.e[m] = ptr(t)
    a.w_att, a.b_att, a.pos, a.role, a.ln_g, a.ln_b = ptr(w_att), ptr(b_att), ptr(pos), ptr(role), ptr(ln_g), ptr(ln_b)
    a.ln_eps, a.dropout_p, a.dropout_seed, a.dropout_site = eps, p, seed, site
    for k, v in kw.items():
        if k in _PER_MODALITY:
            arr = getattr(a, k)
            for m, t in enumerate(v):
                arr[m] = ptr(t)
        else:
            setattr(a, k, v if isinstance(v, (int, bool)) else ptr(v))
    return a


def embed_multi_fwd(a: EmbedMultiArgs):
    """Embedding fusion for 1..4 modalities (profile tag shared with the two-modality kernel)."""
    T = a.rows * a.L
    _run("embed_fuse_fwd", _lib.lib().pmgt_embed_multi_fwd, (C.byref(a), cur_stream()), 1, 2 * (a.n_mod + 1) * T * a.H)


def embed_multi_bwd(a: EmbedMultiArgs):
    T = a.rows * a.L
    _run("embed_fuse_bwd", _lib.lib().pmgt_embed_multi_bwd, (C.byref(a), cur_stream()), 1, 2 * (2 * a.n_mod + 1) * T * a.H)


def attn_args(rows, L, H, heads, beta, qkvc, mask, p, seed, site, **kw):
    a = AttnArgs()
    a.rows, a.L, a.H, a.heads, a.beta = rows, L, H, heads, beta
    a.qkvc, a.mask = ptr(qkvc), ptr(mask)
    a.dropout_p, a.dropout_seed, a.dropout_site = p, seed, site
    for k, v in kw.items():
        setattr(a, k, ptr(v))
    return a


def attn_core_fwd(a: AttnArgs):
    T = a.rows * a.L
    _run("attn_core_fwd", _lib.lib().pmgt_attn_core_fwd, (C.byref(a), cur_stream()), 1, 10 * T * a.H,
         6 * T * a.L * a.H)


def attn_core_bwd(a: AttnArgs):
    T = a.rows * a.L
    n_col = (4 * a.H + 2047) // 2048 if a.d_bias_qkvc else 0
    _run("attn_core_bwd", _lib.lib().pmgt_attn_core_bwd, (C.byref(a), cur_stream()), 1 + n_col,
         (18 + (8 if n_col else 0)) * T * a.H, 14 * T * a.L * a.H)


def resln_args(T, H, o, res, ln_g, ln_b, eps, p, seed, site, **kw):
    a = ResLnArgs()
    a.T, a.H = T, H
    a.o, a.res, a.ln_g, a.ln_b = ptr(o), ptr(res), ptr(ln_g), ptr(ln_b)
    a.ln_eps, a.dropout_p, a.dropout_seed, a.dropout_site = eps, p, seed, site
    for k, v in kw.items():
        setattr(a, k, ptr(v))
    return a


def res_ln_fwd(a: ResLnArgs):
    _run("res_ln_fwd", _lib.lib().pmgt_res_ln_fwd, (C.byref(a), cur_stream()), 1, (6 + (4 if a.y_f32 else 0)) * a.T * a.H)


def res_ln_bwd(a: ResLnArgs):
    per = 4 + (2 if a.dy else 0) + (4 if a.dy_f32 else 0) + 2 + (2 if (a.d_o and a.d_o != a.dz) else 0)
    _run("res_ln_bwd", _lib.lib().pmgt_res_ln_bwd, (C.byref(a), cur_stream()), 1, per * a.T * a.H)


def colsum(x, out_f32):
    T, N = x.shape
    _run("colsum", _lib.lib().pmgt_colsum_bf16, (ptr(x), T, N, x.stride(0), ptr(out_f32), cur_stream()),
         (N + 2047) // 2048, 2 * T * N)


def gsr(fwd: bool, B, SP, H, tgt_h, ld_t, pair_h, ld_p, pair_off, labels, logits=None, loss_out=None, grad_out=None,
        d_tgt=None, d_pair=None):
    a = GsrArgs(B, SP, H, ptr(tgt_h), ld_t, ptr(pair_h), ld_p, ptr(pair_off), ptr(labels), ptr(logits), ptr(loss_out),
                ptr(grad_out), ptr(d_tgt), ptr(d_pair))
    fn = _lib.lib().pmgt_gsr_fwd if fwd else _lib.lib().pmgt_gsr_bwd
    _run("gsr_fwd" if fwd else "gsr_bwd", fn, (C.byref(a), cur_stream()), 1, (4 if fwd else 8) * (B + SP) * H)


def nfr_mse(fwd: bool, Mm, D, proj, table, target_ids, weight, loss_out=None, grad_out=None, dproj=None):
    a = NfrArgs(Mm, D, ptr(proj), proj.stride(0) if proj is not None else 0, ptr(table), table.stride(0),
                ptr(target_ids), weight, ptr(loss_out), ptr(grad_out), ptr(dproj))
    fn = _lib.lib().pmgt_nfr_mse_fwd if fwd else _lib.lib().pmgt_nfr_mse_bwd
    _run("nfr_mse_fwd" if fwd else "nfr_mse_bwd", fn, (C.byref(a), cur_stream()), 1, (4 if fwd else 6) * Mm * D)


def cast_f32_bf16(src, dst):
    _run("cast_f32_bf16", _lib.lib().pmgt_cast_f32_bf16, (ptr(src), ptr(dst), src.numel(), cur_stream()), 1, 6 * src.numel())


def sumsq(x, out):
    _run("sumsq", _lib.lib().pmgt_sumsq_f32, (ptr(x), x.numel(), ptr(out), cur_stream()), 1, 4 * x.numel())


def peer_reduce(peer_ptrs, rank: int, n: int):
    """In-place sum of the flat fp32 vector whose per-rank copies are at ``peer_ptrs`` (symmetric memory); the caller
    brackets it with barriers over the ranks."""
    ws = len(peer_ptrs)
    arr = (C.c_uint64 * ws)(*[int(p) for p in peer_ptrs])
    _run("peer_reduce", _lib.lib().pmgt_peer_reduce_f32, (arr, ws, int(rank), int(n), cur_stream()), 1, 8 * n * (ws - 1) // ws)


def clip_coef(sumsq_buf, scale: float, max_norm: float, out):
    """out[0] = scale * min(1, max_norm / (sqrt(sumsq) * scale + 1e-6)); resets ``sumsq_buf`` (clip_grad_norm_)."""
    _run("clip_coef", _lib.lib().pmgt_clip_coef, (ptr(sumsq_buf), float(scale), float(max_norm), ptr(out), cur_stream()), 1, 8)


def gather_rows(src, idx, out):
    _run("gather_rows", _lib.lib().pmgt_gather_rows_bf16, (ptr(src), src.stride(0), ptr(idx), idx.numel(), src.shape[1],
                                                           ptr(out), out.stride(0), cur_stream()), 1,
         4 * idx.numel() * src.shape[1])


def scatter_rows(src, idx, dst):
    """dst[idx[r]] = src[r] (bf16 rows; idx unique)."""
    _run("scatter_rows", _lib.lib().pmgt_scatter_rows_bf16, (ptr(src), src.stride(0), ptr(idx), idx.numel(), src.shape[1],
                                                             ptr(dst), dst.stride(0), cur_stream()), 1,
         4 * idx.numel() * src.shape[1])


def adamw_step(p, g, m, v, decay_mask, lr, beta1, beta2, eps, weight_decay, step, grad_scale=1.0, grad_scale_dev=None):
    _run("adamw", _lib.lib().pmgt_adamw_step, (ptr(p), ptr(g), ptr(m), ptr(v), ptr(decay_mask), p.numel(), lr, beta1, beta2,
                                               eps, weight_decay, step, grad_scale, ptr(grad_scale_dev), cur_stream()),
         1, 29 * p.numel())


def sample_contexts(graph_handle, roots, keys, hops, max_ctx, seed, out_ids, out_mask, out_visited_deg=None):
    h = (C.c_int32 * len(hops))(*hops)
    _run("sample_contexts", _lib.lib().pmgt_sample_contexts,
         (graph_handle, ptr(roots), ptr(keys), roots.numel(), h, len(hops), max_ctx, seed, ptr(out_ids), ptr(out_mask),
          ptr(out_visited_deg), cur_stream()), 1, 0)


def sample_pairs(graph_handle, targets, keys, max_pos, min_neg, max_total, stride, seed, out_pairs, out_labels, out_num):
    _run("sample_pairs", _lib.lib().pmgt_sample_pairs,
         (graph_handle, ptr(targets), ptr(keys), targets.numel(), max_pos, min_neg, max_total, stride, seed,
          ptr(out_pairs), ptr(out_labels), ptr(out_num), cur_stream()), 1, 0)
