"""Per-kernel parity (forward and backward) of the row-wise / attention / loss /
optimizer kernels against the fp32 torch oracle pieces (oracle/model_ref.py) on
identical inputs.  Inputs are rounded to bf16 first so the comparison isolates
the kernel arithmetic; outputs are bf16 -> tolerance 1e-2 of the tensor scale."""
import math
import os

import pytest
import torch

from oracle import model_ref

pytestmark = pytest.mark.gpu
BF16 = torch.bfloat16


def _ops():
    from pmgt_b200 import ops
    return ops


def _close(got, want, tol=1e-2, name=""):
    scale = want.abs().max().clamp_min(1e-6)
    err = float((got.float() - want).abs().max() / scale)
    assert torch.isfinite(got.float()).all(), f"{name}: non-finite"
    assert err < tol, f"{name}: max scaled error {err:.4g} >= {tol}"


def _r(*shape, s=1.0):
    return (torch.randn(*shape, device="cuda") * s).to(BF16)


@pytest.mark.parametrize("R,L,H", [(7, 6, 128), (5, 9, 64), (3, 33, 256), (4, 6, 32), (20001, 6, 128), (1, 1, 128)])
def test_embed_fuse_fwd_bwd(R, L, H):
    ops = _ops()
    T = R * L
    ev, et = _r(T, H), _r(T, H)
    w_att = torch.randn(2, 2 * H, device="cuda") * 0.2
    b_att = torch.randn(2, device="cuda") * 0.1
    pos = torch.randn(100, H, device="cuda") * 0.1
    role = torch.randn(2, H, device="cuda") * 0.1
    g = 1 + 0.1 * torch.randn(H, device="cuda")
    b = 0.1 * torch.randn(H, device="cuda")
    x = torch.empty(T, H, device="cuda", dtype=BF16)
    ops.embed_fuse_fwd(ops.embed_args(R, L, H, ev, et, w_att, b_att, pos, role, g, b, 1e-12, 0.0, 0, 0, x_out=x))

    leaves = [t.float().requires_grad_(True) for t in (ev, et)]
    leaves += [t.clone().requires_grad_(True) for t in (w_att, b_att, pos, role, g, b)]
    evf, etf, wa, ba, po, ro, gg, bb = leaves
    e = [evf.view(R, L, H), etf.view(R, L, H)]
    att = torch.softmax(torch.nn.functional.linear(torch.tanh(torch.cat(e, -1)), wa, ba), -1)
    fused = att[..., :1] * e[0] + att[..., 1:] * e[1]
    role_ids = torch.tensor([0] + [1] * (L - 1), device="cuda")
    want = torch.nn.functional.layer_norm(fused + po[:L] + ro[role_ids], (H,), gg, bb, 1e-12)
    _close(x.view(R, L, H), want.detach(), name="x")

    dx = _r(T, H)
    want.backward(dx.float().view(R, L, H))
    dev_, det_ = torch.empty_like(ev), torch.empty_like(et)

    def z(*s):
        return torch.zeros(*s, device="cuda")

    d = dict(d_w_att=z(2, 2 * H), d_b_att=z(2), d_pos=z(100, H), d_role=z(2, H), d_ln_g=z(H), d_ln_b=z(H),
             d_bias_v=z(H), d_bias_t=z(H))
    ops.embed_fuse_bwd(ops.embed_args(R, L, H, ev, et, w_att, b_att, pos, role, g, b, 1e-12, 0.0, 0, 0, dx=dx,
                                      dev=dev_, det=det_, **d))
    _close(dev_, evf.grad, name="dev")
    _close(det_, etf.grad, name="det")
    _close(d["d_w_att"], wa.grad, 5e-3, "d_w_att")
    _close(d["d_b_att"], ba.grad, 5e-3, "d_b_att")
    _close(d["d_pos"], po.grad, 5e-3, "d_pos")
    _close(d["d_role"], ro.grad, 5e-3, "d_role")
    _close(d["d_ln_g"], gg.grad, 5e-3, "d_ln_g")
    _close(d["d_ln_b"], bb.grad, 5e-3, "d_ln_b")
    _close(d["d_bias_v"], evf.grad.sum(0), 1e-2, "d_bias_v")
    _close(d["d_bias_t"], etf.grad.sum(0), 1e-2, "d_bias_t")


@pytest.mark.parametrize("R,L,rows", [(9, 6, 40), (9001, 6, 300)])
def test_embed_fuse_projected_table_mode(R, L, rows):
    """Projected-table mode (row_idx gather, fp32 per-row gradient accumulation) + the second gradient term dx_b."""
    ops = _ops()
    H, T = 128, R * L
    tv, tt = _r(rows, H), _r(rows, H)
    idx = torch.randint(0, rows, (T,), device="cuda")
    idx[::7] = 0  # pad rows
    w_att = torch.randn(2, 2 * H, device="cuda") * 0.2
    b_att = torch.randn(2, device="cuda") * 0.1
    pos = torch.randn(100, H, device="cuda") * 0.1
    role = torch.randn(2, H, device="cuda") * 0.1
    g = 1 + 0.1 * torch.randn(H, device="cuda")
    b = 0.1 * torch.randn(H, device="cuda")
    x = torch.empty(T, H, device="cuda", dtype=BF16)
    ops.embed_fuse_fwd(ops.embed_args(R, L, H, tv, tt, w_att, b_att, pos, role, g, b, 1e-12, 0.0, 0, 0, x_out=x, row_idx=idx))
    leaves = [t.float().requires_grad_(True) for t in (tv, tt)]
    leaves += [t.clone().requires_grad_(True) for t in (w_att, b_att, pos, role, g, b)]
    tvf, ttf, wa, ba, po, ro, gg, bb = leaves
    e = [tvf[idx].view(R, L, H), ttf[idx].view(R, L, H)]
    att = torch.softmax(torch.nn.functional.linear(torch.tanh(torch.cat(e, -1)), wa, ba), -1)
    fused = att[..., :1] * e[0] + att[..., 1:] * e[1]
    role_ids = torch.tensor([0] + [1] * (L - 1), device="cuda")
    want = torch.nn.functional.layer_norm(fused + po[:L] + ro[role_ids], (H,), gg, bb, 1e-12)
    _close(x.view(R, L, H), want.detach(), name="x")
    dx, dxb = _r(T, H), _r(T, H)
    want.backward((dx.float() + dxb.float()).view(R, L, H))

    def z(*s):
        return torch.zeros(*s, device="cuda")

    d = dict(d_w_att=z(2, 2 * H), d_b_att=z(2), d_pos=z(100, H), d_role=z(2, H), d_ln_g=z(H), d_ln_b=z(H),
             d_bias_v=z(H), d_bias_t=z(H))
    acc_v, acc_t = z(rows, H), z(rows, H)
    ops.embed_fuse_bwd(ops.embed_args(R, L, H, tv, tt, w_att, b_att, pos, role, g, b, 1e-12, 0.0, 0, 0, dx=dx, dx_b=dxb,
                                      row_idx=idx, dev_acc=acc_v, det_acc=acc_t, skip_row0=0, **d))
    _close(acc_v, tvf.grad, name="dev_acc")
    _close(acc_t, ttf.grad, name="det_acc")
    for k, want_g in (("d_w_att", wa.grad), ("d_b_att", ba.grad), ("d_pos", po.grad), ("d_role", ro.grad),
                      ("d_ln_g", gg.grad), ("d_ln_b", bb.grad)):
        _close(d[k], want_g, 5e-3, k)
    _close(d["d_bias_v"], tvf.grad.sum(0), 1e-2, "d_bias_v")
    _close(d["d_bias_t"], ttf.grad.sum(0), 1e-2, "d_bias_t")
    # skip_row0: the <pad> row receives nothing, every other row is unchanged
    acc_v2, acc_t2 = z(rows, H), z(rows, H)
    d2 = {k: torch.zeros_like(v) for k, v in d.items()}
    ops.embed_fuse_bwd(ops.embed_args(R, L, H, tv, tt, w_att, b_att, pos, role, g, b, 1e-12, 0.0, 0, 0, dx=dx, dx_b=dxb,
                                      row_idx=idx, dev_acc=acc_v2, det_acc=acc_t2, skip_row0=1, **d2))
    assert float(acc_v2[0].abs().max()) == 0.0 and float(acc_t2[0].abs().max()) == 0.0
    _close(acc_v2[1:], tvf.grad[1:], name="dev_acc[1:]")


def test_embed_fuse_dropout_mask_agrees_between_fwd_and_bwd():
    """Train-mode dropout of the embedding block: keep rate, 1/(1-p) scaling, and the backward pass regenerating the
    same mask (gradient of dropped elements is exactly zero in d LayerNorm beta's per-element view)."""
    ops = _ops()
    R, L, H, p = 3000, 6, 128, 0.1
    T = R * L
    ev, et = _r(T, H), _r(T, H)
    w_att = torch.randn(2, 2 * H, device="cuda") * 0.2
    b_att = torch.zeros(2, device="cuda")
    pos = torch.zeros(100, H, device="cuda")
    role = torch.zeros(2, H, device="cuda")
    g = torch.ones(H, device="cuda")
    b = torch.full((H,), 3.0, device="cuda")  # keeps every undropped output away from zero
    x0 = torch.empty(T, H, device="cuda", dtype=BF16)
    x1 = torch.empty(T, H, device="cuda", dtype=BF16)
    ops.embed_fuse_fwd(ops.embed_args(R, L, H, ev, et, w_att, b_att, pos, role, g, b, 1e-12, 0.0, 5, 0, x_out=x0))
    ops.embed_fuse_fwd(ops.embed_args(R, L, H, ev, et, w_att, b_att, pos, role, g, b, 1e-12, p, 5, 0, x_out=x1))
    keep = x1 != 0
    rate = float(keep.float().mean())
    assert abs(rate - (1 - p)) < 5e-3, rate
    _close(x1[keep].float(), x0[keep].float() / (1 - p), 1e-2, "kept values scaled by 1/(1-p)")

    def z(*s):
        return torch.zeros(*s, device="cuda")

    d = dict(d_w_att=z(2, 2 * H), d_b_att=z(2), d_pos=z(100, H), d_role=z(2, H), d_ln_g=z(H), d_ln_b=z(H),
             d_bias_v=z(H), d_bias_t=z(H))
    dx = torch.ones(T, H, device="cuda", dtype=BF16)
    dev_, det_ = torch.empty_like(ev), torch.empty_like(et)
    ops.embed_fuse_bwd(ops.embed_args(R, L, H, ev, et, w_att, b_att, pos, role, g, b, 1e-12, p, 5, 0, dx=dx, dev=dev_,
                                      det=det_, **d))
    # d LayerNorm beta = column sums of the masked, rescaled upstream gradient (all ones here)
    _close(d["d_ln_b"], keep.float().sum(0) / (1 - p), 1e-4, "d_ln_b counts the kept elements")


@pytest.mark.parametrize("R,L,H,heads,beta", [(9, 6, 128, 1, 0.5), (5, 9, 64, 4, 0.3), (3, 33, 192, 3, 0.5),
                                              (4, 6, 32, 1, 1.0),
                                              # medium-L tensor-core kernel (attention_mid.cu): config-5 heads, L = 64,
                                              # one / three k-tiles, head sizes 32 / 48 / 128, more items than warps
                                              (4, 33, 768, 12, 0.5), (3, 64, 128, 4, 0.7), (40, 17, 256, 2, 0.2),
                                              (5, 12, 96, 2, 0.0), (2, 48, 64, 1, 0.5),
                                              # register-resident kernel (attention_reg.cu): one row block (L = 12 / 16), L an exact
                                              # multiple of 16, head sizes 32 / 64 / 128
                                              (6, 12, 128, 2, 0.5), (3, 16, 64, 2, 0.4), (4, 32, 256, 2, 0.6), (7, 10, 128, 1, 0.5)])
def test_attention_core_fwd_bwd(R, L, H, heads, beta):
    ops = _ops()
    T = R * L
    qkvc = _r(T, 4 * H, s=0.7)
    mask = torch.ones(R, L, device="cuda")
    for r in range(R):  # ragged padding on the right, at least one real neighbour
        n_real = 1 + (r * 7) % (L - 1)
        mask[r, n_real + 1:] = 0
    ctx = torch.empty(T, H, device="cuda", dtype=BF16)
    ops.attn_core_fwd(ops.attn_args(R, L, H, heads, beta, qkvc, mask, 0.0, 0, 0, ctx=ctx))

    x = qkvc.float().requires_grad_(True)
    dh = H // heads
    q, k, v, c = [x[:, i * H:(i + 1) * H].view(R, L, heads, dh).permute(0, 2, 1, 3) for i in range(4)]
    ext = (1.0 - mask[:, None, None, :]) * -10000.0
    n = torch.linalg.norm(c, dim=-1, keepdim=True)
    s1 = 1.0 - (c @ c.transpose(-1, -2)) / (n @ n.transpose(-1, -2)) + torch.eye(L, device="cuda")
    p1 = torch.softmax(s1 + ext, -1)
    p2 = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(dh) + ext, -1)
    want = ((beta * p1 + (1 - beta) * p2) @ v).permute(0, 2, 1, 3).reshape(T, H)
    _close(ctx, want.detach(), name="ctx")

    dctx = _r(T, H)
    want.backward(dctx.float())
    dqkvc = torch.empty_like(qkvc)
    dbias = torch.zeros(4 * H, device="cuda")
    ops.attn_core_bwd(ops.attn_args(R, L, H, heads, beta, qkvc, mask, 0.0, 0, 0, dctx=dctx, dqkvc=dqkvc,
                                    d_bias_qkvc=dbias))
    for i, nm in enumerate("qkvc"):
        _close(dqkvc[:, i * H:(i + 1) * H], x.grad[:, i * H:(i + 1) * H], 1.5e-2, "d" + nm)
    _close(dbias, dqkvc.float().sum(0), 1e-3, "d_bias_qkvc")


@pytest.mark.parametrize("L,dh", [(33, 64), (20, 32), (64, 128),  # attn_reg
                                  (6, 128), (33, 48), (70, 128)])  # attn_mma, attn_mid, generic
def test_attention_dropout_mask_agrees_between_fwd_and_bwd(L, dh):
    """Attention core in train mode, one shape per kernel family: with V = the first L unit vectors the forward output
    rows ARE the dropped attention matrix A; the backward pass (which regenerates the mask, attn_reg in the transposed
    orientation) must see the same A: dV_j[c] = A_{i j} for dctx = e_c at row i.  Also the keep rate."""
    ops = _ops()
    R, H, heads, p = max(6, 2048 // (L * L)), dh, 1, 0.25  # >= 2048 dropout draws for the keep-rate check
    T = R * L
    qkvc = _r(T, 4 * H, s=0.7)
    v = torch.zeros(R, L, H, device="cuda")
    v[:, torch.arange(L), torch.arange(L)] = 1.0
    qkvc[:, 2 * H:3 * H] = v.view(T, H).to(BF16)
    mask = torch.ones(R, L, device="cuda")
    ctx = torch.empty(T, H, device="cuda", dtype=BF16)
    ops.attn_core_fwd(ops.attn_args(R, L, H, heads, 1.0, qkvc, mask, p, 77, 3, ctx=ctx))
    A = ctx.view(R, L, H)[:, :, :L].float()            # A[r, i, j]
    zero_rate = float((A == 0).float().mean())
    assert abs(zero_rate - p) < 0.03, zero_rate
    ctx0 = torch.empty_like(ctx)
    ops.attn_core_fwd(ops.attn_args(R, L, H, heads, 1.0, qkvc, mask, 0.0, 77, 3, ctx=ctx0))
    A0 = ctx0.view(R, L, H)[:, :, :L].float()
    kept = A != 0
    assert torch.allclose(A[kept], (A0 / (1 - p))[kept], rtol=3e-2, atol=2e-3)
    for i_star in (0, L // 2, L - 1):
        dctx = torch.zeros(R, L, H, device="cuda")
        dctx[:, i_star, 5] = 1.0
        dqkvc = torch.empty_like(qkvc)
        ops.attn_core_bwd(ops.attn_args(R, L, H, heads, 1.0, qkvc, mask, p, 77, 3, dctx=dctx.view(T, H).to(BF16), dqkvc=dqkvc))
        dV = dqkvc[:, 2 * H:3 * H].float().view(R, L, H)[:, :, 5]     # dV[r, j] = A[r, i*, j]
        assert torch.allclose(dV, A[:, i_star, :], rtol=2e-2, atol=2e-3), (i_star, float((dV - A[:, i_star, :]).abs().max()))


@pytest.mark.parametrize("which", ["ctx", "dctx", "dqkvc"])
def test_attention_rejects_misaligned_buffers(which):
    """qkvc / ctx / dctx / dqkvc must be 16-byte aligned.  A view 8 bytes into a buffer is rejected and named, whichever
    kernel the shape selects, instead of switching kernels (which changed the dropout stream between fwd and bwd)."""
    from pmgt_b200._lib import PMGTError
    ops = _ops()
    R, L, H, heads, p = 4, 33, 768, 12, 0.1  # attn_reg
    T = R * L
    qkvc = _r(T, 4 * H, s=0.7)
    mask = torch.ones(R, L, device="cuda")
    bufs = dict(ctx=torch.empty(T, H, device="cuda", dtype=BF16), dctx=_r(T, H), dqkvc=torch.empty_like(qkvc))
    t = bufs[which]
    bufs[which] = torch.empty(t.numel() + 4, device="cuda", dtype=BF16)[4:4 + t.numel()].view(t.shape).copy_(t)
    assert bufs[which].data_ptr() % 16 == 8
    with pytest.raises(PMGTError, match=f"{which} must be 16-byte aligned"):
        if which == "ctx":
            ops.attn_core_fwd(ops.attn_args(R, L, H, heads, 0.5, qkvc, mask, p, 7, 3, ctx=bufs["ctx"]))
        else:
            ops.attn_core_bwd(ops.attn_args(R, L, H, heads, 0.5, qkvc, mask, p, 7, 3, dctx=bufs["dctx"],
                                            dqkvc=bufs["dqkvc"]))
    torch.cuda.synchronize()


@pytest.mark.parametrize("T,H", [(50, 128), (33, 64), (20, 768), (9, 32), (5001, 768), (3000, 256), (1300, 1024), (77, 512)])
def test_res_ln_fwd_bwd(T, H):
    ops = _ops()
    o, res = _r(T, H), _r(T, H)
    g = 1 + 0.1 * torch.randn(H, device="cuda")
    b = 0.1 * torch.randn(H, device="cuda")
    y = torch.empty(T, H, device="cuda", dtype=BF16)
    y32 = torch.empty(T, H, device="cuda")
    ops.res_ln_fwd(ops.resln_args(T, H, o, res, g, b, 1e-12, 0.0, 0, 0, y=y, y_f32=y32))
    of, rf = o.float().requires_grad_(True), res.float().requires_grad_(True)
    gg, bb = g.clone().requires_grad_(True), b.clone().requires_grad_(True)
    want = torch.nn.functional.layer_norm(of + rf, (H,), gg, bb, 1e-12)
    _close(y, want.detach(), name="y")
    _close(y32, want.detach(), 1e-4, name="y_f32")
    dy = _r(T, H)
    dy32 = torch.randn(T, H, device="cuda")
    want.backward(dy.float() + dy32)
    dz = torch.empty(T, H, device="cuda", dtype=BF16)
    dg, db, dbias = torch.zeros(H, device="cuda"), torch.zeros(H, device="cuda"), torch.zeros(H, device="cuda")
    ops.res_ln_bwd(ops.resln_args(T, H, o, res, g, None, 1e-12, 0.0, 0, 0, dy=dy, dy_f32=dy32, dz=dz, d_o=dz, d_g=dg,
                                  d_b=db, d_bias=dbias))
    _close(dz, of.grad, name="dz")
    _close(dg, gg.grad, 5e-3, "d_g")
    _close(db, bb.grad, 5e-3, "d_b")
    _close(dbias, of.grad.sum(0), 1e-2, "d_bias")


@pytest.mark.parametrize("H", [768, 256])
def test_wide_res_ln_dropout_is_consistent_between_fwd_and_bwd(H):
    """res_ln_wide.cu (H a multiple of 256): keep rate, the backward pass regenerating the forward mask, and the
    same mask as the generic row-wise kernels would draw (one stream, common.cuh)."""
    ops = _ops()
    T, p = 3000, 0.25
    o = torch.ones(T, H, device="cuda", dtype=BF16)
    res = torch.zeros(T, H, device="cuda", dtype=BF16)
    g, b = torch.ones(H, device="cuda"), torch.zeros(H, device="cuda")
    y = torch.empty(T, H, device="cuda", dtype=BF16)
    ops.res_ln_fwd(ops.resln_args(T, H, o, res, g, b, 1e-12, p, 1234, 7, y=y))
    dropped = y.float() < 0
    rate = float(dropped.float().mean())
    assert abs(rate - p) < 0.01, rate
    dy = torch.randn(T, H, device="cuda").to(BF16)
    dz, d_o = torch.empty_like(y), torch.empty_like(y)
    dbias = torch.zeros(H, device="cuda")
    ops.res_ln_bwd(ops.resln_args(T, H, o, res, g, None, 1e-12, p, 1234, 7, dy=dy, dz=dz, d_o=d_o,
                                  d_g=torch.zeros(H, device="cuda"), d_b=torch.zeros(H, device="cuda"), d_bias=dbias))
    assert bool((d_o.float()[dropped] == 0).all())
    kept = ~dropped
    assert torch.allclose(d_o.float()[kept], (dz.float() / (1 - p))[kept], rtol=2e-2, atol=1e-3)
    _close(dbias, d_o.float().sum(0), 2e-3, "d_bias = column sums of the stored d_o")
    # the 4-columns-per-lane kernels (a sliced view breaks the 16-byte alignment the wide kernels ask for) draw the same mask
    pad = torch.ones(T * H + 4, device="cuda", dtype=BF16)
    o2 = pad[4:].view(T, H)
    y2 = torch.empty(T * H + 4, device="cuda", dtype=BF16)[4:].view(T, H)
    ops.res_ln_fwd(ops.resln_args(T, H, o2, res, g, b, 1e-12, p, 1234, 7, y=y2))
    assert torch.equal(y2.float() < 0, dropped)


def test_dropout_is_consistent_between_fwd_and_bwd():
    """Philox dropout: keep-rate ~ 1-p, kept values scaled by 1/(1-p), and the backward
    regenerates the same mask (gradient is zero exactly where the forward dropped)."""
    ops = _ops()
    T, H, p = 400, 128, 0.25
    o = torch.ones(T, H, device="cuda", dtype=BF16)
    res = torch.zeros(T, H, device="cuda", dtype=BF16)
    g, b = torch.ones(H, device="cuda"), torch.zeros(H, device="cuda")
    y = torch.empty(T, H, device="cuda", dtype=BF16)
    ops.res_ln_fwd(ops.resln_args(T, H, o, res, g, b, 1e-12, p, 1234, 7, y=y))
    dropped = y.float() < 0  # LayerNorm of a dropped row: dropped entries are the row minimum
    rate = float(dropped.float().mean())
    assert abs(rate - p) < 0.02, rate
    dy = torch.randn(T, H, device="cuda").to(BF16)
    dz = torch.empty_like(y)
    d_o = torch.empty_like(y)
    ops.res_ln_bwd(ops.resln_args(T, H, o, res, g, None, 1e-12, p, 1234, 7, dy=dy, dz=dz, d_o=d_o,
                                  d_g=torch.zeros(H, device="cuda"), d_b=torch.zeros(H, device="cuda"),
                                  d_bias=torch.zeros(H, device="cuda")))
    assert bool((d_o.float()[dropped] == 0).all())
    kept = ~dropped
    assert torch.allclose(d_o.float()[kept], (dz.float() / (1 - p))[kept], rtol=2e-2, atol=1e-3)
    y2 = torch.empty_like(y)
    ops.res_ln_fwd(ops.resln_args(T, H, o, res, g, b, 1e-12, p, 1235, 7, y=y2))
    assert not torch.equal(y, y2)  # another seed, another mask


def test_clip_coef_matches_clip_grad_norm():
    """pmgt_clip_coef: scale * min(1, max_norm / (sqrt(sumsq) * scale + 1e-6)) and the accumulator reset."""
    ops = _ops()
    for ss, scale, mx in ((4.0, 1.0, 1.0), (0.25, 0.5, 1.0), (9.0e4, 0.125, 2.0), (0.0, 1.0, 1.0)):
        acc = torch.tensor([ss], device="cuda")
        out = torch.empty(1, device="cuda")
        ops.clip_coef(acc, scale, mx, out)
        norm = ss ** 0.5 * scale
        want = scale * min(1.0, mx / (norm + 1e-6))
        assert abs(float(out) - want) <= 1e-6 * max(1.0, abs(want)), (float(out), want)
        assert float(acc) == 0.0


@pytest.mark.parametrize("ws,n", [(2, 1000), (4, 1_187_003), (8, 4099), (3, 5)])
def test_peer_reduce_sums_every_copy_in_place(ws, n):
    """pmgt_peer_reduce_f32 with the ranks' copies emulated by `ws` buffers on one device: after every rank has reduced
    its slice, every copy holds the sum (including the elements beyond the last whole float4)."""
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(n)
    bufs = [torch.randn(n, device="cuda", generator=g) for _ in range(ws)]
    want = torch.stack(bufs).double().sum(0)
    ptrs = [b.data_ptr() for b in bufs]
    for r in range(ws):
        ops.peer_reduce(ptrs, r, n)
    torch.cuda.synchronize()
    for b in bufs:
        assert torch.allclose(b.double(), want, rtol=1e-5, atol=1e-5)
    assert all(torch.equal(bufs[0], b) for b in bufs)


def test_colsum_cast_gather_sumsq():
    ops = _ops()
    x = _r(1234, 512)
    out = torch.ones(512, device="cuda")
    ops.colsum(x, out)
    _close(out, x.float().sum(0) + 1, 1e-4, "colsum")
    x2 = _r(77, 3072)
    out2 = torch.zeros(3072, device="cuda")
    ops.colsum(x2, out2)
    _close(out2, x2.float().sum(0), 1e-4, "colsum wide")
    src = torch.randn(100003, device="cuda")
    dst = torch.empty(100003, device="cuda", dtype=BF16)
    ops.cast_f32_bf16(src, dst)
    assert torch.equal(dst, src.to(BF16))
    table = _r(50, 64)
    idx = torch.randint(0, 50, (33,), device="cuda")
    g = torch.empty(33, 64, device="cuda", dtype=BF16)
    ops.gather_rows(table, idx, g)
    assert torch.equal(g, table[idx])
    s = torch.zeros(1, device="cuda")
    ops.sumsq(src, s)
    assert abs(float(s) - float((src.double() ** 2).sum())) < 1e-3 * float(s)


@pytest.mark.parametrize("B,P,H", [(5, 10, 128), (3, 2, 64), (4, 7, 768)])
def test_gsr_loss_fwd_bwd(B, P, H):
    from pmgt_b200.modeling_pmgt import PMGTGraphConstructLoss
    t = torch.randn(B, H, device="cuda", requires_grad=True)
    p = torch.randn(B * P, H, device="cuda", requires_grad=True)
    labels = (torch.rand(B * P, device="cuda") < 0.5).float()
    off = torch.arange(0, B * P + 1, P, device="cuda", dtype=torch.int64)
    loss, logits = PMGTGraphConstructLoss.batched(t, p, off, labels)
    (loss * 1.7).backward()
    t2, p2 = t.detach().clone().requires_grad_(True), p.detach().clone().requires_grad_(True)
    ls, lg = zip(*[model_ref.gsr_loss(p2[i * P:(i + 1) * P], t2[i], labels[i * P:(i + 1) * P]) for i in range(B)])
    want = torch.stack(ls).mean()
    (want * 1.7).backward()
    assert torch.allclose(loss, want, rtol=1e-4, atol=1e-6)
    assert torch.allclose(logits, torch.cat(lg), rtol=1e-4, atol=1e-5)
    _close(t.grad, t2.grad, 1e-3, "d_tgt")
    _close(p.grad, p2.grad, 1e-3, "d_pair")
    # reference per-target signature
    l1, g1 = PMGTGraphConstructLoss()(p[:P].detach(), t[0].detach(), labels[:P])
    assert torch.allclose(l1, ls[0], rtol=1e-4) and torch.allclose(g1, lg[0], rtol=1e-4, atol=1e-5)


def test_nfr_loss_fwd_bwd():
    from pmgt_b200 import PMGTConfig
    from pmgt_b200.modeling_pmgt import PMGTNodeConstructLoss
    cfg = PMGTConfig(hidden_size=64, feat_hidden_sizes=[128, 64])
    mod = PMGTNodeConstructLoss(cfg).cuda()
    Mm = 37
    h = torch.randn(Mm, 64, device="cuda").to(BF16).float().requires_grad_(True)
    targets = [_r(Mm, 128).float(), _r(Mm, 64).float()]
    loss = mod(h, targets)
    loss.backward()
    sd = {}
    for m in range(2):
        sd[f"nfr_loss.projections.{m}.weight"] = mod.projections[m].weight.detach().to(BF16).float().requires_grad_(True)
        sd[f"nfr_loss.projections.{m}.bias"] = mod.projections[m].bias.detach().clone().requires_grad_(True)
    h2 = h.detach().clone().requires_grad_(True)
    want = model_ref.nfr_loss(sd, h2, targets)
    want.backward()
    assert torch.allclose(loss, want, rtol=2e-2), (float(loss), float(want))
    _close(h.grad, h2.grad, 2e-2, "d_h")
    for m in range(2):
        _close(mod.projections[m].weight.grad, sd[f"nfr_loss.projections.{m}.weight"].grad, 2e-2, f"dW{m}")
        _close(mod.projections[m].bias.grad, sd[f"nfr_loss.projections.{m}.bias"].grad, 2e-2, f"db{m}")


def test_adamw_matches_reference_golden(golden_dir):
    from pmgt_b200 import DenseSparseAdamW
    g = torch.load(os.path.join(golden_dir, "adamw_golden.pt"), weights_only=False)
    p = torch.nn.Parameter(g["p0"].clone().cuda())
    opt = DenseSparseAdamW([{"params": [p], "weight_decay": g["weight_decay"], "lr": g["lr"]}])
    for gr, want in zip(g["grads"], g["traj"]):
        p.grad = gr.clone().cuda()
        opt.step()
        assert torch.allclose(p.detach().cpu(), want, rtol=1e-5, atol=1e-6)
