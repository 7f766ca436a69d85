"""Neighbour contexts of 64 < L <= 128 tokens on the B200: the attn_long attention core (attention_long.cu) against torch
fp32, its dropout mask against a numpy port of the common.cuh stream, the sampler at long contexts against the CPU
Philox replay, whole pre-training steps against the oracle, and the trainer end to end at max_ctx_neigh = 99.
Tolerances are those of test_kernels_gpu.py (attention core) and test_model_gpu.py (whole steps)."""
import math

import numpy as np
import pytest
import torch

from oracle import model_ref, sampler_ref

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


# ---------------------------------------------------------------------------------------------------------------------
# attention core parity
# ---------------------------------------------------------------------------------------------------------------------
def _attn_parity(R, L, H, heads, beta):
    ops = _ops()
    T = R * L
    qkvc = _r(T, 4 * H, s=0.7)
    mask = torch.ones(R, L, device="cuda")
    for r in range(R):  # ragged padding on the right; row 0 holds the target alone
        n_real = 0 if r == 0 else 1 + (r * 7) % (L - 1)
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


# (H, heads) per head size: two heads of 32, twelve heads of 64 (config-5 widths), one head of 128 (the default)
_HEADS = {32: (64, 2), 64: (768, 12), 128: (128, 1)}


@pytest.mark.parametrize("beta", [0.0, 0.3, 1.0])
@pytest.mark.parametrize("dh", [32, 64, 128])
@pytest.mark.parametrize("L", [65, 73, 74, 80, 96, 100, 113, 127, 128])
def test_long_attention_core_fwd_bwd(L, dh, beta):
    H, heads = _HEADS[dh]
    _attn_parity(5, L, H, heads, beta)


@pytest.mark.parametrize("L,H,heads", [(100, 768, 12), (128, 128, 1)])
def test_long_attention_core_many_ctas(L, H, heads):
    """rows * heads far above the 148 SMs: 4,800 and 600 CTAs."""
    _attn_parity(600 if heads == 1 else 400, L, H, heads, 0.5)


# ---------------------------------------------------------------------------------------------------------------------
# dropout: the generic kernel's element stream, ported to numpy
# ---------------------------------------------------------------------------------------------------------------------
_M32 = np.uint64(0xFFFFFFFF)


def _fmix32(x):
    x = x ^ (x >> np.uint64(16))
    x = (x * np.uint64(0x85EBCA6B)) & _M32
    x = x ^ (x >> np.uint64(13))
    x = (x * np.uint64(0xC2B2AE35)) & _M32
    return x ^ (x >> np.uint64(16))


def _dmix32(x):
    x = (x * np.uint64(0x85EBCA6B)) & _M32
    x = x ^ (x >> np.uint64(15))
    x = (x * np.uint64(0xC2B2AE35)) & _M32
    return x ^ (x >> np.uint64(16))


def dropout_keep_np(seed, site, idx, p):
    """dropout_keep(seed, site, idx, p) of common.cuh for an array of element indices."""
    idx = np.asarray(idx, dtype=np.uint64)
    seed, site = np.uint64(seed), np.uint64(site)
    blk = idx >> np.uint64(3)
    k1 = _fmix32((seed & _M32) ^ ((site * np.uint64(0x9E3779B9)) & _M32) ^ np.uint64(0x5EED))
    k2 = _fmix32(((seed >> np.uint64(32)) + site) & _M32) ^ (((blk >> np.uint64(30)) * np.uint64(0x9E3779B9)) & _M32)
    c = (blk << np.uint64(2)) & _M32
    w = _dmix32(((c + ((idx & np.uint64(7)) >> np.uint64(1))) & _M32) ^ k1) ^ k2
    field = np.where((idx & np.uint64(1)) == 1, w >> np.uint64(16), w & np.uint64(0xFFFF))
    thr = np.uint64(int(np.float32(p) * np.float32(65536.0) + np.float32(0.5)))
    return field >= thr


def _attention_matrix(R, L, dh, heads, beta, p, seed, site, qkvc=None):
    """A[r, h, i, j] of the forward pass: V set to unit vectors, a window of dh key columns per call."""
    ops = _ops()
    H = dh * heads
    T = R * L
    if qkvc is None:
        qkvc = _r(T, 4 * H, s=0.7)
    mask = torch.ones(R, L, device="cuda")
    A = torch.zeros(R, heads, L, L, device="cuda")
    for w0 in range(0, L, dh):
        w = min(dh, L - w0)
        v = torch.zeros(R, L, heads, dh, device="cuda")
        v[:, w0 + torch.arange(w), :, torch.arange(w)] = 1.0
        qkvc[:, 2 * H:3 * H] = v.view(T, H).to(BF16)
        ctx = torch.empty(T, H, device="cuda", dtype=BF16)
        ops.attn_core_fwd(ops.attn_args(R, L, H, heads, beta, qkvc, mask, p, seed, site, ctx=ctx))
        A[:, :, :, w0:w0 + w] = ctx.view(R, L, heads, dh)[..., :w].permute(0, 2, 1, 3).float()
    return A, qkvc, mask


def _port_keep(R, L, heads, seed, site, p):
    item = np.arange(R * heads, dtype=np.uint64).reshape(R, heads, 1, 1)
    ij = np.arange(L * L, dtype=np.uint64).reshape(1, 1, L, L)
    return torch.from_numpy(dropout_keep_np(seed, site, item * np.uint64(L * L) + ij, p))


def test_dropout_port_matches_the_generic_kernel():
    """The port itself, pinned to the device stream on a shape the generic kernel runs (L = 70, head size 16)."""
    R, L, dh, p = 3, 70, 16, 0.25
    A, _, _ = _attention_matrix(R, L, dh, 1, 1.0, p, 77, 3)
    assert torch.equal((A != 0).cpu(), _port_keep(R, L, 1, 77, 3, p))


@pytest.mark.parametrize("L,dh,heads", [(73, 128, 1), (128, 32, 2), (100, 64, 2), (65, 64, 1)])
def test_long_attention_dropout_is_the_generic_stream(L, dh, heads):
    R, p = 4, 0.25
    for beta, site in ((1.0, 3), (0.0, 4)):   # beta = 1: P1 only, mask of site 3; beta = 0: P2 only, site 3 + 1
        A, qkvc, mask = _attention_matrix(R, L, dh, heads, beta, p, 77, 3)
        keep = _port_keep(R, L, heads, 77, site, p)
        assert torch.equal((A != 0).cpu(), keep), (beta, int(((A != 0).cpu() != keep).sum()))
        assert abs(float(keep.float().mean()) - (1 - p)) < 0.015
        A0, _, _ = _attention_matrix(R, L, dh, heads, beta, 0.0, 77, 3, qkvc=qkvc.clone())
        kept = A != 0
        assert torch.allclose(A[kept], (A0 / (1 - p))[kept], rtol=3e-2, atol=2e-3)
    # the backward pass regenerates the same A: dV_j[5] = A[i*, j] for dctx = e_5 on row i* (dV does not depend on V)
    ops = _ops()
    H, T = dh * heads, R * L
    A, qkvc, mask = _attention_matrix(R, L, dh, heads, 1.0, p, 77, 3)
    for i_star in (0, L // 2, L - 1):
        dctx = torch.zeros(R, L, heads, dh, device="cuda")
        dctx[:, i_star, :, 5] = 1.0
        dqkvc = torch.empty_like(qkvc)
        ops.attn_core_bwd(ops.attn_args(R, L, H, heads, 1.0, qkvc, mask, p, 77, 3, dctx=dctx.view(T, H).to(BF16),
                                        dqkvc=dqkvc))
        dV = dqkvc[:, 2 * H:3 * H].float().view(R, L, heads, dh)[..., 5].permute(0, 2, 1)   # dV[r, h, j] = A[r, h, i*, j]
        want = A[:, :, i_star, :]
        assert torch.allclose(dV, want, rtol=2e-2, atol=2e-3), (i_star, float((dV - want).abs().max()))


# ---------------------------------------------------------------------------------------------------------------------
# sampler
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hops,max_ctx", [([16, 8, 4], 63), ([16, 8, 4], 99), ([16, 8, 4], 127), ([8, 6, 4, 3, 2], 99)])
def test_long_contexts_bit_exact_vs_cpu_replay(hops, max_ctx):
    from pmgt_b200 import synthetic
    from pmgt_b200.datasets import sample_contexts
    g = synthetic.make_item_graph((300, 4000), seed=4)
    roots = np.arange(2, g.num_nodes + 2, dtype=np.int64)
    keys = (np.arange(len(roots), dtype=np.int64) << 8) | 3
    dev = torch.device("cuda", 0)
    seed = 0x1234_5678_9ABC
    ids, mask, vdeg = sample_contexts(g, torch.as_tensor(roots, device=dev), torch.as_tensor(keys, device=dev), hops,
                                      max_ctx, seed, want_visited_deg=True)
    want = sampler_ref.philox_sample_contexts(g.indptr, g.indices, g.cdf, g.num_nodes, roots, keys, hops, max_ctx, seed)
    for a, b, name in zip((ids.cpu().numpy(), mask.cpu().numpy(), vdeg.cpu().numpy()), want, ("ids", "mask", "visited_deg")):
        assert np.array_equal(a, b), name
    assert ids.shape == (len(roots), max_ctx + 1)
    assert float(mask.sum(1).max()) > min(max_ctx, 64)   # some contexts are longer than 64 tokens (all full at 63)


# ---------------------------------------------------------------------------------------------------------------------
# whole pre-training steps
# ---------------------------------------------------------------------------------------------------------------------
def _check_grads(net, ref_grads, cos_min=0.995, norm_tol=0.05):
    """test_model_gpu.py's tolerances.  Tensors whose reference norm is ~0 are checked absolutely; at L = 100 that
    includes the modality-fusion bias, whose gradient sums ~8,000 per-token terms of a two-way softmax that cancel to a
    norm of ~3e-4, so ~0 here means a reference norm below 1e-3 and an absolute error below 1e-4."""
    for name, p in net.named_parameters():
        if not p.requires_grad:
            continue
        assert p.grad is not None, name
        want = ref_grads[name].to(p.grad.device).float()
        got = p.grad.float()
        assert torch.isfinite(got).all(), name
        wn = float(want.norm())
        if wn < 1e-3:
            assert float((got - want).abs().max()) < 1e-4, (name, float((got - want).abs().max()))
            continue
        cos = float((got * want).sum() / (got.norm() * want.norm()).clamp_min(1e-20))
        assert cos >= cos_min, f"{name}: cosine {cos:.5f}"
        assert abs(float(got.norm()) / wn - 1) <= norm_tol, f"{name}: norm ratio {float(got.norm()) / wn:.4f}"


@pytest.mark.parametrize("over,B,P,L,node_size", [
    (dict(), 16, 4, 100, 500),                                                          # default widths, L = 100
    (dict(hidden_size=256, num_hidden_layers=2, num_attention_heads=4, intermediate_size=512, feat_hidden_sizes=[256, 128],
          max_position_embeddings=128, mask_node_ratio=0.3), 8, 3, 128, 300),           # 4 heads of 64, L = 128
    (dict(hidden_size=64, num_hidden_layers=2, num_attention_heads=2, intermediate_size=64), 8, 4, 80, 300),  # 2 x 32
])
@pytest.mark.parametrize("projection", ["gather", "table"])
def test_long_context_pretrain_step_matches_oracle(over, B, P, L, node_size, projection, monkeypatch):
    from pmgt_b200 import PMGT, PMGTConfig, modeling_pmgt
    monkeypatch.setattr(modeling_pmgt, "PROJECTION_MODE", projection)
    cfg = model_ref.default_cfg(**over)
    sd = model_ref.init_state_dict(cfg, node_size, seed=21, perturb=0.05)
    c = PMGTConfig(hidden_size=cfg["hidden_size"], feat_hidden_sizes=cfg["feat_hidden_sizes"],
                   num_hidden_layers=cfg["num_hidden_layers"], num_attention_heads=cfg["num_attention_heads"],
                   intermediate_size=cfg["intermediate_size"], beta=cfg["beta"], hidden_dropout_prob=0.0,
                   attention_probs_dropout_prob=0.0, max_position_embeddings=cfg["max_position_embeddings"])
    net = PMGT(node_size, cfg["random_node_ratio"], cfg["mask_node_ratio"], c,
               feat_init_emb=[sd[f"feat_embeddings.{m}.weight"].cpu().numpy() for m in range(2)])
    missing, unexpected = net.load_state_dict({k: v.cpu() for k, v in sd.items()}, strict=False)
    assert not unexpected and all(k.endswith(("position_ids", "role_ids")) for k in missing)
    net = net.cuda().train()
    gen = torch.Generator().manual_seed(B + L)

    def ctx(rows):  # ragged: 1 .. L - 1 real neighbours
        ids = torch.randint(2, node_size + 2, (rows, L), generator=gen)
        n_real = torch.randint(1, L, (rows,), generator=gen)
        mask = (torch.arange(L)[None, :] <= n_real[:, None]).float()
        return {"node_ids": (ids * mask.long()).cuda(), "attention_mask": mask.cuda()}

    target, pair = ctx(B), ctx(B * P)
    num_pairs = torch.full((B,), P, dtype=torch.long).cuda()
    labels = (torch.rand(B * P, generator=gen) < 0.5).float().cuda()
    torch.manual_seed(77)
    masked = net.mask_nodes(target["node_ids"])
    out = net(target, pair, num_pairs, labels, masked_inputs=masked)
    out.loss.backward()
    sdc = {k: v.cuda() for k, v in sd.items()}
    for m in range(2):
        sdc[f"feat_embeddings.{m}.weight"] = sdc[f"feat_embeddings.{m}.weight"].to(BF16).float()
    params = {k: v.requires_grad_(True) for k, v in sdc.items() if not k.startswith("feat_embeddings")}
    ref = model_ref.pretrain_forward(sdc, cfg, node_size, target, pair, num_pairs, labels, training=True, masked=masked)
    ref["loss"].backward()
    assert abs(float(out.loss) - float(ref["loss"])) <= 2e-2 * abs(float(ref["loss"]))
    assert float((out.prediction_logits - ref["prediction_logits"]).abs().max()) < 3e-2
    rh = ref["last_hidden_state"].detach()
    assert float((out.last_hidden_state - rh).abs().max()) < 3e-2 * float(rh.abs().max())
    _check_grads(net, {k: v.grad for k, v in params.items()})


def test_long_context_launch_plan_matches_the_unplanned_path():
    """L = 100 with dropout on: recorded-and-replayed encoder launches give the losses of the unplanned path."""
    from pmgt_b200 import PMGT, PMGTConfig, PMGTDataset, modeling_pmgt, synthetic
    g = synthetic.make_item_graph((400, 6000), seed=1)
    feats = synthetic.make_features(g.num_nodes, seed=3)
    ds = PMGTDataset(g, max_ctx_neigh=99, seed=0)
    losses = []
    for planned in (False, True):
        torch.manual_seed(0)
        modeling_pmgt._seed_counter[0] = 0
        net = PMGT(g.num_nodes, config=PMGTConfig(num_hidden_layers=2), feat_init_emb=feats).cuda().train()
        net.bert.use_launch_plans = planned
        run = []
        for step in range(3):
            batch = ds.sample_batch(torch.arange(0, 64), epoch=step)
            assert batch[0]["node_ids"].shape[1] == 100
            for p in net.parameters():
                p.grad = None
            out = net(*batch)
            out.loss.backward()
            run.append(float(out.loss))
        if planned:
            plans = list(net.bert._plans.values())
            assert len(plans) == 1 and plans[0].fwd_tape and plans[0].bwd_tape, "the plan was not used"
        losses.append(run)
    for a, b in zip(*losses):
        assert np.isfinite(a) and abs(a - b) <= 1e-5 * abs(a), losses


# ---------------------------------------------------------------------------------------------------------------------
# trainer
# ---------------------------------------------------------------------------------------------------------------------
def test_trainer_end_to_end_at_99_neighbours(tmp_path):
    from pmgt_b200 import trainer
    kw = dict(synthetic=(400, 6000), train_batch_size=64, test_batch_size=128, num_epochs=2, num_hidden_layers=2, seed=3,
              log_dir=str(tmp_path), lr=2e-3, early=5, max_ctx_neigh=99, hidden_dropout_prob=0.1,
              attention_probs_dropout_prob=0.1)
    args = trainer.make_args(**kw)
    trainer.check_args(args)
    trainer.init_run(args)
    trainer.init_dataloader(args)
    trainer.init_model(args)
    best, tm = trainer.train(args)
    assert len(args.history) == 2
    for h in args.history:
        assert np.isfinite(h["loss/train"]) and np.isfinite(h["loss/val"])
        assert 0.0 <= h["val/auc"] <= 1.0
    ckpt = torch.load(args.best_model_path, map_location="cpu", weights_only=False)
    args2 = trainer.make_args(**kw)
    trainer.init_run(args2)
    trainer.init_dataloader(args2)
    trainer.init_model(args2)
    tm2 = trainer.PMGTTrainerModel(args2)
    tm2.load_state_dict(ckpt)
    tm.load_state_dict(ckpt)
    a, b = tm.evaluate(args.valid_dataset, 128), tm2.evaluate(args2.valid_dataset, 128)
    assert abs(a["loss"] - b["loss"]) <= 1e-5 * abs(a["loss"]) + 1e-6
    emb = trainer.inference(args)
    assert emb.shape == (len(args.graph), args.hidden_size) and np.isfinite(emb).all()
