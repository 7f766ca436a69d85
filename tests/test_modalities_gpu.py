"""One, three and four feature modalities on the B200: the fusion kernels (pmgt_embed_multi_fwd / _bwd) against torch
fp32, their dropout mask against the two-modality kernels, whole pre-training steps against the fp32 oracle (tolerances
of DESIGN section 2, as in test_model_gpu.py), launch plans, and the trainer end to end."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import model_ref
from test_modalities import pretrain_forward  # the oracle's pre-training forward for any number of modalities

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------------
# fusion kernels
# ---------------------------------------------------------------------------------------------------------------------
def _fusion_inputs(M, H, rows, L, table_rows, seed):
    g = torch.Generator().manual_seed(seed)
    dev = "cuda"
    n_src = table_rows if table_rows else rows * L
    e = [torch.randn(n_src, H, generator=g).to(dev, torch.bfloat16) for _ in range(M)]
    p = dict(w_att=torch.randn(M, M * H, generator=g) * 0.05, b_att=torch.randn(M, generator=g) * 0.3,
             pos=torch.randn(L + 3, H, generator=g) * 0.1, role=torch.randn(2, H, generator=g) * 0.1,
             ln_g=1 + torch.randn(H, generator=g) * 0.1, ln_b=torch.randn(H, generator=g) * 0.1)
    p = {k: v.to(dev) for k, v in p.items()}
    row_idx = None
    if table_rows:
        row_idx = torch.randint(0, table_rows, (rows * L,), generator=g).to(dev)
        row_idx[::7] = 0   # <pad> tokens
    dx = torch.randn(rows * L, H, generator=g).to(dev, torch.bfloat16)
    dx_b = torch.randn(rows * L, H, generator=g).to(dev, torch.bfloat16)
    return e, p, row_idx, dx, dx_b


def _torch_fusion(e, p, row_idx, L, eps, keep=None, scale=1.0):
    """PMGTEmbeddings.forward in fp32 (oracle/model_ref.embeddings on flat tokens); keep = dropout mask."""
    x = [t.float() if row_idx is None else t.float()[row_idx] for t in e]
    T, H = x[0].shape
    att = torch.softmax(torch.tanh(torch.cat(x, dim=-1)) @ p["w_att"].T + p["b_att"], dim=-1)
    fused = sum(att[:, m: m + 1] * x[m] for m in range(len(x)))
    l = torch.arange(T, device=fused.device) % L
    z = fused + p["pos"][l] + p["role"][(l > 0).long()]
    y = F.layer_norm(z, (H,), p["ln_g"], p["ln_b"], eps)
    if keep is not None:
        y = y * keep * scale
    return y


def _rel(got, want):
    return float((got.float() - want.float()).norm() / want.float().norm().clamp_min(1e-30))


def _run_kernels(e, p, row_idx, dx, dx_b, rows, L, H, eps, drop=0.0, seed=0, skip_row0=0):
    from pmgt_b200 import ops
    M = len(e)
    T = rows * L
    x = torch.empty(T, H, dtype=torch.bfloat16, device="cuda")
    kw = dict(row_idx=row_idx) if row_idx is not None else {}
    ops.embed_multi_fwd(ops.embed_multi_args(rows, L, H, e, p["w_att"], p["b_att"], p["pos"], p["role"], p["ln_g"],
                                             p["ln_b"], eps, drop, seed, 0, x_out=x, **kw))
    grads = {k: torch.zeros_like(v) for k, v in p.items()}
    d_bias = [torch.zeros(H, device="cuda") for _ in range(M)]
    if row_idx is not None:
        outs = [torch.zeros(t.shape[0], H, device="cuda") for t in e]
        kw.update(de_acc=outs, skip_row0=skip_row0)
    else:
        outs = [torch.empty(T, H, dtype=torch.bfloat16, device="cuda") for _ in range(M)]
        kw.update(de=outs)
    ops.embed_multi_bwd(ops.embed_multi_args(
        rows, L, H, e, p["w_att"], p["b_att"], p["pos"], p["role"], p["ln_g"], p["ln_b"], eps, drop, seed, 0, dx=dx,
        dx_b=dx_b, d_w_att=grads["w_att"], d_b_att=grads["b_att"], d_pos=grads["pos"], d_role=grads["role"],
        d_ln_g=grads["ln_g"], d_ln_b=grads["ln_b"], d_bias=d_bias, **kw))
    torch.cuda.synchronize()
    return x, outs, grads, d_bias


@pytest.mark.parametrize("M", [1, 3, 4])
@pytest.mark.parametrize("H", [32, 64, 128, 768])
@pytest.mark.parametrize("mode", ["tokens", "table"])
def test_fusion_kernels_match_torch(M, H, mode):
    rows, L, eps = 53, 6, 1e-12            # T = 318 tokens: not a multiple of any CTA's tokens
    table_rows = 41 if mode == "table" else 0
    e, p, row_idx, dx, dx_b = _fusion_inputs(M, H, rows, L, table_rows, seed=M * 1000 + H)
    if mode == "tokens":
        dx_b = None
    x, outs, grads, d_bias = _run_kernels(e, p, row_idx, dx, dx_b, rows, L, H, eps, skip_row0=int(mode == "table"))

    ef = [t.float().requires_grad_(True) for t in e]
    pf = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    y = _torch_fusion(ef, pf, row_idx, L, eps)
    dy = dx.float() + (dx_b.float() if dx_b is not None else 0.0)
    y.backward(dy)

    assert float((x.float() - y.detach()).abs().max()) < 2e-2 * float(y.detach().abs().max())
    for m in range(M):
        want = ef[m].grad
        if mode == "table":
            assert torch.count_nonzero(outs[m][0]) == 0, "skip_row0: the <pad> row's gradient is never accumulated"
            assert _rel(outs[m][1:], want[1:]) < 1e-2, m
        else:
            assert _rel(outs[m], want) < 1e-2, m
        assert _rel(d_bias[m], want.sum(0)) < 1e-2, m
    for k in ("pos", "role", "ln_g", "ln_b"):
        assert _rel(grads[k], pf[k].grad) < 1e-2, k
    if M == 1:
        assert torch.count_nonzero(grads["w_att"]) == 0 and torch.count_nonzero(grads["b_att"]) == 0
    else:
        assert _rel(grads["w_att"], pf["w_att"].grad) < 1e-2
        assert _rel(grads["b_att"], pf["b_att"].grad) < 1e-2


@pytest.mark.parametrize("H", [64, 128])
def test_dropout_mask_is_the_two_modality_mask(H):
    """Same seed and site: the zero pattern at M = 3 is the one of the M = 2 kernel, and backward applies it."""
    from pmgt_b200 import ops
    rows, L, eps, drop, seed = 61, 6, 1e-12, 0.3, 0x1234ABCD5678
    e, p, _, dx, _ = _fusion_inputs(3, H, rows, L, 0, seed=H)
    x3, outs, grads, d_bias = _run_kernels(e, p, None, dx, None, rows, L, H, eps, drop=drop, seed=seed)
    p2 = dict(p, w_att=p["w_att"][:2, : 2 * H].contiguous(), b_att=p["b_att"][:2].contiguous())
    x2 = torch.empty_like(x3)
    ops.embed_fuse_fwd(ops.embed_args(rows, L, H, e[0], e[1], p2["w_att"], p2["b_att"], p["pos"], p["role"], p["ln_g"],
                                      p["ln_b"], eps, drop, seed, 0, x_out=x2))
    torch.cuda.synchronize()
    keep = x3 != 0
    assert torch.equal(keep, x2 != 0)
    assert 0.2 < 1 - float(keep.float().mean()) < 0.4
    ef = [t.float().requires_grad_(True) for t in e]
    pf = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    y = _torch_fusion(ef, pf, None, L, eps, keep=keep.float(), scale=1 / (1 - drop))
    assert float((x3.float() - y.detach()).abs().max()) < 2e-2 * float(y.detach().abs().max())
    y.backward(dx.float())
    for m in range(3):
        assert _rel(outs[m], ef[m].grad) < 1e-2
    assert _rel(grads["w_att"], pf["w_att"].grad) < 1e-2 and _rel(grads["ln_g"], pf["ln_g"].grad) < 1e-2


# ---------------------------------------------------------------------------------------------------------------------
# whole pre-training step against the fp32 oracle
# ---------------------------------------------------------------------------------------------------------------------
def _build(cfg, node_size, sd):
    from pmgt_b200 import PMGT, PMGTConfig
    n = len(cfg["feat_hidden_sizes"])
    c = PMGTConfig(hidden_size=cfg["hidden_size"], feat_hidden_sizes=cfg["feat_hidden_sizes"],
                   num_hidden_layers=cfg["num_hidden_layers"], num_attention_heads=cfg["num_attention_heads"],
                   intermediate_size=cfg["intermediate_size"], beta=cfg["beta"], hidden_dropout_prob=0.0,
                   attention_probs_dropout_prob=0.0)
    net = PMGT(node_size, cfg["random_node_ratio"], cfg["mask_node_ratio"], c,
               feat_init_emb=[sd[f"feat_embeddings.{m}.weight"].cpu().numpy() for m in range(n)])
    missing, unexpected = net.load_state_dict({k: v.cpu() for k, v in sd.items()}, strict=False)
    assert not unexpected, unexpected
    assert all(k.endswith(("position_ids", "role_ids")) for k in missing), missing
    return net.cuda()


def _check_grads(net, ref_grads, cos_min=0.995, norm_tol=0.05):
    for name, p in net.named_parameters():
        if not p.requires_grad:
            continue
        assert p.grad is not None, name
        want = ref_grads[name].to(p.grad.device).float()
        got = p.grad.float()
        assert torch.isfinite(got).all(), name
        wn = float(want.norm())
        if wn < 1e-6:
            assert float(got.norm()) < 1e-4, (name, float(got.norm()))
            continue
        cos = float((got * want).sum() / (got.norm() * want.norm()).clamp_min(1e-20))
        assert cos >= cos_min, f"{name}: cosine {cos:.5f}"
        assert abs(float(got.norm()) / wn - 1) <= norm_tol, f"{name}: norm ratio {float(got.norm()) / wn:.4f}"


@pytest.mark.parametrize("over,B,P,L,node_size", [
    (dict(feat_hidden_sizes=[1536]), 64, 10, 6, 500),
    (dict(feat_hidden_sizes=[1536, 768, 512]), 64, 10, 6, 500),                    # 512: TMA gather projection
    (dict(hidden_size=64, num_hidden_layers=2, num_attention_heads=4, intermediate_size=64,
          feat_hidden_sizes=[128, 64, 200]), 16, 10, 6, 200),                      # multihead; 200: general GEMM
    (dict(hidden_size=256, num_hidden_layers=2, num_attention_heads=4, intermediate_size=512,
          feat_hidden_sizes=[256, 128, 96], mask_node_ratio=0.3), 8, 4, 33, 120),  # wide-style: L = 33
    (dict(feat_hidden_sizes=[1536, 768, 512, 200]), 32, 10, 6, 300),
])
@pytest.mark.parametrize("projection", ["gather", "table"])
def test_pretrain_step_matches_oracle(over, B, P, L, node_size, projection, monkeypatch):
    from pmgt_b200 import modeling_pmgt
    monkeypatch.setattr(modeling_pmgt, "PROJECTION_MODE", projection)
    cfg = model_ref.default_cfg(**over)
    n = len(cfg["feat_hidden_sizes"])
    sd = model_ref.init_state_dict(cfg, node_size, seed=21, perturb=0.05)
    net = _build(cfg, node_size, sd)
    net.train()
    gen = torch.Generator().manual_seed(B + L + n)

    def ctx(rows):
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
    for m in range(n):  # the oracle sees the same bf16-rounded feature rows the kernels gather
        sdc[f"feat_embeddings.{m}.weight"] = sdc[f"feat_embeddings.{m}.weight"].to(torch.bfloat16).float()
    params = {k: v.requires_grad_(True) for k, v in sdc.items() if not k.startswith("feat_embeddings")}
    ref = pretrain_forward(sdc, cfg, node_size, target, pair, num_pairs, labels, training=True, masked=masked)
    ref["loss"].backward()
    assert abs(float(out.loss) - float(ref["loss"])) <= 2e-2 * abs(float(ref["loss"]))
    assert float((out.prediction_logits - ref["prediction_logits"]).abs().max()) < 3e-2
    rh = ref["last_hidden_state"].detach()
    assert float((out.last_hidden_state - rh).abs().max()) < 3e-2 * float(rh.abs().max())
    _check_grads(net, {k: v.grad for k, v in params.items()})
    if n == 1:
        g = dict(net.named_parameters())
        assert torch.count_nonzero(g["bert.embeddings.attention.1.weight"].grad) == 0
        assert torch.count_nonzero(g["bert.embeddings.attention.1.bias"].grad) == 0


def test_dense_inputs_through_pmgt_model():
    """PMGTModel.forward(*input_feat_embeds) with three dense inputs matches oracle.encode, and refuses two."""
    from pmgt_b200 import PMGTConfig
    from pmgt_b200.modeling_pmgt import PMGTModel
    cfg = model_ref.default_cfg(num_hidden_layers=2, feat_hidden_sizes=[256, 128, 384])
    sd = model_ref.init_state_dict(cfg, 10, seed=8, perturb=0.05)
    c = PMGTConfig(num_hidden_layers=2, feat_hidden_sizes=cfg["feat_hidden_sizes"], hidden_dropout_prob=0.0,
                   attention_probs_dropout_prob=0.0)
    bert = PMGTModel(c)
    bert.load_state_dict({k[5:]: v for k, v in sd.items() if k.startswith("bert.")}, strict=False)
    bert = bert.cuda().eval()
    g = torch.Generator().manual_seed(0)
    feats = [torch.randn(12, 6, d, generator=g).to(torch.bfloat16).float().cuda() for d in cfg["feat_hidden_sizes"]]
    mask = torch.ones(12, 6, device="cuda")
    with torch.no_grad():
        got = bert(*feats, attention_mask=mask).last_hidden_state
        want = model_ref.encode({k: v.cuda() for k, v in sd.items()}, feats, mask, cfg)
    assert float((got - want).abs().max()) < 3e-2 * float(want.abs().max())
    with pytest.raises(AssertionError):
        bert(*feats[:2], attention_mask=mask)


# ---------------------------------------------------------------------------------------------------------------------
# launch plans and the trainer
# ---------------------------------------------------------------------------------------------------------------------
def _trainer_args(tmp_path, **over):
    from pmgt_b200 import trainer
    kw = dict(synthetic=(400, 3000), train_batch_size=64, test_batch_size=128, num_epochs=1, num_hidden_layers=2, seed=3,
              log_dir=str(tmp_path), lr=2e-3, early=5)
    kw.update(over)
    return trainer.make_args(**kw)


def _three_modality_model(args, seed=11):
    from pmgt_b200 import synthetic, trainer
    trainer.init_run(args)
    trainer.init_dataloader(args)
    args.feat_init_emb = synthetic.make_features(len(args.graph), dims=(1536, 768, 512), seed=seed)
    trainer.init_model(args)
    assert args.model.config.feat_hidden_sizes == [1536, 768, 512]


@pytest.mark.parametrize("projection", ["gather", "table"])
def test_launch_plans_at_three_modalities(tmp_path, projection, monkeypatch):
    from pmgt_b200 import modeling_pmgt, trainer
    monkeypatch.setattr(modeling_pmgt, "PROJECTION_MODE", projection)
    results = []
    for planned in (True, False):
        if not planned:
            monkeypatch.setattr(modeling_pmgt.PMGTModel, "_plan_for", lambda self, *a, **k: None)
        args = _trainer_args(tmp_path)
        _three_modality_model(args)
        modeling_pmgt._seed_counter[0] = 0
        tm = trainer.PMGTTrainerModel(args)
        ds = args.train_dataset
        losses = [float(tm.train_on_indices(ds, np.arange(s, s + 64), 0)) for s in (0, 64)]
        torch.cuda.synchronize()
        if planned:
            assert tm.net.bert._plans, "the launch plan was not used"
        trained = [p for p in tm.net.parameters() if p.requires_grad]
        results.append((losses, [p.detach().clone() for p in trained], [p.grad.clone() for p in trained]))
    (l0, p0, g0), (l1, p1, g1) = results
    for a, b in zip(l0, l1):  # the second loss already depends on the first update
        assert abs(a - b) <= 1e-5 * abs(a), (l0, l1)
    # Gradient sums use fp32 atomics, so the two paths agree to rounding, not bit for bit; AdamW's normalised update
    # turns a rounding difference of a near-zero gradient into up to one step of size lr per element (README), so
    # parameters are bounded by that, and the last step's gradients are compared by direction.
    lr = 2e-3
    for a, b in zip(p0, p1):
        assert float((a - b).abs().max()) <= 2 * lr * len(l0)
    for a, b in zip(g0, g1):  # near-zero gradients (reference norm < 1e-6) are rounding noise: checked absolutely
        if float(a.norm()) < 1e-6:
            assert float(b.norm()) < 1e-4
        else:
            assert float((a * b).sum() / (a.norm() * b.norm())) >= 0.99


def test_trainer_end_to_end_at_three_modalities(tmp_path):
    from pmgt_b200 import PMGTDataset, trainer
    args = _trainer_args(tmp_path, num_epochs=2)
    _three_modality_model(args)
    best, tm = trainer.train(args)
    assert len(args.history) == 2
    for h in args.history:
        assert np.isfinite(h["loss/train"]) and np.isfinite(h["loss/val"])
    # checkpoint round trip into a fresh three-modality model
    ckpt = torch.load(args.best_model_path, map_location="cpu", weights_only=False)
    assert "net.bert.embeddings.feat_linear.2.weight" in ckpt["state_dict"]
    args2 = _trainer_args(tmp_path)
    _three_modality_model(args2)
    tm2 = trainer.PMGTTrainerModel(args2)
    tm2.load_state_dict(ckpt)
    tm.load_state_dict(ckpt)
    for (n1, a), (n2, b) in zip(tm.net.state_dict().items(), tm2.net.state_dict().items()):
        if not n1.startswith("feat_embeddings"):
            assert n1 == n2 and torch.equal(a.cpu(), b.cpu()), n1
    a, b = tm.evaluate(args.valid_dataset, 128), tm2.evaluate(args2.valid_dataset, 128)
    assert abs(a["loss"] - b["loss"]) <= 1e-5 * abs(a["loss"]) + 1e-6
    # bulk inference agrees with item_embeddings
    emb = trainer.inference(args)
    n = len(args.graph)
    assert emb.shape == (n, args.hidden_size) and np.isfinite(emb).all()
    ds = PMGTDataset(args.graph, is_training=False, is_inference=True, seed=args.seed)
    args.model.eval()
    direct = args.model.item_embeddings(ds.sample_batch(np.array([0, 7, n - 1]))).cpu().numpy()
    assert np.allclose(direct, emb[[0, 7, n - 1]], rtol=0, atol=1e-5)
