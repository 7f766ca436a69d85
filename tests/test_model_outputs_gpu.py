"""Per-layer hidden states and attention maps on the B200: pmgt_attn_maps_fwd against torch fp32 for every attention
family, its dropout mask against the one the attention core applied (read back from the core itself), PMGTModel /
PMGT outputs and their gradients against the fp32 reference of test_model_outputs.py, bit-identical behaviour when
the outputs are requested, and launch plans around such a call."""
import math

import pytest
import torch

from oracle import model_ref
from test_model_outputs import encode_with_outputs

pytestmark = pytest.mark.gpu
BF16 = torch.bfloat16


def _ops():
    from pmgt_b200 import ops
    return ops


def _close(got, want, tol, name=""):
    scale = want.abs().max().clamp_min(1e-6)
    err = float((got.float() - want).abs().max() / scale)
    assert torch.isfinite(got.float()).all(), f"{name}: non-finite"
    assert err < tol, f"{name}: max scaled error {err:.4g} >= {tol}"


# ---------------------------------------------------------------------------------------------------------------------
# the kernel
# ---------------------------------------------------------------------------------------------------------------------
# (L, H, heads) with the family pmgt_attn_core_fwd runs for it
SHAPES = [
    (6, 64, 2), (6, 768, 12), (6, 128, 1),                    # attn_mma, dh 32 / 64 / 128
    (6, 64, 4),                                               # generic, dh 16
    (9, 64, 4), (33, 96, 2),                                  # attn_mid, dh 16 / 48
    (10, 64, 2), (10, 768, 12), (10, 128, 1),                 # attn_reg
    (33, 64, 2), (33, 768, 12), (33, 128, 1),
    (64, 64, 2), (64, 768, 12), (64, 128, 1),
    (65, 64, 2), (65, 768, 12), (65, 128, 1),                 # attn_long
    (100, 64, 2), (100, 768, 12), (100, 128, 1),
    (128, 64, 2), (128, 768, 12), (128, 128, 1),
    (70, 64, 4),                                              # generic, dh 16
    (6, 32, 4), (33, 48, 2),                                  # generic, dh 8 / 24: the scalar maps kernel
]
_IDS = [f"L{L}-H{H}x{h}" for L, H, h in SHAPES]


def _inputs(R, L, H, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    qkvc = (torch.randn(R * L, 4 * H, device="cuda", generator=g) * 0.7).to(BF16)
    mask = torch.ones(R, L, device="cuda")
    for r in range(R):  # ragged padding on the right; row 0 holds the target alone
        n_real = 0 if r == 0 else 1 + (r * 7) % max(L - 1, 1)
        mask[r, n_real + 1:] = 0
    return qkvc, mask


def _torch_maps(qkvc, mask, R, L, H, heads, beta):
    dh = H // heads
    x = qkvc.float()
    q, k, c = [x[:, i * H:(i + 1) * H].view(R, L, heads, dh).permute(0, 2, 1, 3) for i in (0, 1, 3)]
    ext = (1.0 - mask[:, None, None, :]) * -10000.0
    n = torch.linalg.norm(c, dim=-1, keepdim=True)
    s1 = 1.0 - (c @ c.transpose(-1, -2)) / (n @ n.transpose(-1, -2)) + torch.eye(L, device="cuda")
    p1 = torch.softmax(s1 + ext, -1)
    p2 = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(dh) + ext, -1)
    return beta * p1 + (1 - beta) * p2


def _maps(qkvc, mask, R, L, H, heads, beta, p=0.0, seed=0, site=10):
    ops = _ops()
    maps = torch.full((R, heads, L, L), float("nan"), device="cuda")
    ops.attn_maps_fwd(ops.attn_args(R, L, H, heads, beta, qkvc, mask, p, seed, site), maps)
    return maps


def _core(qkvc, mask, R, L, H, heads, beta, p=0.0, seed=0, site=10):
    ops = _ops()
    ctx = torch.empty(R * L, H, device="cuda", dtype=BF16)
    ops.attn_core_fwd(ops.attn_args(R, L, H, heads, beta, qkvc, mask, p, seed, site, ctx=ctx))
    return ctx


def _apply(maps, qkvc, R, L, H, heads):
    """maps @ V in fp32 from the bf16 V, as [R * L, H]"""
    dh = H // heads
    v = qkvc[:, 2 * H:3 * H].float().view(R, L, heads, dh).permute(0, 2, 1, 3)
    return (maps @ v).permute(0, 2, 1, 3).reshape(R * L, H)


def _core_matrix(qkvc, mask, R, L, H, heads, beta, p, seed, site):
    """The matrix the core multiplied V with, read back from the core: V = one-hot rows selecting dh keys at a time,
    so ctx row i holds A[i, c0 .. c0 + dh) (bf16-rounded)."""
    dh = H // heads
    out = torch.empty(R, heads, L, L, device="cuda")
    for c0 in range(0, L, dh):
        q = qkvc.clone()
        v = torch.zeros(R, L, heads, dh, device="cuda")
        j = torch.arange(c0, min(L, c0 + dh), device="cuda")
        v[:, j, :, j - c0] = 1.0
        q[:, 2 * H:3 * H] = v.view(R * L, H).to(BF16)
        ctx = _core(q, mask, R, L, H, heads, beta, p, seed, site).float().view(R, L, heads, dh).permute(0, 2, 1, 3)
        out[..., c0:c0 + len(j)] = ctx[..., :len(j)]
    return out


@pytest.mark.parametrize("beta", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("L,H,heads", SHAPES, ids=_IDS)
def test_maps_match_torch(L, H, heads, beta):
    R = 5
    qkvc, mask = _inputs(R, L, H, seed=L * 31 + H + heads)
    maps = _maps(qkvc, mask, R, L, H, heads, beta)
    want = _torch_maps(qkvc, mask, R, L, H, heads, beta)
    assert torch.isfinite(maps).all()
    assert float((maps - want).abs().max()) < 2e-3
    assert float((maps.sum(-1) - 1).abs().max()) < 1e-4          # eval: every row sums to 1
    assert float(maps[mask[:, None, None, :].expand_as(maps) == 0].abs().max(), ) == 0.0  # padded keys: no weight
    _close(_core(qkvc, mask, R, L, H, heads, beta), _apply(maps, qkvc, R, L, H, heads), 1e-2, "ctx")


@pytest.mark.parametrize("p", [0.1, 0.5])
@pytest.mark.parametrize("beta", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("L,H,heads", SHAPES, ids=_IDS)
def test_maps_carry_the_cores_dropout_mask(L, H, heads, beta, p):
    R = max(4, -(-4096 // (L * L * heads)))   # at least 4096 draws per matrix for the keep-rate bound
    qkvc, mask = _inputs(R, L, H, seed=L * 17 + H)
    seed, site = 0x1234_5678_9ABC_DEF0 + L, 20
    maps = _maps(qkvc, mask, R, L, H, heads, beta, p, seed, site)
    assert torch.isfinite(maps).all()
    ctx = _core(qkvc, mask, R, L, H, heads, beta, p, seed, site)
    _close(ctx, _apply(maps, qkvc, R, L, H, heads), 1e-2, "maps @ V vs ctx")
    core = _core_matrix(qkvc, mask, R, L, H, heads, beta, p, seed, site)
    assert torch.equal(maps == 0, core == 0), f"zero pattern differs at {int(((maps == 0) != (core == 0)).sum())} entries"
    _close(core, maps, 1e-2, "A read back from the core")
    if beta in (0.0, 1.0):  # A is one dropped matrix: its kept share over the real keys is 1 - p
        live = mask[:, None, None, :].expand_as(maps) > 0
        n = int(live.sum())
        rate = float((maps[live] > 0).float().mean())
        assert abs(rate - (1 - p)) <= 5 * math.sqrt(p * (1 - p) / n) + 1e-3, (rate, n)


def test_maps_many_ctas():
    """rows * heads > 65,535 (attn_reg at L = 10, two heads of 32), with dropout."""
    R, L, H, heads = 33_000, 10, 64, 2
    qkvc, mask = _inputs(R, L, H, seed=5)
    maps = _maps(qkvc, mask, R, L, H, heads, 0.5)
    assert float((maps - _torch_maps(qkvc, mask, R, L, H, heads, 0.5)).abs().max()) < 2e-3
    maps = _maps(qkvc, mask, R, L, H, heads, 0.5, 0.1, 99, 30)
    _close(_core(qkvc, mask, R, L, H, heads, 0.5, 0.1, 99, 30), _apply(maps, qkvc, R, L, H, heads), 1e-2, "ctx")


# ---------------------------------------------------------------------------------------------------------------------
# the model against the fp32 reference
# ---------------------------------------------------------------------------------------------------------------------
def _build(cfg, node_size, sd, **over):
    from pmgt_b200 import PMGT, PMGTConfig
    n = len(cfg["feat_hidden_sizes"])
    kw = dict(hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    kw.update(over)
    c = PMGTConfig(hidden_size=cfg["hidden_size"], feat_hidden_sizes=cfg["feat_hidden_sizes"],
                   num_hidden_layers=cfg["num_hidden_layers"], num_attention_heads=cfg["num_attention_heads"],
                   intermediate_size=cfg["intermediate_size"], beta=cfg["beta"],
                   max_position_embeddings=cfg["max_position_embeddings"], **kw)
    net = PMGT(node_size, cfg["random_node_ratio"], cfg["mask_node_ratio"], c,
               feat_init_emb=[sd[f"feat_embeddings.{m}.weight"].cpu().numpy() for m in range(n)])
    missing, unexpected = net.load_state_dict({k: v.cpu() for k, v in sd.items()}, strict=False)
    assert not unexpected, unexpected
    return net.cuda()


def _contexts(rows, L, node_size, gen):
    ids = torch.randint(2, node_size + 2, (rows, L), generator=gen)
    n_real = torch.randint(1, L, (rows,), generator=gen)
    mask = (torch.arange(L)[None, :] <= n_real[:, None]).float()
    return {"node_ids": (ids * mask.long()).cuda(), "attention_mask": mask.cuda()}


def _reference(sd, cfg, target):
    n = len(cfg["feat_hidden_sizes"])
    sdc = {k: v.cuda() for k, v in sd.items()}
    for m in range(n):  # the reference sees the same bf16-rounded feature rows the kernels gather
        sdc[f"feat_embeddings.{m}.weight"] = sdc[f"feat_embeddings.{m}.weight"].to(BF16).float()
    params = {k: v.requires_grad_(True) for k, v in sdc.items() if k.startswith("bert.")}
    feats = model_ref.gather_feats(sdc, target["node_ids"], n)
    hs, att = encode_with_outputs(sdc, feats, target["attention_mask"], cfg)
    return hs, att, params


def _check_grads(net, ref_grads, cos_min=0.995, norm_tol=0.05):
    for name, p in net.named_parameters():
        if not name.startswith("bert."):
            continue
        assert p.grad is not None, name
        want = ref_grads[name].float()
        got = p.grad.float()
        assert torch.isfinite(got).all(), name
        wn = float(want.norm())
        if wn < 1e-6:
            assert float(got.norm()) < 1e-4, (name, float(got.norm()))
            continue
        cos = float((got * want).sum() / (got.norm() * want.norm()).clamp_min(1e-20))
        assert cos >= cos_min, f"{name}: cosine {cos:.5f}"
        assert abs(float(got.norm()) / wn - 1) <= norm_tol, f"{name}: norm ratio {float(got.norm()) / wn:.4f}"


MODELS = {
    "default": (dict(), 32, 6, 300),
    "multihead": (dict(num_attention_heads=4, num_hidden_layers=2), 32, 6, 300),
    "run_pmgt": (dict(hidden_size=32, num_hidden_layers=3, intermediate_size=32, beta=1.0), 32, 6, 200),  # general path
    "wide": (dict(hidden_size=768, num_attention_heads=12, intermediate_size=768, num_hidden_layers=2,
                  feat_hidden_sizes=[256, 128]), 8, 33, 120),
    "L100": (dict(num_hidden_layers=2, num_attention_heads=2), 8, 100, 200),
}


@pytest.mark.parametrize("projection", ["gather", "table"])
@pytest.mark.parametrize("name", list(MODELS))
def test_pmgt_outputs_match_reference(name, projection, monkeypatch):
    from pmgt_b200 import modeling_pmgt
    monkeypatch.setattr(modeling_pmgt, "PROJECTION_MODE", projection)
    over, B, L, node_size = MODELS[name]
    cfg = model_ref.default_cfg(**over)
    n_layers, heads, H = cfg["num_hidden_layers"], cfg["num_attention_heads"], cfg["hidden_size"]
    sd = model_ref.init_state_dict(cfg, node_size, seed=13, perturb=0.05)
    net = _build(cfg, node_size, sd).eval()
    target = _contexts(B, L, node_size, torch.Generator().manual_seed(B + L))
    with torch.no_grad():
        out = net(target, output_hidden_states=True, output_attentions=True)
        hs, att, _ = _reference(sd, cfg, target)
    assert len(out.hidden_states) == n_layers + 1 and len(out.attentions) == n_layers
    assert out.hidden_states[-1] is out.last_hidden_state
    for k, (got, want) in enumerate(zip(out.hidden_states, hs)):
        assert got.shape == (B, L, H) and got.dtype == torch.float32
        _close(got, want, 3e-2, f"hidden_states[{k}]")
    for k, (got, want) in enumerate(zip(out.attentions, att)):
        assert got.shape == (B, heads, L, L) and got.dtype == torch.float32
        _close(got, want, 3e-2, f"attentions[{k}]")
        assert float((got.sum(-1) - 1).abs().max()) < 1e-4

    # PMGTModel.forward on dense inputs, and the tuple form
    bert = net.bert
    feats = [t.to(BF16).float() for t in model_ref.gather_feats({k: v.cuda() for k, v in sd.items()},
                                                                  target["node_ids"], len(cfg["feat_hidden_sizes"]))]
    with torch.no_grad():
        o = bert(*feats, attention_mask=target["attention_mask"], output_hidden_states=True, output_attentions=True)
        t = bert(*feats, attention_mask=target["attention_mask"], output_attentions=True, return_dict=False)
        plain = bert(*feats, attention_mask=target["attention_mask"], return_dict=False)
    for k, want in enumerate(hs):
        _close(o.hidden_states[k], want, 3e-2, f"PMGTModel hidden_states[{k}]")
    for k, want in enumerate(att):
        _close(o.attentions[k], want, 3e-2, f"PMGTModel attentions[{k}]")
    assert len(plain) == 2 and len(t) == 3 and plain[1] is None
    assert isinstance(t[2], tuple) and len(t[2]) == n_layers
    assert torch.equal(t[0], plain[0]) and torch.equal(t[2][0], o.attentions[0])


def test_config_flags_and_tuple_layout():
    over, B, L, node_size = MODELS["multihead"]
    cfg = model_ref.default_cfg(**over)
    sd = model_ref.init_state_dict(cfg, node_size, seed=2)
    net = _build(cfg, node_size, sd, output_hidden_states=True).eval()
    target = _contexts(B, L, node_size, torch.Generator().manual_seed(0))
    with torch.no_grad():
        out = net(target)
        assert out.attentions is None and len(out.hidden_states) == cfg["num_hidden_layers"] + 1
        assert net(target, output_hidden_states=False).hidden_states is None
        tup = net(target, output_attentions=True, return_dict=False)
        assert len(tup) == 6 and tup[0] is None and tup[3] is None
        assert len(tup[4]) == cfg["num_hidden_layers"] + 1 and len(tup[5]) == cfg["num_hidden_layers"]
        assert torch.equal(tup[4][-1], tup[2])


def _pretrain_batch(cfg, B, P, L, node_size, seed):
    gen = torch.Generator().manual_seed(seed)
    target, pair = _contexts(B, L, node_size, gen), _contexts(B * P, L, node_size, gen)
    num_pairs = torch.full((B,), P, dtype=torch.long).cuda()
    labels = (torch.rand(B * P, generator=gen) < 0.5).float().cuda()
    return target, pair, num_pairs, labels


def _same(got, want, rel, name):
    """Equal up to the summation order of the kernels' atomic reductions (loss accumulators, red.add gradient rows),
    which varies from run to run with or without the output flags."""
    err = float((got.float() - want.float()).abs().max())
    assert err <= rel * float(want.float().abs().max()), f"{name}: max difference {err:.3g}"


@pytest.mark.parametrize("name", ["default", "run_pmgt"])
def test_requesting_outputs_changes_nothing(name):
    """Training mode with dropout, same dropout seed and corruption: the forward outputs are bit-identical with and
    without both flags; the loss and every gradient agree up to the order of atomic accumulation, which differs between
    two plain calls as well."""
    from pmgt_b200 import modeling_pmgt
    over, B, L, node_size = MODELS[name]
    cfg = model_ref.default_cfg(**over)
    sd = model_ref.init_state_dict(cfg, node_size, seed=4, perturb=0.05)
    net = _build(cfg, node_size, sd, hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1).train()
    target, pair, num_pairs, labels = _pretrain_batch(cfg, B, 5, L, node_size, 1)
    torch.manual_seed(3)
    masked = net.mask_nodes(target["node_ids"], with_positions=True)
    runs = []
    for flags in (False, True, False):
        modeling_pmgt._seed_counter[0] = 1000
        out = net(target, pair, num_pairs, labels, masked_inputs=masked, output_hidden_states=flags,
                  output_attentions=flags)
        out.loss.backward()
        grads = {n: p.grad.clone() for n, p in net.named_parameters() if p.grad is not None}
        net.zero_grad(set_to_none=True)
        runs.append((out, grads))
    (a, ga), (b, gb), (c, gc) = runs
    for x in (b, c):
        assert torch.equal(x.prediction_logits, a.prediction_logits)
        assert torch.equal(x.last_hidden_state, a.last_hidden_state)
        _same(x.loss, a.loss, 1e-6, "loss")
    for g in (gb, gc):
        assert g.keys() == ga.keys()
        for n in ga:
            _same(g[n], ga[n], 1e-4, n)
    assert a.hidden_states is None and a.attentions is None
    H, heads, n_layers = cfg["hidden_size"], cfg["num_attention_heads"], cfg["num_hidden_layers"]
    assert b.hidden_states[-1] is b.last_hidden_state
    assert all(h.shape == (B, L, H) for h in b.hidden_states) and len(b.hidden_states) == n_layers + 1
    assert all(m.shape == (B, heads, L, L) for m in b.attentions) and len(b.attentions) == n_layers
    # training mode: the maps carry the attention dropout (some entries of real keys are exactly zero)
    live = target["attention_mask"][:, None, None, :].expand_as(b.attentions[0]) > 0
    if cfg["beta"] in (0.0, 1.0):
        assert float((b.attentions[0][live] == 0).float().mean()) > 0.02


@pytest.mark.parametrize("name", ["default", "run_pmgt"])
def test_hidden_state_gradients_match_reference(name):
    over, B, L, node_size = MODELS[name]
    cfg = model_ref.default_cfg(**over)
    n_layers = cfg["num_hidden_layers"]
    sd = model_ref.init_state_dict(cfg, node_size, seed=6, perturb=0.05)
    net = _build(cfg, node_size, sd).train()
    target = _contexts(B, L, node_size, torch.Generator().manual_seed(7))
    for k in sorted({0, n_layers // 2, n_layers}):
        w = torch.randn(B, L, cfg["hidden_size"], generator=torch.Generator().manual_seed(k)).cuda()
        out = net(target, output_hidden_states=True)
        (out.hidden_states[k] * w).mean().backward()
        hs, _, params = _reference(sd, cfg, target)
        (hs[k] * w).mean().backward()
        _check_grads(net, {n: (p.grad if p.grad is not None else torch.zeros_like(p)) for n, p in params.items()})
        net.zero_grad(set_to_none=True)


def test_backward_through_attention_maps_raises():
    over, B, L, node_size = MODELS["multihead"]
    cfg = model_ref.default_cfg(**over)
    sd = model_ref.init_state_dict(cfg, node_size, seed=8)
    net = _build(cfg, node_size, sd).train()
    target = _contexts(B, L, node_size, torch.Generator().manual_seed(8))
    out = net(target, output_attentions=True)
    assert all(m.requires_grad for m in out.attentions)
    with pytest.raises(NotImplementedError, match="not differentiable"):
        (out.attentions[1].sum() + out.last_hidden_state.sum()).backward()
    net.zero_grad(set_to_none=True)
    out = net(target, output_attentions=True)
    out.last_hidden_state.sum().backward()   # the maps themselves stay out of a backward pass that does not reach them
    assert all(p.grad is not None for n, p in net.named_parameters() if n.startswith("bert."))


def test_launch_plans_around_a_flagged_call():
    """With plans on, a call that requests outputs runs unplanned and leaves the plans alone: the next plain call
    replays its plan and matches the plain call before, bit for bit (dropout 0)."""
    over, B, L, node_size = MODELS["default"]
    cfg = model_ref.default_cfg(**over)
    sd = model_ref.init_state_dict(cfg, node_size, seed=9, perturb=0.05)
    net = _build(cfg, node_size, sd).train()
    net.bert.use_launch_plans = True
    target, pair, num_pairs, labels = _pretrain_batch(cfg, B, 5, L, node_size, 2)
    torch.manual_seed(5)
    masked = net.mask_nodes(target["node_ids"], with_positions=True)

    def step(**flags):
        out = net(target, pair, num_pairs, labels, masked_inputs=masked, **flags)
        plan = net.bert._active_plan
        out.loss.backward()
        res = (out.loss.clone(), out.prediction_logits.clone(), out.last_hidden_state.clone(),
               {n: p.grad.clone() for n, p in net.named_parameters() if p.grad is not None}, plan)
        net.zero_grad(set_to_none=True)
        return res

    step()                                  # records the plan
    before = step()                         # replays it
    plan = before[4]
    assert plan is not None and plan.fwd_tape is not None and plan.bwd_tape is not None
    tapes, n_plans = (plan.fwd_tape, plan.bwd_tape), len(net.bert._plans)
    flagged = step(output_hidden_states=True, output_attentions=True)
    assert flagged[4] is None and len(net.bert._plans) == n_plans
    after = step()
    assert after[4] is plan and (plan.fwd_tape, plan.bwd_tape) == tapes
    assert torch.equal(before[1], after[1]) and torch.equal(before[2], after[2])   # logits, last_hidden_state
    _same(after[0], before[0], 1e-6, "loss")   # atomic loss accumulation: see _same
    assert before[3].keys() == after[3].keys()
    for n in before[3]:
        _same(after[3][n], before[3][n], 1e-4, n)
    _same(flagged[0], before[0], 1e-6, "loss of the flagged call")
