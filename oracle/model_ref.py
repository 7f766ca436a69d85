"""TEST INFRASTRUCTURE ONLY -- fp32 PyTorch restatement of the PMGT model math.

A functional (no ``nn.Module``) restatement of the reference's pre-training
forward pass, operating on a plain ``dict`` of tensors that uses the
reference's state-dict key names.  Autograd provides the gradients.  Pinned in
``tests/test_oracle_model.py`` against the unmodified reference (when
``PMGT_REFERENCE_ROOT`` names a checkout) and against the committed golden vectors in
``tests/golden/model_golden.pt`` (generated from the unmodified reference by
``tests/golden/make_golden.py``).

Third-party arithmetic restated here (transformers==4.11.2, absent from
the reference tree): BertSelfOutput / BertOutput = dense -> dropout ->
LayerNorm(x + residual); BertIntermediate = dense -> erf-GELU;
get_extended_attention_mask = (1 - mask)[:, None, None, :] * -10000.
"""
import math
from typing import Dict, List, Optional

import torch
import torch.nn.functional as F


def _linear(x, sd, prefix):
    return F.linear(x, sd[prefix + ".weight"], sd[prefix + ".bias"])


def _layer_norm(x, sd, prefix, eps):
    return F.layer_norm(x, (x.shape[-1],), sd[prefix + ".weight"], sd[prefix + ".bias"], eps)


def embeddings(sd: Dict[str, torch.Tensor], feats: List[torch.Tensor], eps: float) -> torch.Tensor:
    """PMGTEmbeddings.forward (modeling_pmgt.py:189-210), dropout = identity."""
    p = "bert.embeddings."
    L = feats[0].shape[1]
    e = [_linear(f, sd, f"{p}feat_linear.{m}") for m, f in enumerate(feats)]
    att = torch.softmax(_linear(torch.tanh(torch.cat(e, dim=-1)), sd, p + "attention.1"), dim=-1)
    fused = sum(att[..., m: m + 1] * e[m] for m in range(len(e)))
    pos = sd[p + "position_embeddings.weight"][:L]
    role_ids = torch.tensor([0] + [1] * (L - 1), device=fused.device)
    role = sd[p + "role_embeddings.weight"][role_ids]
    return _layer_norm(fused + pos + role, sd, p + "LayerNorm", eps)


def self_attention(sd, prefix, x, ext_mask, heads: int, beta: float) -> torch.Tensor:
    """PMGTSelfAttention.forward (modeling_pmgt.py:420-534), absolute positions, dropout = identity."""
    R, L, H = x.shape
    dh = H // heads

    def split(t):
        return t.view(R, L, heads, dh).permute(0, 2, 1, 3)

    q = split(_linear(x, sd, prefix + "query"))
    k = split(_linear(x, sd, prefix + "key"))
    v = split(_linear(x, sd, prefix + "value"))
    c = split(_linear(x, sd, prefix + "ctx_attention"))
    n = torch.linalg.norm(c, dim=-1, keepdim=True)
    s1 = 1.0 - (c @ c.transpose(-1, -2)) / (n @ n.transpose(-1, -2)) + torch.eye(L, device=x.device, dtype=x.dtype)
    p1 = torch.softmax(s1 + ext_mask, dim=-1)
    s2 = (q @ k.transpose(-1, -2)) / math.sqrt(dh)
    p2 = torch.softmax(s2 + ext_mask, dim=-1)
    ctx = (beta * p1 + (1.0 - beta) * p2) @ v
    return ctx.permute(0, 2, 1, 3).reshape(R, L, H)


def layer(sd, i: int, x, ext_mask, heads: int, beta: float, eps: float) -> torch.Tensor:
    """PMGTLayer.forward (modeling_pmgt.py:296-325)."""
    p = f"bert.encoder.layer.{i}."
    ctx = self_attention(sd, p + "attention.self.", x, ext_mask, heads, beta)
    a = _layer_norm(_linear(ctx, sd, p + "attention.output.dense") + x, sd, p + "attention.output.LayerNorm", eps)
    h = F.gelu(_linear(a, sd, p + "intermediate.dense"))
    return _layer_norm(_linear(h, sd, p + "output.dense") + a, sd, p + "output.LayerNorm", eps)


def encode(sd, feats: List[torch.Tensor], attention_mask: torch.Tensor, cfg) -> torch.Tensor:
    """PMGTModel.forward (modeling_pmgt.py:80-152) -> last_hidden_state."""
    ext = (1.0 - attention_mask[:, None, None, :].to(feats[0].dtype)) * -10000.0
    x = embeddings(sd, feats, cfg["layer_norm_eps"])
    for i in range(cfg["num_hidden_layers"]):
        x = layer(sd, i, x, ext, cfg["num_attention_heads"], cfg["beta"], cfg["layer_norm_eps"])
    return x


def gather_feats(sd, node_ids: torch.Tensor, n_modal: int = 2) -> List[torch.Tensor]:
    """get_input_feat_embeds (pmgt/pmgt/utils.py:43-50)."""
    return [sd[f"feat_embeddings.{m}.weight"][node_ids] for m in range(n_modal)]


def gsr_loss(pair_h0, tgt_h0, labels):
    """PMGTGraphConstructLoss (modeling_pmgt.py:543-546) for one target."""
    logits = F.normalize(pair_h0, dim=-1) @ F.normalize(tgt_h0, dim=-1)
    return F.binary_cross_entropy_with_logits(logits, labels), logits


def nfr_loss(sd, h_masked, targets: List[torch.Tensor]):
    """PMGTNodeConstructLoss (modeling_pmgt.py:566-569)."""
    losses = [F.mse_loss(_linear(h_masked, sd, f"nfr_loss.projections.{m}"), t) for m, t in enumerate(targets)]
    return torch.stack(losses).mean()


def mask_nodes(node_ids: torch.Tensor, node_size: int, random_ratio: float, mask_ratio: float):
    """The NFR corruption of PMGT.forward (models.py:131-151), consuming torch's
    global RNG in the same order: rand, randint(#replaced), rand."""
    ids = node_ids.clone()
    dev = ids.device
    rand = torch.rand(ids.shape[0], ids.shape[1] - 1, device=dev)
    m = (rand < random_ratio) * (ids[:, 1:] != 0)
    ids[:, 1:][m] = torch.randint(2, node_size + 2, (int(m.sum()),), device=dev)
    rand = torch.rand(ids.shape[0], ids.shape[1] - 1, device=dev)
    m = (rand < mask_ratio) * (ids[:, 1:] != 0)
    target_idx = ids[:, 1:][m]
    ids[:, 1:][m] = 1
    return ids, m, target_idx


def pretrain_forward(sd, cfg, node_size, target_inputs, pair_inputs=None, num_pairs=None, labels=None,
                     training=True, masked: Optional[tuple] = None):
    """PMGT.forward (models.py:56-176).  Returns dict(loss, prediction_logits,
    last_hidden_state, gsr, nfr).  ``masked`` = (masked_ids, mask, target_idx)
    overrides the random corruption (for deterministic comparisons)."""
    t_ids, t_mask = target_inputs["node_ids"], target_inputs["attention_mask"]
    h_t = encode(sd, gather_feats(sd, t_ids), t_mask, cfg)
    out = {"last_hidden_state": h_t, "loss": None, "prediction_logits": None}
    if pair_inputs is None:
        return out
    # models.py:111-124 runs one encoder call per target; the math per row is
    # independent of batching, so one batched call is an exact restatement.
    h_p = encode(sd, gather_feats(sd, pair_inputs["node_ids"]), pair_inputs["attention_mask"], cfg)
    losses, logits = [], []
    bs = 0
    for i, n in enumerate(num_pairs.tolist()):
        l, lg = gsr_loss(h_p[bs: bs + n, 0], h_t[i, 0], labels[bs: bs + n])
        losses.append(l)
        logits.append(lg)
        bs += n
    gsr = torch.stack(losses).mean()
    out["prediction_logits"] = torch.cat(logits)
    nfr = torch.zeros((), dtype=gsr.dtype, device=gsr.device)
    if training:
        if masked is None:
            masked = mask_nodes(t_ids, node_size, cfg["random_node_ratio"], cfg["mask_node_ratio"])
        m_ids, m_mask, target_idx = masked
        h_m = encode(sd, gather_feats(sd, m_ids), t_mask, cfg)
        nfr = nfr_loss(sd, h_m[:, 1:][m_mask], gather_feats(sd, target_idx))
    out.update(loss=gsr + nfr, gsr=gsr, nfr=nfr)
    return out


def adamw_step(p, g, m, v, step, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2):
    """Dense branch of DenseSparseAdamW.step (pmgt/optimizers.py:256-270), in place."""
    b1, b2 = betas
    p.mul_(1 - lr * weight_decay)
    m.mul_(b1).add_(g, alpha=1 - b1)
    v.mul_(b2).addcmul_(g, g, value=1 - b2)
    denom = (v.sqrt() / math.sqrt(1 - b2 ** step)).add_(eps)
    p.addcdiv_(m, denom, value=-(lr / (1 - b1 ** step)))


def default_cfg(**over):
    cfg = dict(hidden_size=128, feat_hidden_sizes=[1536, 768], num_hidden_layers=5, num_attention_heads=1,
               intermediate_size=128, layer_norm_eps=1e-12, beta=0.5, max_position_embeddings=100,
               initializer_range=0.02, random_node_ratio=0.02, mask_node_ratio=0.16)
    cfg.update(over)
    return cfg


def init_state_dict(cfg, node_size: int, feats: Optional[List[torch.Tensor]] = None, seed: int = 0,
                    device="cpu", dtype=torch.float32, perturb: float = 0.0):
    """Random weights with the reference's key names / shapes (N(0, 0.02) for
    ``bert.*`` like ``_init_weights``, modeling_pmgt.py:44-58).  ``perturb`` adds
    noise to biases / LayerNorm so gradient tests are not run at the trivial point."""
    g = torch.Generator().manual_seed(seed)
    H, I = cfg["hidden_size"], cfg["intermediate_size"]
    std = cfg["initializer_range"]
    sd = {}

    def lin(name, out_f, in_f, s=std):
        sd[name + ".weight"] = torch.randn(out_f, in_f, generator=g) * s
        sd[name + ".bias"] = torch.randn(out_f, generator=g) * perturb

    def ln(name):
        sd[name + ".weight"] = 1.0 + torch.randn(H, generator=g) * perturb
        sd[name + ".bias"] = torch.randn(H, generator=g) * perturb

    e = "bert.embeddings."
    sd[e + "position_embeddings.weight"] = torch.randn(cfg["max_position_embeddings"], H, generator=g) * std
    sd[e + "role_embeddings.weight"] = torch.randn(2, H, generator=g) * std
    for m, d in enumerate(cfg["feat_hidden_sizes"]):
        lin(f"{e}feat_linear.{m}", H, d)
    lin(e + "attention.1", len(cfg["feat_hidden_sizes"]), len(cfg["feat_hidden_sizes"]) * H)
    ln(e + "LayerNorm")
    for i in range(cfg["num_hidden_layers"]):
        p = f"bert.encoder.layer.{i}."
        for n in ("query", "key", "value", "ctx_attention"):
            lin(p + "attention.self." + n, H, H)
        lin(p + "attention.output.dense", H, H)
        ln(p + "attention.output.LayerNorm")
        lin(p + "intermediate.dense", I, H)
        lin(p + "output.dense", H, I)
        ln(p + "output.LayerNorm")
    for m, d in enumerate(cfg["feat_hidden_sizes"]):
        lin(f"nfr_loss.projections.{m}", d, H, s=1.0 / math.sqrt(H))
    for m, d in enumerate(cfg["feat_hidden_sizes"]):
        if feats is not None:
            sd[f"feat_embeddings.{m}.weight"] = feats[m].clone()
        else:
            t = torch.randn(node_size + 2, d, generator=g)
            t[:2] = 0
            sd[f"feat_embeddings.{m}.weight"] = t
    return {k: v.to(device=device, dtype=dtype) for k, v in sd.items()}
