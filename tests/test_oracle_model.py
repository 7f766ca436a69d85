"""Pins oracle/model_ref.py (the fp32 torch restatement) against the golden
vectors generated from the unmodified reference, and -- when PMGT_REFERENCE_ROOT
names a checkout of it -- against the reference itself on fresh inputs."""
import os

import pytest
import torch

from oracle import model_ref, ref_shim


def _load(golden_dir, name):
    return torch.load(os.path.join(golden_dir, "model_golden.pt"), weights_only=False)[name]


def _oracle_run(g):
    cfg = g["cfg"]
    sd = model_ref.init_state_dict(cfg, g["node_size"], seed=g["weights_seed"], perturb=g["weights_perturb"])
    assert abs(float(sum(v.double().sum() for v in sd.values())) - g["weights_checksum"]) < 1e-6 * max(
        1.0, abs(g["weights_checksum"])), "seeded weight recipe drifted"
    params = {k: v.requires_grad_(True) for k, v in sd.items() if not k.startswith("feat_embeddings")}
    sd.update(params)
    out = model_ref.pretrain_forward(
        sd, cfg, g["node_size"], g["target"], g["pair"], g["num_pairs"], g["labels"], training=True,
        masked=(g["masked_ids"], g["masked_mask"], g["masked_target_idx"]))
    out["loss"].backward()
    return sd, params, out


@pytest.mark.parametrize("name", ["default", "multihead"])
def test_oracle_matches_reference_golden(golden_dir, name):
    g = _load(golden_dir, name)
    sd, params, out = _oracle_run(g)
    assert torch.allclose(out["loss"], g["loss"], rtol=1e-5, atol=1e-6)
    assert torch.allclose(out["prediction_logits"], g["prediction_logits"], rtol=1e-4, atol=1e-5)
    assert torch.allclose(out["last_hidden_state"], g["last_hidden_state"], rtol=1e-4, atol=1e-5)
    assert len(params) == g["n_trainable"]
    for k, n in g["grad_norms"].items():
        got = float(params[k].grad.norm())
        assert abs(got - n) <= 1e-4 * max(n, 1e-3) + 1e-7, (k, got, n)
    for k, ref in g["grads_small"].items():
        assert torch.allclose(params[k].grad, ref, rtol=1e-3, atol=1e-6), k
    assert torch.allclose(params["bert.embeddings.feat_linear.0.weight"].grad[:4], g["grad_feat_linear0_rows"],
                          rtol=1e-3, atol=1e-6)


@pytest.mark.parametrize("name", ["default", "multihead"])
def test_oracle_inference_matches_golden(golden_dir, name):
    g = _load(golden_dir, name)
    sd = model_ref.init_state_dict(g["cfg"], g["node_size"], seed=g["weights_seed"], perturb=g["weights_perturb"])
    with torch.no_grad():
        out = model_ref.pretrain_forward(sd, g["cfg"], g["node_size"], g["target"], training=False)
    assert torch.allclose(out["last_hidden_state"], g["inference_last_hidden_state"], rtol=1e-4, atol=1e-5)


def test_mask_nodes_follows_reference_rng_order(golden_dir):
    g = _load(golden_dir, "multihead")
    torch.manual_seed(g["torch_seed"])
    ids, m, tgt = model_ref.mask_nodes(g["target"]["node_ids"], g["node_size"], g["cfg"]["random_node_ratio"],
                                       g["cfg"]["mask_node_ratio"])
    assert torch.equal(ids, g["masked_ids"]) and torch.equal(m, g["masked_mask"]) and torch.equal(tgt, g["masked_target_idx"])


@pytest.mark.parametrize("name", ["default", "multihead"])
def test_oracle_masking_inside_forward_matches_reference_golden(golden_dir, name):
    """The reference drew its NFR corruption inside PMGT.forward under torch.manual_seed(torch_seed); the oracle, left
    to draw it itself under the same seed, reproduces the stored loss and logits."""
    g = _load(golden_dir, name)
    sd = model_ref.init_state_dict(g["cfg"], g["node_size"], seed=g["weights_seed"], perturb=g["weights_perturb"])
    torch.manual_seed(g["torch_seed"])
    with torch.no_grad():
        out = model_ref.pretrain_forward(sd, g["cfg"], g["node_size"], g["target"], g["pair"], g["num_pairs"],
                                         g["labels"], training=True)
    assert torch.allclose(out["loss"], g["loss"], rtol=1e-5, atol=1e-6)
    assert torch.allclose(out["prediction_logits"], g["prediction_logits"], rtol=1e-4, atol=1e-5)


def test_adamw_oracle_matches_reference_golden(golden_dir):
    g = torch.load(os.path.join(golden_dir, "adamw_golden.pt"), weights_only=False)
    p = g["p0"].clone()
    m = torch.zeros_like(p)
    v = torch.zeros_like(p)
    for step, (gr, want) in enumerate(zip(g["grads"], g["traj"]), start=1):
        model_ref.adamw_step(p, gr, m, v, step, lr=g["lr"], weight_decay=g["weight_decay"])
        assert torch.allclose(p, want, rtol=1e-6, atol=1e-7)


@pytest.mark.needs_reference
def test_oracle_matches_live_reference():
    """Fresh inputs, live reference (PMGT_REFERENCE_ROOT)."""
    R = ref_shim.load()
    cfg = model_ref.default_cfg(num_hidden_layers=2, mask_node_ratio=0.5)
    node_size = 30
    sd = model_ref.init_state_dict(cfg, node_size, seed=3, perturb=0.1)
    rcfg = R.PMGTConfig(num_hidden_layers=2, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    net = R.PMGT(node_size, cfg["random_node_ratio"], cfg["mask_node_ratio"], rcfg,
                 feat_init_emb=[sd[f"feat_embeddings.{m}.weight"].numpy() for m in range(2)])
    net.load_state_dict(sd, strict=False)
    net.train()
    g = torch.Generator().manual_seed(9)
    B, P, L = 3, 4, 6
    tgt = {"node_ids": torch.randint(2, node_size + 2, (B, L), generator=g), "attention_mask": torch.ones(B, L)}
    pair = {"node_ids": torch.randint(2, node_size + 2, (B * P, L), generator=g), "attention_mask": torch.ones(B * P, L)}
    pair["attention_mask"][:, -2:] = 0
    pair["node_ids"][:, -2:] = 0
    num_pairs = torch.tensor([4, 4, 4])
    labels = (torch.rand(B * P, generator=g) < 0.5).float()
    torch.manual_seed(1)
    ref = net(tgt, pair, num_pairs, labels)
    torch.manual_seed(1)
    ours = model_ref.pretrain_forward(sd, cfg, node_size, tgt, pair, num_pairs, labels, training=True)
    assert torch.allclose(ours["loss"], ref.loss, rtol=1e-5)
    assert torch.allclose(ours["prediction_logits"], ref.prediction_logits, rtol=1e-4, atol=1e-5)
