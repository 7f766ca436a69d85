"""Generates the committed golden vectors from the UNMODIFIED reference.

Needs a checkout of the upstream reference (uoo723/PMGT):

    PMGT_REFERENCE_ROOT=<checkout> python tests/golden/make_golden.py

Outputs (small, committed):
  tests/golden/model_golden.pt        reference PMGT.forward/backward outputs for two
                                      configurations; weights come from the seeded
                                      recipe oracle.model_ref.init_state_dict so only
                                      inputs and outputs are stored
  tests/golden/sampler_ref_golden.npz reference PMGTDataset / pmgt_collate_fn outputs
                                      under a fixed np.random seed on a seeded graph
  tests/golden/adamw_golden.pt        three steps of the reference DenseSparseAdamW
"""
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))
warnings.filterwarnings("ignore")

from oracle import model_ref, ref_shim  # noqa: E402

MODEL_CASES = {
    # name: (cfg overrides, node_size, B, P, L)
    "default": (dict(), 60, 4, 10, 6),
    "multihead": (dict(hidden_size=64, feat_hidden_sizes=[128, 64], num_hidden_layers=2, num_attention_heads=4,
                       intermediate_size=96, beta=0.3, mask_node_ratio=0.4, random_node_ratio=0.1), 40, 3, 4, 9),
}


def make_inputs(node_size, B, P, L, seed):
    g = torch.Generator().manual_seed(seed)

    def ctx(rows):
        ids = torch.randint(2, node_size + 2, (rows, L), generator=g)
        n_real = torch.randint(1, L, (rows,), generator=g)  # at least one real neighbour
        mask = (torch.arange(L)[None, :] <= n_real[:, None]).float()
        ids = ids * mask.long()
        return {"node_ids": ids, "attention_mask": mask}

    target = ctx(B)
    pair = ctx(B * P)
    num_pairs = torch.full((B,), P, dtype=torch.long)
    labels = (torch.rand(B * P, generator=g) < 0.5).float()
    return target, pair, num_pairs, labels


def run_reference_model(R, name):
    over, node_size, B, P, L = MODEL_CASES[name]
    cfg = model_ref.default_cfg(**over)
    sd = model_ref.init_state_dict(cfg, node_size, seed=11, perturb=0.05)
    rcfg = R.PMGTConfig(hidden_size=cfg["hidden_size"], feat_hidden_sizes=cfg["feat_hidden_sizes"],
                        num_hidden_layers=cfg["num_hidden_layers"], num_attention_heads=cfg["num_attention_heads"],
                        intermediate_size=cfg["intermediate_size"], beta=cfg["beta"],
                        hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    net = R.PMGT(node_size, cfg["random_node_ratio"], cfg["mask_node_ratio"], rcfg,
                 feat_init_emb=[sd[f"feat_embeddings.{m}.weight"].numpy() for m in range(2)])
    missing, unexpected = net.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.endswith(("position_ids", "role_ids")) for k in missing), (missing, unexpected)
    net.train()
    target, pair, num_pairs, labels = make_inputs(node_size, B, P, L, seed=5)
    torch.manual_seed(123)  # drives the NFR corruption inside PMGT.forward
    out = net(target, pair, num_pairs, labels)
    out.loss.backward()
    grads = {k: p.grad.clone() for k, p in net.named_parameters() if p.requires_grad}
    # recover the corruption the reference drew (same RNG order)
    torch.manual_seed(123)
    m_ids, m_mask, target_idx = model_ref.mask_nodes(target["node_ids"], node_size, cfg["random_node_ratio"],
                                                     cfg["mask_node_ratio"])
    net.eval()
    with torch.no_grad():
        inf = net(target)[0]
    small = [k for k in grads if grads[k].numel() <= 4096]
    return {
        "cfg": cfg, "node_size": node_size, "weights_seed": 11, "weights_perturb": 0.05,
        "weights_checksum": float(sum(v.double().sum() for k, v in sd.items())),
        "target": target, "pair": pair, "num_pairs": num_pairs, "labels": labels,
        "torch_seed": 123, "masked_ids": m_ids, "masked_mask": m_mask, "masked_target_idx": target_idx,
        "loss": out.loss.detach(), "prediction_logits": out.prediction_logits.detach(),
        "last_hidden_state": out.last_hidden_state.detach(),
        "inference_last_hidden_state": inf,
        "grad_norms": {k: float(g.norm()) for k, g in grads.items()},
        "grads_small": {k: grads[k] for k in small},
        "grad_feat_linear0_rows": grads["bert.embeddings.feat_linear.0.weight"][:4].clone(),
        "grad_query0_rows": grads["bert.encoder.layer.0.attention.self.query.weight"][:4].clone(),
        "n_trainable": len(grads),
    }


def run_reference_sampler(R):
    import networkx as nx

    rng = np.random.default_rng(3)
    n = 40
    g = nx.Graph()
    edges = set()
    for u in range(n):  # ring keeps every node non-isolated
        edges.add((u, (u + 1) % n))
    while len(edges) < 140:
        u, v = rng.integers(0, n, 2)
        if u != v and (v, u) not in edges:
            edges.add((int(u), int(v)))
    edges = sorted(edges)
    perm = rng.permutation(len(edges))
    w = rng.uniform(0.2, 2.0, len(edges))
    g.add_nodes_from(range(2, n + 2))
    for i in perm:
        u, v = edges[i]
        g.add_edge(u + 2, v + 2, weight=float(w[i]))
    src = np.asarray([edges[i][0] + 2 for i in perm])
    dst = np.asarray([edges[i][1] + 2 for i in perm])
    ww = np.asarray([w[i] for i in perm], dtype=np.float64)

    out = {"num_nodes": n, "src": src, "dst": dst, "weight": ww}
    for mode, kw in {"train": dict(), "valid": dict(is_training=False),
                     "infer": dict(is_training=False, is_inference=True)}.items():
        ds = R.PMGTDataset(g, max_ctx_neigh=5, hop_sampling_sizes=[4, 3, 2], **kw)
        np.random.seed(77)
        batch = [ds[i] for i in (0, 7, 19, 33)]
        col = R.pmgt_collate_fn(batch)
        if mode == "infer":
            out[f"{mode}_t_ids"] = col["node_ids"].numpy()
            out[f"{mode}_t_mask"] = col["attention_mask"].numpy()
        else:
            t, p, npairs, lab = col
            out[f"{mode}_t_ids"] = t["node_ids"].numpy()
            out[f"{mode}_t_mask"] = t["attention_mask"].numpy()
            out[f"{mode}_p_ids"] = p["node_ids"].numpy()
            out[f"{mode}_p_mask"] = p["attention_mask"].numpy()
            out[f"{mode}_num_pairs"] = npairs.numpy()
            out[f"{mode}_labels"] = lab.numpy()
    return out


def run_reference_adamw(R):
    g = torch.Generator().manual_seed(2)
    p0 = torch.randn(37, generator=g)
    grads = [torch.randn(37, generator=g) for _ in range(3)]
    p = torch.nn.Parameter(p0.clone())
    opt = R.DenseSparseAdamW([{"params": [p], "weight_decay": 1e-2, "lr": 1e-3}])
    traj = []
    for gr in grads:
        p.grad = gr.clone()
        opt.step()
        traj.append(p.detach().clone())
    return {"p0": p0, "grads": grads, "traj": traj, "lr": 1e-3, "weight_decay": 1e-2}


def main():
    R = ref_shim.load()
    model = {name: run_reference_model(R, name) for name in MODEL_CASES}
    torch.save(model, os.path.join(HERE, "model_golden.pt"))
    np.savez_compressed(os.path.join(HERE, "sampler_ref_golden.npz"), **run_reference_sampler(R))
    torch.save(run_reference_adamw(R), os.path.join(HERE, "adamw_golden.pt"))
    for f in ("model_golden.pt", "sampler_ref_golden.npz", "adamw_golden.pt"):
        print(f, os.path.getsize(os.path.join(HERE, f)), "bytes")
    for name, m in model.items():
        print(name, "loss", float(m["loss"]), "masked", int(m["masked_mask"].sum()), "trainable", m["n_trainable"])


if __name__ == "__main__":
    main()
