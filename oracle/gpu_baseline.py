"""TEST / BENCH INFRASTRUCTURE ONLY -- the reference's model step run EAGERLY on the GPU (BASELINE.md section 4 item 5,
SURVEY section 2.2: "the bar is beat stock PyTorch eager on the same B200").

The unmodified reference is not part of this repository, so this is the oracle
restatement (``oracle/model_ref.py``, pinned to the reference by the golden vectors) executed the way the reference
executes it (``pmgt/pmgt/models.py:56-176``): fp32 stock PyTorch ops on ``cuda:0``, feature rows gathered with
``nn.Embedding``-style indexing, ONE encoder call for the targets, then the reference's Python loop over targets with a
device->host sync (``num.item()``, models.py:112) and one encoder call per target's pair group (models.py:111-124), one
encoder call for the masked targets, autograd backward, and the per-parameter ``DenseSparseAdamW`` dense branch
(``pmgt/optimizers.py:256-270``: ~8 launches per tensor x 104 tensors).  Batches are pre-materialised with the CPU port of
the reference sampler outside the timed region, so this number is the MODEL step only -- optimistic for the reference,
whose DataLoader workers (~105 ms per item per core) would starve the GPU long before.

None of pmgt_b200's kernels run here.  Only bench.py may call this (``gpu_baseline`` leg and ``--impl reference-gpu``).
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

from . import model_ref


def eager_step(sd, params, m_state, v_state, cfg, node_size, batch, step_no, loop=True):
    """One reference-style training step on the GPU; returns the loss tensor (no sync)."""
    t, p, n, lab = batch
    for prm in params.values():
        prm.grad = None
    h_t = model_ref.encode(sd, model_ref.gather_feats(sd, t["node_ids"]), t["attention_mask"], cfg)
    losses = []
    bs = 0
    if loop:
        for i, num in enumerate(n):
            k = int(num.item())  # the reference's per-target host sync (models.py:112)
            h_p = model_ref.encode(sd, model_ref.gather_feats(sd, p["node_ids"][bs: bs + k]),
                                   p["attention_mask"][bs: bs + k], cfg)
            l, _ = model_ref.gsr_loss(h_p[:, 0], h_t[i, 0], lab[bs: bs + k])
            losses.append(l)
            bs += k
    else:  # one batched pair encode (what a careful user of the reference would write)
        h_p = model_ref.encode(sd, model_ref.gather_feats(sd, p["node_ids"]), p["attention_mask"], cfg)
        for i, k in enumerate(n.tolist()):
            l, _ = model_ref.gsr_loss(h_p[bs: bs + k, 0], h_t[i, 0], lab[bs: bs + k])
            losses.append(l)
            bs += k
    gsr = torch.stack(losses).mean()
    m_ids, m_mask, target_idx = model_ref.mask_nodes(t["node_ids"], node_size, cfg["random_node_ratio"], cfg["mask_node_ratio"])
    h_m = model_ref.encode(sd, model_ref.gather_feats(sd, m_ids), t["attention_mask"], cfg)
    nfr = model_ref.nfr_loss(sd, h_m[:, 1:][m_mask], model_ref.gather_feats(sd, target_idx))
    loss = gsr + nfr
    loss.backward()
    with torch.no_grad():
        for k, prm in params.items():
            if prm.grad is None:
                continue
            wd = 0.0 if ("bias" in k or "LayerNorm.weight" in k) else 1e-2
            model_ref.adamw_step(prm, prm.grad, m_state[k], v_state[k], step_no, weight_decay=wd)
    return loss


def run_cli(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="TG", choices=["VG", "TG"])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--batched-pairs", action="store_true", help="one batched pair encode instead of the reference's loop")
    a = ap.parse_args(argv)
    sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
    from pmgt_b200 import synthetic  # synthetic input generators only (numpy); no kernels

    from . import cpu_baseline

    g = synthetic.make_item_graph(a.workload)
    feats = synthetic.make_features(g.num_nodes, seed=synthetic.SHAPES[a.workload][3])
    # batches from the CPU port of the reference sampler, before CUDA is initialised (fork-safe)
    cp = cpu_baseline.CpuPretrainer(g.indptr, g.indices, g.weights.astype(np.float64), g.num_nodes, feats)
    rng = np.random.default_rng(0)
    try:
        batches = [cp.sample(rng.integers(2, g.num_nodes + 2, size=a.batch)) for _ in range(a.steps + a.warmup)]
    finally:
        cp.close()
    del cp
    dev = torch.device("cuda", 0)
    cfg = model_ref.default_cfg()
    sd = model_ref.init_state_dict(cfg, g.num_nodes, feats=[torch.as_tensor(f) for f in feats], seed=0, device=dev)
    params = {k: v.requires_grad_(True) for k, v in sd.items() if not k.startswith("feat_embeddings")}
    m_state = {k: torch.zeros_like(v) for k, v in params.items()}
    v_state = {k: torch.zeros_like(v) for k, v in params.items()}
    to_dev = lambda b: ({k: v.to(dev) for k, v in b[0].items()}, {k: v.to(dev) for k, v in b[1].items()}, b[2].to(dev), b[3].to(dev))
    batches = [to_dev(b) for b in batches]
    step_no = 0
    for b in batches[: a.warmup]:
        step_no += 1
        eager_step(sd, params, m_state, v_state, cfg, g.num_nodes, b, step_no, loop=not a.batched_pairs)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ctx = 0
    loss = None
    for b in batches[a.warmup:]:
        step_no += 1
        loss = eager_step(sd, params, m_state, v_state, cfg, g.num_nodes, b, step_no, loop=not a.batched_pairs)
        ctx += a.batch + int(b[2].sum())
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    print(json.dumps({"value": ctx / dt, "unit": "contexts/s", "ms_per_step": 1e3 * dt / a.steps, "steps": a.steps,
                      "warmup": a.warmup, "targets_per_step": a.batch, "contexts": ctx, "workload": a.workload,
                      "pair_encode": "batched" if a.batched_pairs else "per-target loop (models.py:111-124)",
                      "dtype": "f32", "device": torch.cuda.get_device_name(0), "loss_last": float(loss),
                      "sampler": "excluded (batches pre-materialised by the CPU port)"}))


if __name__ == "__main__":
    run_cli()
