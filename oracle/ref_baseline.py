"""TEST / BENCH INFRASTRUCTURE ONLY -- the UNMODIFIED reference's pre-training path timed on the host CPU cores.

Uses the reference's own modules (the checkout named by ``PMGT_REFERENCE_ROOT``, else the byte-for-byte copies
``oracle/build.py::build_ref`` staged under the git-ignored ``oracle/_ref/``) through ``oracle/ref_shim.py`` (transformers
5.x -> 4.11.2 semantics, no edits to the reference code):

  sampler  ``PMGTDataset.__getitem__`` + ``pmgt_collate_fn`` (pmgt/pmgt/datasets.py:82-208) on a weighted ``nx.Graph``,
           inside ``torch.utils.data.DataLoader`` worker PROCESSES, one per core (pmgt/pmgt/trainer.py:90-103);
  model    ``PMGT.forward`` with its per-target pair-encoding loop (pmgt/pmgt/models.py:56-176), autograd backward and
           ``DenseSparseAdamW.step`` with the two parameter groups (pmgt/optimizers.py:169-272, pmgt/base_trainer.py:35-59),
           fp32, ``torch.set_num_threads(all cores)``.

Reported: contexts/s of the sampler alone, of the model step alone (batches pre-materialised) and of both run back to
back (``value``).  ``kind = "reference"``.  Only bench.py may call this (cpu_baseline leg and --impl reference).
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch


def run_cli(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="TG", choices=["VG", "TG"])
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=0)
    ap.add_argument("--batch", type=int, default=256, help="reference default train_batch_size (train.py:34)")
    ap.add_argument("--budget-s", type=float, default=30.0)
    a = ap.parse_args(argv)
    sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
    import networkx as nx

    from oracle import ref_shim
    from pmgt_b200 import synthetic  # synthetic input generators only (numpy)

    from_tree = ref_shim.available()
    ref = ref_shim.load_any()
    cores = os.cpu_count() or 1
    n, src, dst, w = synthetic.make_edge_list(a.workload)
    g = nx.Graph()
    g.add_nodes_from(range(2, n + 2))
    g.add_weighted_edges_from(zip(src.tolist(), dst.tolist(), w.astype(np.float64).tolist()))
    feats = synthetic.make_features(n, seed=synthetic.SHAPES[a.workload][3])
    rng = np.random.default_rng(0)
    train_nodes = np.sort(rng.permutation(np.arange(2, n + 2))[: int(0.8 * n)])
    ds = ref.PMGTDataset(g, train_nodes)
    np.random.seed(0)
    torch.manual_seed(0)

    net = ref.PMGT(node_size=n, config=ref.PMGTConfig(), feat_init_emb=feats)
    no_decay = ["bias", "LayerNorm.weight"]
    named = [(k, p) for k, p in net.named_parameters() if p.requires_grad]
    opt = ref.DenseSparseAdamW([
        {"params": [p for k, p in named if not any(nd in k for nd in no_decay)], "weight_decay": 1e-2},
        {"params": [p for k, p in named if any(nd in k for nd in no_decay)], "weight_decay": 0.0}], lr=1e-3)
    net.train()
    torch.set_num_threads(cores)

    # calibrate the batch so that the requested steps fit the budget (the reference's default is 256)
    t0 = time.perf_counter()
    ds[0]
    per_item_s = time.perf_counter() - t0
    total = a.steps + a.warmup
    B = int(max(16, min(a.batch, a.budget_s / max(total, 1) / max(per_item_s / cores + 0.02, 1e-4))))

    # DataLoader parallelism is ACROSS batches (one worker builds one batch), so steady-state sampler throughput is
    # measured with many small batches in flight -- the reference's own Dataset / collate code in worker processes --
    # and the model batches of B targets are then assembled from them (same tensors a B-sized collate would give).
    workers = min(cores, 16)
    small = 8
    n_small = (B * total + small - 1) // small
    loader = torch.utils.data.DataLoader(ds, batch_size=small, shuffle=True, num_workers=workers,
                                         collate_fn=ref.pmgt_collate_fn, persistent_workers=False)
    it = iter(loader)
    parts = [next(it) for _ in range(min(workers, n_small))]      # worker start-up and first batches: not timed
    t0 = time.perf_counter()
    timed_items = 0
    while len(parts) < n_small + min(workers, n_small):
        try:
            parts.append(next(it))
        except StopIteration:
            break
        timed_items += parts[-1][0]["node_ids"].shape[0]
    t_sample_all = time.perf_counter() - t0
    del it
    sampler_items_per_s = timed_items / max(t_sample_all, 1e-9)

    def assemble(chunk):
        return ({k: torch.cat([c[0][k] for c in chunk]) for k in chunk[0][0]},
                {k: torch.cat([c[1][k] for c in chunk]) for k in chunk[0][1]},
                torch.cat([c[2] for c in chunk]), torch.cat([c[3] for c in chunk]))

    per = B // small
    batches = [assemble(parts[i * per: (i + 1) * per]) for i in range(total) if len(parts[i * per: (i + 1) * per]) == per]
    total = len(batches)
    a.steps = max(1, total - a.warmup)
    B = per * small

    def step(batch):
        opt.zero_grad()
        loss = net(*batch)[0]
        loss.backward()
        opt.step()
        return float(loss)

    for b in batches[: a.warmup]:
        step(b)
    t0 = time.perf_counter()
    ctx = 0
    loss = float("nan")
    for b in batches[a.warmup:]:
        loss = step(b)
        ctx += b[0]["node_ids"].shape[0] + b[1]["node_ids"].shape[0]
    t_model = time.perf_counter() - t0
    t_sample_timed = (ctx / 11.0) / sampler_items_per_s   # time the DataLoader needs for the items of the timed steps
    print(json.dumps({
        "contexts": ctx, "sampler_s": t_sample_timed, "model_s": t_model, "steps": a.steps, "warmup": a.warmup,
        "targets_per_step": B, "cores": cores, "value": ctx / (t_sample_timed + t_model),
        "sampler_contexts_per_s": ctx / t_sample_timed, "model_contexts_per_s": ctx / t_model, "loss_last": loss,
        "ms_per_step": 1e3 * (t_sample_timed + t_model) / a.steps, "kind": "reference",
        "reference_root": ref_shim.REFERENCE_ROOT if from_tree else "oracle/_ref (staged copy of the unmodified modules)",
    }))


if __name__ == "__main__":
    run_cli()
