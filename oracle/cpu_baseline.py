"""TEST / BENCH INFRASTRUCTURE ONLY -- the reference's CPU path, timed.

Runs the oracle *port* of the reference's pre-training step on the host cores:
  sampler  oracle.sampler_ref.ref_getitem  (= PMGTDataset.__getitem__, datasets.py:113-183)
           in a process pool, one worker per core (the reference uses DataLoader
           worker processes, trainer.py:90-103), then ref_collate;
  model    oracle.model_ref.pretrain_forward + autograd backward + adamw_step
           (= PMGT.forward, models.py:56-176, DenseSparseAdamW, optimizers.py:256-270),
           fp32, torch.set_num_threads(all cores), with the reference's per-target
           pair-encoding loop replaced by one batched call (an *optimistic* baseline:
           the batched call is ~4.9x faster than the loop on CPU, SURVEY section 6).
The upstream reference is not part of this repository, hence kind = "port".
Only bench.py may call this (cpu_baseline leg and --impl reference).
"""
import multiprocessing as mp
import os
import time

import numpy as np
import torch

from . import model_ref, sampler_ref

_G = {}


def _init_worker(indptr, indices, weights, num_nodes, hops, max_ctx, seed):
    _G.update(indptr=indptr, indices=indices, weights=weights, num_nodes=num_nodes, hops=hops, max_ctx=max_ctx)
    np.random.seed((seed + os.getpid()) % (2 ** 31))
    torch.set_num_threads(1)


def _work(target):
    g = _G
    return sampler_ref.ref_getitem(g["indptr"], g["indices"], g["weights"], g["num_nodes"], int(target),
                                   hops=g["hops"], max_ctx=g["max_ctx"])


class CpuPretrainer:
    """Oracle-port pre-training on the CPU with all host cores."""

    def __init__(self, indptr, indices, weights, num_nodes, feats, cfg=None, hops=(16, 8, 4), max_ctx=5, seed=0,
                 cores=None):
        self.cores = cores or os.cpu_count() or 1
        self.num_nodes = num_nodes
        self.cfg = cfg or model_ref.default_cfg()
        self.pool = mp.get_context("fork").Pool(self.cores, initializer=_init_worker,
                                                initargs=(indptr, indices, weights, num_nodes, tuple(hops), max_ctx, seed))
        torch.set_num_threads(self.cores)
        sd = model_ref.init_state_dict(self.cfg, num_nodes, feats=[torch.as_tensor(f) for f in feats], seed=seed)
        self.sd = sd
        self.params = {k: v.requires_grad_(True) for k, v in sd.items() if not k.startswith("feat_embeddings")}
        self.m = {k: torch.zeros_like(v) for k, v in self.params.items()}
        self.v = {k: torch.zeros_like(v) for k, v in self.params.items()}
        self.step_no = 0

    def close(self):
        self.pool.terminate()
        self.pool.join()

    def sample(self, targets):
        items = self.pool.map(_work, list(targets), chunksize=max(1, len(targets) // (4 * self.cores)))
        t, p, n, lab = sampler_ref.ref_collate(items)
        as_t = lambda d: {k: torch.from_numpy(v) for k, v in d.items()}
        return as_t(t), as_t(p), torch.from_numpy(n), torch.from_numpy(lab)

    def train_step(self, batch):
        t, p, n, lab = batch
        for v in self.params.values():
            v.grad = None
        out = model_ref.pretrain_forward(self.sd, self.cfg, self.num_nodes, t, p, n, lab, training=True)
        out["loss"].backward()
        self.step_no += 1
        with torch.no_grad():
            for k, prm in self.params.items():
                if prm.grad is None:
                    continue
                wd = 0.0 if ("bias" in k or "LayerNorm.weight" in k) else 1e-2
                model_ref.adamw_step(prm, prm.grad, self.m[k], self.v[k], self.step_no, weight_decay=wd)
        return float(out["loss"])

    def timed_step(self, targets):
        """One full CPU step; returns (contexts, sampler_seconds, model_seconds, loss)."""
        t0 = time.perf_counter()
        batch = self.sample(targets)
        t1 = time.perf_counter()
        loss = self.train_step(batch)
        t2 = time.perf_counter()
        contexts = len(targets) + int(batch[2].sum())
        return contexts, t1 - t0, t2 - t1, loss


def run_cli(argv=None):
    """``python -m oracle.cpu_baseline --workload TG --steps K --warmup W --budget-s S``: prints one JSON line.
    Run as a separate process (never initialises CUDA) so that forking the sampler pool is safe."""
    import argparse
    import json
    import sys

    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="TG")
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--budget-s", type=float, default=25.0, help="target total CPU seconds for all steps")
    ap.add_argument("--max-batch", type=int, default=256, help="reference default train_batch_size (train.py:34)")
    a = ap.parse_args(argv)
    sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
    from pmgt_b200 import synthetic

    g = synthetic.make_item_graph(a.workload)
    feats = synthetic.make_features(g.num_nodes, seed=synthetic.SHAPES.get(a.workload, (0, 0, 0, 1234))[3])
    cp = CpuPretrainer(g.indptr, g.indices, g.weights.astype(np.float64), g.num_nodes, feats)
    rng = np.random.default_rng(0)
    try:
        # calibrate the per-step sample on a tiny step, then size steps to the budget
        c, ts, tm, _ = cp.timed_step(rng.integers(2, g.num_nodes + 2, size=16))
        per_target = (ts + tm) / 16.0
        total_steps = a.steps + a.warmup
        B = int(max(8, min(a.max_batch, a.budget_s / max(total_steps, 1) / max(per_target, 1e-6))))
        for _ in range(a.warmup):
            cp.timed_step(rng.integers(2, g.num_nodes + 2, size=B))
        ctx = s_s = s_m = 0.0
        losses = []
        for _ in range(a.steps):
            c, ts, tm, loss = cp.timed_step(rng.integers(2, g.num_nodes + 2, size=B))
            ctx += c
            s_s += ts
            s_m += tm
            losses.append(loss)
    finally:
        cp.close()
    print(json.dumps({
        "contexts": ctx, "sampler_s": s_s, "model_s": s_m, "steps": a.steps, "warmup": a.warmup,
        "targets_per_step": B, "cores": cp.cores, "value": ctx / (s_s + s_m),
        "sampler_contexts_per_s": ctx / s_s, "model_contexts_per_s": ctx / s_m, "loss_last": losses[-1],
        "ms_per_step": 1e3 * (s_s + s_m) / a.steps,
    }))


if __name__ == "__main__":
    run_cli()
