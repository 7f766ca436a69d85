"""Cost of the number of feature modalities on one B200.

(a) The embedding fusion kernels alone (pmgt_embed_multi_fwd / _bwd, M = 2 through the two-modality kernels) at the
    token count of a bench.py step (T = 294,912: 4,096 targets, 40,960 pairs, 4,096 masked targets, L = 6), H = 128,
    M = 1..4, in both output modes: per-token rows (gather-fused projections) and projected-table rows (row_idx into a
    1,000,002-row table, fp32 red.add of the row gradients).  CUDA-event time per call over `--reps` calls after a
    warm-up; algorithmic bytes from shapes: forward reads M rows and writes one (256 B each), backward reads M rows plus
    dx and dx_b and writes M rows (256 B bf16 per token, or 512 B fp32 per table-row update).  The operands (>= 0.3 GB)
    exceed the 126 MB L2.
(b) Whole training steps on BASELINE config 3 (1M-node / 20M-edge synthetic graph, 4,096 targets per step) through
    PMGTTrainerModel.train_on_indices with device-resident index batches, for the modality sets 1536 + 768 (today's
    workload), 1536 + 768 + 512 and 1536 alone.  ms/step and contexts/s (11 contexts per target) as bench.py reports them.

    python tools/bench_modalities.py [--out FILE] [--steps 20] [--warmup 5] [--reps 20]

Prints one JSON document (and writes it to --out).  Needs a CUDA device.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU
ROWS, L, H = 49152, 6, 128  # T = 294,912 tokens
TABLE_ROWS = 1_000_002


def card():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(q[0]), float(q[1])
    except Exception as exc:  # the numbers are still reported, without the power limit
        info["power_limit_w"] = f"unavailable ({exc})"
    return info


def kernels(reps):
    import torch

    from pmgt_b200 import ops
    dev = "cuda"
    T = ROWS * L
    g = torch.Generator(device=dev).manual_seed(0)
    out = []
    prev = ops.set_pdl(False)
    for mode in ("tokens", "table"):
        n_src = TABLE_ROWS if mode == "table" else T
        row_idx = torch.randint(0, TABLE_ROWS, (T,), device=dev, generator=g) if mode == "table" else None
        for M in (1, 2, 3, 4):
            e = [torch.randn(n_src, H, device=dev, generator=g).to(torch.bfloat16) for _ in range(M)]
            p = dict(w_att=torch.randn(M, M * H, device=dev, generator=g) * 0.05, b_att=torch.zeros(M, device=dev),
                     pos=torch.randn(100, H, device=dev, generator=g) * 0.02, role=torch.randn(2, H, device=dev, generator=g) * 0.02,
                     ln_g=torch.ones(H, device=dev), ln_b=torch.zeros(H, device=dev))
            x = torch.empty(T, H, dtype=torch.bfloat16, device=dev)
            dx = torch.randn(T, H, device=dev, generator=g).to(torch.bfloat16)
            dx_b = torch.randn(T, H, device=dev, generator=g).to(torch.bfloat16)
            grads = {k: torch.zeros_like(v) for k, v in p.items()}
            d_bias = [torch.zeros(H, device=dev) for _ in range(M)]
            kw = {}
            if mode == "table":
                kw = dict(row_idx=row_idx, de_acc=[torch.zeros(TABLE_ROWS, H, device=dev) for _ in range(M)], skip_row0=1)
            else:
                kw = dict(de=[torch.empty(T, H, dtype=torch.bfloat16, device=dev) for _ in range(M)])
            common = (ROWS, L, H, e, p["w_att"], p["b_att"], p["pos"], p["role"], p["ln_g"], p["ln_b"], 1e-12, 0.1, 7, 0)
            fa = ops.embed_multi_args(*common, x_out=x, **({"row_idx": row_idx} if row_idx is not None else {}))
            ba = ops.embed_multi_args(*common, dx=dx, dx_b=dx_b, d_w_att=grads["w_att"], d_b_att=grads["b_att"],
                                      d_pos=grads["pos"], d_role=grads["role"], d_ln_g=grads["ln_g"], d_ln_b=grads["ln_b"],
                                      d_bias=d_bias, **kw)
            res = {"mode": mode, "M": M, "T": T, "H": H}
            for name, fn, a in (("fwd", ops.embed_multi_fwd, fa), ("bwd", ops.embed_multi_bwd, ba)):
                for _ in range(3):
                    fn(a)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    fn(a)
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / reps
                idx = 8 if mode == "table" else 0
                if name == "fwd":
                    nbytes = T * ((M + 1) * 2 * H + idx)
                else:
                    nbytes = T * ((M + 2) * 2 * H + idx + M * (4 if mode == "table" else 2) * H)
                res[name] = {"us": round(ms * 1e3, 2), "bytes": nbytes, "GB_s": round(nbytes / (ms / 1e3) / 1e9, 1),
                             "frac_of_7.7TB_s": round(nbytes / (ms / 1e3) / HBM_BYTES_PER_S, 3)}
            res["fwd_plus_bwd_us"] = round(res["fwd"]["us"] + res["bwd"]["us"], 2)
            out.append(res)
            print(json.dumps(res), file=sys.stderr, flush=True)
            del e, x, dx, dx_b, grads, d_bias, kw, fa, ba
            torch.cuda.empty_cache()
    ops.set_pdl(prev)
    for mode in ("tokens", "table"):
        two = next(r for r in out if r["mode"] == mode and r["M"] == 2)["fwd_plus_bwd_us"]
        for r in out:
            if r["mode"] == mode:
                r["fwd_plus_bwd_vs_M2"] = round(r["fwd_plus_bwd_us"] / two, 3)
    return out


def steps(dims, n_steps, warmup):
    import numpy as np
    import torch

    from pmgt_b200 import synthetic, trainer
    dev = torch.device("cuda", 0)
    args = trainer.make_args(synthetic="1M", train_batch_size=4096, seed=0)
    args.device = dev
    trainer.set_seed(0)
    args.graph, feats = trainer._load_graph_and_features(args)
    if tuple(dims) == (1536, 768):
        args.feat_init_emb = feats
    elif tuple(dims) == (1536,):
        args.feat_init_emb = feats[:1]
    else:
        extra = synthetic.make_features_device(args.graph.num_nodes, dims=dims[2:], seed=4321, device=dev)
        args.feat_init_emb = list(feats) + list(extra)
    del feats
    trainer.init_dataloader(args)
    trainer.init_model(args)
    assert args.model.config.feat_hidden_sizes == list(dims)
    tm = trainer.PMGTTrainerModel(args)
    ds = args.train_dataset
    perm = trainer.epoch_permutation(len(ds), 0, 0)
    idx = [torch.from_numpy(trainer.shard_indices(perm, s, 4096, 0, 1).astype(np.int64)).to(dev)
           for s in range(warmup + n_steps)]

    def run(first, n):
        loss = None
        for k in range(n):
            s = first + k
            loss = tm.train_on_indices(ds, idx[s], epoch=s)
            if k + 1 < n:
                tm.prefetch(ds, idx[s + 1], epoch=s + 1)
        return loss

    run(0, warmup)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    loss = run(warmup, n_steps)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n_steps
    res = {"feat_hidden_sizes": list(dims), "ms_per_step": round(ms, 3),
           "contexts_per_s": round(4096 * 11 / (ms / 1e3), 1), "loss_last": float(loss),
           "trainable_params": sum(p.numel() for p in args.model.parameters() if p.requires_grad)}
    print(json.dumps(res), file=sys.stderr, flush=True)
    del tm, args, ds, idx
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--skip-steps", action="store_true", help="fusion kernels only")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_modalities.py needs a CUDA device")
    torch.cuda.set_device(0)
    doc = {"card": card(), "fusion_kernels": kernels(a.reps)}
    if not a.skip_steps:
        doc["training_step_config3"] = [steps(d, a.steps, a.warmup) for d in ((1536, 768), (1536, 768, 512), (1536,))]
    doc["card_after"] = card()
    text = json.dumps(doc, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
