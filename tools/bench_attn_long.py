"""Cost of long neighbour contexts (64 < L <= 128) on one B200.

(a) The attention core alone (pmgt_attn_core_fwd / _bwd) at about the token count of a bench.py step (294,912 tokens:
    rows = 294,912 // L), L in {65, 73, 80, 100, 128}, (H, heads) in {(128, 1), (256, 4), (768, 12), (128, 4)}.
    CUDA-event time per call over `--reps` calls after a warm-up.  Algorithmic bytes per token: 5 bf16 rows of H
    forward (q, k, v, c read, ctx written), 9 backward (q, k, v, c, dctx read, dq, dk, dv, dc written).  FLOPs: the
    L x L x dh products the kernel issues, 2 flops per multiply-add, over the padded length LP = 16 ceil(L / 16):
    attn_long issues 5 of them forward (S1, S2 twice, A V once) and 14 backward.  Shares of peak: against 7.7 TB/s and
    against a measured mma.sync bf16 rate if one is given (--mma-tflops), else "not measured".
(b) With --parent-lib (the library built from the parent commit): every shape of (a) that the parent ran on the generic
    kernel is timed with both libraries in the same process, alternating, `--rounds` times; the outputs of both are
    compared.
(c) Whole training steps (PMGTTrainerModel.train_on_indices) on the TG-shaped synthetic graph, 1,024 targets per
    step, max_ctx_neigh in {5, 32, 63, 99}, then one profiled pass (ops.PROFILE) for the per-tag share of the step:
    the attention core's and the sampler's share at long contexts.

    python tools/bench_attn_long.py [--out FILE] [--parent-lib PATH] [--reps 20] [--rounds 3] [--steps 10]

Prints one JSON document (and writes it to --out).  Needs a CUDA device.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU
TOKENS = 294_912
LS = (65, 73, 80, 100, 128)
WIDTHS = ((128, 1), (256, 4), (768, 12), (128, 4))


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


def generic_at_parent(L, dh, bwd):
    """Shapes the parent commit ran on the generic kernel (attn_layout's 200 KB per-warp budget)."""
    if dh == 128:
        return L <= (73 if bwd else 107)
    return L <= {64: 85, 32: 92}[dh]


def _inputs(L, H, heads, seed=0):
    import torch
    rows = TOKENS // L
    T = rows * L
    g = torch.Generator(device="cuda").manual_seed(seed + L + H)
    qkvc = (torch.randn(T, 4 * H, device="cuda", generator=g) * 0.7).to(torch.bfloat16)
    mask = torch.ones(rows, L, device="cuda")
    n_real = torch.randint(1, L, (rows,), device="cuda", generator=g)
    mask[torch.arange(L, device="cuda")[None, :] > n_real[:, None]] = 0
    dctx = torch.randn(T, H, device="cuda", generator=g).to(torch.bfloat16)
    return rows, qkvc, mask, dctx


def _time(fn, reps):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3   # us


def kernels(reps, mma_tflops):
    import torch

    from pmgt_b200 import ops
    out = []
    for H, heads in WIDTHS:
        dh = H // heads
        for L in LS:
            rows, qkvc, mask, dctx = _inputs(L, H, heads)
            T = rows * L
            ctx = torch.empty(T, H, device="cuda", dtype=torch.bfloat16)
            dq = torch.empty_like(qkvc)
            fa = ops.attn_args(rows, L, H, heads, 0.5, qkvc, mask, 0.1, 7, 3, ctx=ctx)
            ba = ops.attn_args(rows, L, H, heads, 0.5, qkvc, mask, 0.1, 7, 3, dctx=dctx, dqkvc=dq)
            LP = 16 * ((L + 15) // 16)
            res = {"L": L, "H": H, "heads": heads, "dh": dh, "rows": rows, "tokens": T}
            for name, fn, a, nrows, nprod in (("fwd", ops.attn_core_fwd, fa, 5, 5), ("bwd", ops.attn_core_bwd, ba, 9, 14)):
                for _ in range(3):
                    fn(a)
                torch.cuda.synchronize()
                us = _time(lambda: fn(a), reps)
                nbytes = T * nrows * H * 2
                flops = 2 * nprod * rows * heads * LP * LP * dh
                res[name] = {"us": round(us, 1), "bytes_per_token": nrows * H * 2, "GB_s": round(nbytes / us / 1e3, 1),
                             "frac_of_7.7TB_s": round(nbytes / (us * 1e-6) / HBM_BYTES_PER_S, 4),
                             "issued_tflops": round(flops / us / 1e6, 1),
                             "frac_of_mma_sync_rate": (round(flops / us / 1e6 / mma_tflops, 3) if mma_tflops
                                                       else "not measured")}
            out.append(res)
            print(json.dumps(res), file=sys.stderr, flush=True)
            del qkvc, mask, dctx, ctx, dq
            torch.cuda.empty_cache()
    return out


def against_parent(parent_path, reps, rounds):
    import torch

    from pmgt_b200 import _lib, ops
    par = C.CDLL(os.path.abspath(parent_path))
    for name in ("pmgt_attn_core_fwd", "pmgt_attn_core_bwd"):
        getattr(par, name).restype = C.c_int
        getattr(par, name).argtypes = [C.POINTER(_lib.AttnArgs), C.c_void_p]
    assert par.pmgt_abi_version() == _lib.ABI_VERSION
    ours = _lib.lib()
    out = []
    for H, heads in WIDTHS:
        dh = H // heads
        for L in LS:
            dirs = [d for d in ("fwd", "bwd") if generic_at_parent(L, dh, d == "bwd")]
            if not dirs:
                continue
            rows, qkvc, mask, dctx = _inputs(L, H, heads, seed=1)
            T = rows * L
            res = {"L": L, "H": H, "heads": heads, "dh": dh, "rows": rows}
            for d in dirs:
                bufs = {lib: torch.empty(T, H if d == "fwd" else 4 * H, device="cuda", dtype=torch.bfloat16)
                        for lib in ("parent", "this")}
                args = {}
                for lib, buf in bufs.items():
                    kw = dict(ctx=buf) if d == "fwd" else dict(dctx=dctx, dqkvc=buf)
                    args[lib] = ops.attn_args(rows, L, H, heads, 0.5, qkvc, mask, 0.0, 7, 3, **kw)
                fns = {"parent": getattr(par, f"pmgt_attn_core_{d}"), "this": getattr(ours, f"pmgt_attn_core_{d}")}

                def call(lib):
                    _lib.check(fns[lib](C.byref(args[lib]), ops.cur_stream()), f"{lib} {d}")

                for lib in ("parent", "this"):
                    call(lib)
                torch.cuda.synchronize()
                times = {"parent": [], "this": []}
                for _ in range(rounds):
                    for lib in ("parent", "this"):
                        times[lib].append(_time(lambda: call(lib), reps))
                a, b = bufs["parent"].float(), bufs["this"].float()
                res[d] = {"parent_us": [round(x, 1) for x in times["parent"]], "this_us": [round(x, 1) for x in times["this"]],
                          "speedup_median": round(sorted(times["parent"])[rounds // 2] / sorted(times["this"])[rounds // 2], 2),
                          "max_abs_diff_over_max": float((a - b).abs().max() / a.abs().max().clamp_min(1e-6))}
            out.append(res)
            print(json.dumps(res), file=sys.stderr, flush=True)
            del qkvc, mask, dctx
            torch.cuda.empty_cache()
    return out


def steps(max_ctx, n_steps, warmup):
    import numpy as np
    import torch

    from pmgt_b200 import ops, trainer
    dev = torch.device("cuda", 0)
    B = 1024
    args = trainer.make_args(synthetic="TG", train_batch_size=B, seed=0, max_ctx_neigh=max_ctx)
    trainer.check_args(args)
    args.device = dev
    trainer.set_seed(0)
    trainer.init_dataloader(args)
    trainer.init_model(args)
    tm = trainer.PMGTTrainerModel(args)
    ds = args.train_dataset
    perm = trainer.epoch_permutation(len(ds), 0, 0)
    n_total = warmup + n_steps + 2
    idx = [torch.from_numpy(trainer.shard_indices(np.tile(perm, 4), s, B, 0, 1).astype(np.int64)).to(dev)
           for s in range(n_total)]

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
    # one profiled pass of two steps: per-tag device time (events around every library call)
    ops.PROFILE = []
    run(warmup + n_steps, 2)
    torch.cuda.synchronize()
    summ = ops.profile_summary(ops.PROFILE)
    ops.PROFILE = None
    tot = sum(v["ms"] for v in summ.values())
    share = {k: round(v["ms"] / tot, 4) for k, v in sorted(summ.items(), key=lambda kv: -kv[1]["ms"])}
    res = {"max_ctx_neigh": max_ctx, "L": max_ctx + 1, "targets": B, "ms_per_step": round(ms, 3), "loss_last": float(loss),
           "profiled_ms_per_step": round(tot / 2, 3), "share_of_profiled_time": share,
           "attn_core_share": round(share.get("attn_core_fwd", 0) + share.get("attn_core_bwd", 0), 4),
           "sampler_share": round(share.get("sample_contexts", 0) + share.get("sample_pairs", 0), 4)}
    print(json.dumps(res), file=sys.stderr, flush=True)
    del tm, args, ds, idx
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None)
    ap.add_argument("--parent-lib", default=None, help="libpmgt_b200.so built from the parent commit")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--mma-tflops", type=float, default=None, help="a measured mma.sync bf16 rate, TFLOP/s")
    ap.add_argument("--skip-steps", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_attn_long.py needs a CUDA device")
    torch.cuda.set_device(0)
    doc = {"card": card(), "attn_core": kernels(a.reps, a.mma_tflops)}
    if a.parent_lib:
        doc["against_parent"] = against_parent(a.parent_lib, max(2, a.reps // 4), a.rounds)
    if not a.skip_steps:
        doc["training_step_TG_1024"] = [steps(m, a.steps, a.warmup) for m in (5, 32, 63, 99)]
    doc["card_after"] = card()
    text = json.dumps(doc, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
