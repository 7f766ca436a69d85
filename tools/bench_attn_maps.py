"""Cost of the attention maps (output_attentions) and per-layer hidden states (output_hidden_states) on one B200.

(a) pmgt_attn_maps_fwd next to pmgt_attn_core_fwd at the same shapes, about the token count of a bench.py step
    (294,912 tokens: rows = 294,912 // L): L = 6 / dh 128, L = 33 / 12 x 64, L = 100 / dh 128, L = 128 / 4 x 32, in eval
    (no dropout) and with dropout 0.1.  CUDA-event time per call over `--reps` calls after a warm-up, the two kernels
    alternating `--rounds` times in the same process; the median round is reported.  Bytes: the maps kernel reads the
    q, k, c columns (3 bf16 rows of H per token) and writes heads * L fp32 per token; the core reads q, k, v, c and writes
    ctx (5 bf16 rows of H).  Achieved bandwidth = bytes / time, next to the bandwidth of a device-to-device copy
    (read + write bytes of a 2 GiB torch copy over its time) measured in the same run.
(b) An eval forward the size of PMGT.item_embeddings' default use (B targets of L = 6 at the default config, B * L about
    294,912 tokens) through PMGT.forward with and without both output flags, and item_embeddings itself; host clock
    around calls that end in a device synchronise, alternating, median of `--rounds`.

    python tools/bench_attn_maps.py [--out FILE] [--reps 20] [--rounds 5]

Prints one JSON document (and writes it to --out, default profiles/r6_attn_maps.json).  Needs a CUDA device.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

TOKENS = 294_912
SHAPES = ((6, 128, 1), (33, 768, 12), (100, 128, 1), (128, 128, 4))   # (L, H, heads)


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


def _time(fn, reps):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3   # us


def copy_bandwidth(reps):
    import torch
    n = 1 << 29   # 2 GiB of fp32: far beyond the 126 MB L2
    src = torch.empty(n, device="cuda")
    dst = torch.empty_like(src)
    dst.copy_(src)
    us = _time(lambda: dst.copy_(src), reps)
    del src, dst
    return 2 * 4 * n / (us * 1e-6)


def kernels(reps, rounds, copy_bps):
    import torch
    from pmgt_b200 import ops
    out = []
    for L, H, heads in SHAPES:
        rows = TOKENS // L
        T = rows * L
        g = torch.Generator(device="cuda").manual_seed(L + H)
        qkvc = (torch.randn(T, 4 * H, device="cuda", generator=g) * 0.7).to(torch.bfloat16)
        mask = torch.ones(rows, L, device="cuda")
        n_real = torch.randint(1, L, (rows,), device="cuda", generator=g) if L > 1 else torch.zeros(rows, device="cuda")
        mask[torch.arange(L, device="cuda")[None, :] > n_real[:, None]] = 0
        ctx = torch.empty(T, H, device="cuda", dtype=torch.bfloat16)
        maps = torch.empty(rows, heads, L, L, device="cuda")
        for p in (0.0, 0.1):
            core_a = ops.attn_args(rows, L, H, heads, 0.5, qkvc, mask, p, 7, 10, ctx=ctx)
            maps_a = ops.attn_args(rows, L, H, heads, 0.5, qkvc, mask, p, 7, 10)
            core = lambda: ops.attn_core_fwd(core_a)
            mp = lambda: ops.attn_maps_fwd(maps_a, maps)
            core(), mp()
            torch.cuda.synchronize()
            t_core, t_maps = [], []
            for _ in range(rounds):
                t_core.append(_time(core, reps))
                t_maps.append(_time(mp, reps))
            tc, tm = statistics.median(t_core), statistics.median(t_maps)
            maps_bytes = T * (3 * H * 2 + heads * L * 4)
            core_bytes = T * 5 * H * 2
            res = {"L": L, "H": H, "heads": heads, "dh": H // heads, "rows": rows, "dropout_p": p,
                   "core_fwd_us": round(tc, 2), "maps_fwd_us": round(tm, 2), "maps_over_core": round(tm / tc, 3),
                   "maps_write_GBps": round(T * heads * L * 4 / (tm * 1e-6) / 1e9, 1),
                   "maps_bytes_GBps": round(maps_bytes / (tm * 1e-6) / 1e9, 1),
                   "maps_share_of_copy_bw": round(maps_bytes / (tm * 1e-6) / copy_bps, 3),
                   "core_bytes_GBps": round(core_bytes / (tc * 1e-6) / 1e9, 1),
                   "rounds_core_us": [round(x, 2) for x in t_core], "rounds_maps_us": [round(x, 2) for x in t_maps]}
            out.append(res)
            print(json.dumps(res), file=sys.stderr, flush=True)
        del qkvc, ctx, maps
        torch.cuda.empty_cache()
    return out


def model_eval(rounds):
    import numpy as np
    import torch
    from pmgt_b200 import PMGT, PMGTConfig
    node_size, L = 20_000, 6
    B = TOKENS // L
    rng = np.random.default_rng(0)
    feats = [rng.standard_normal((node_size + 2, d), dtype=np.float32) for d in (1536, 768)]
    net = PMGT(node_size, config=PMGTConfig(), feat_init_emb=feats).cuda().eval()
    g = torch.Generator(device="cuda").manual_seed(1)
    ids = torch.randint(2, node_size + 2, (B, L), device="cuda", generator=g)
    mask = torch.ones(B, L, device="cuda")
    target = {"node_ids": ids, "attention_mask": mask}

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3, r

    runs = {
        "item_embeddings": lambda: net.item_embeddings(target),
        "forward": lambda: net(target),
        "forward_with_outputs": lambda: net(target, output_hidden_states=True, output_attentions=True),
    }
    with torch.no_grad():
        for fn in runs.values():   # warm-up: module loads, first-use attributes
            fn()
        times = {k: [] for k in runs}
        for _ in range(rounds):
            for k, fn in runs.items():
                ms, r = timed(fn)
                times[k].append(ms)
                del r
        out = net(target, output_hidden_states=True, output_attentions=True)
        extra = sum(t.numel() * 4 for t in out.hidden_states[:-1]) + sum(t.numel() * 4 for t in out.attentions)
    res = {"B": B, "L": L, "config": "default (H 128, 5 layers, 1 head)",
           **{f"{k}_ms": round(statistics.median(v), 3) for k, v in times.items()},
           "rounds_ms": {k: [round(x, 3) for x in v] for k, v in times.items()},
           "output_bytes": extra}
    res["outputs_over_forward"] = round(res["forward_with_outputs_ms"] / res["forward_ms"], 3)
    print(json.dumps(res), file=sys.stderr, flush=True)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_attn_maps.json"))
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_attn_maps.py needs a CUDA device")
    from pmgt_b200 import build
    build.build()
    copy_bps = copy_bandwidth(args.reps)
    doc = {"card": card(), "tokens": TOKENS, "copy_GBps": round(copy_bps / 1e9, 1),
           "kernels": kernels(args.reps, args.rounds, copy_bps), "eval_forward": model_eval(args.rounds)}
    text = json.dumps(doc, indent=1)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
