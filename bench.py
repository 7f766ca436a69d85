#!/usr/bin/env python
"""PMGT pre-training throughput benchmark (driver contract: one JSON line on rank 0).

    python bench.py --gpus N --steps K --warmup W            # ours (B200, libpmgt_b200.so)
    python bench.py --impl reference --gpus N --steps K ...  # reference algorithm on the host CPU cores
    python bench.py --impl reference-gpu                     # reference model step, stock PyTorch eager on one B200

Metric (BASELINE.json): node-contexts/s of the pre-training step
{sample -> gather -> encode -> losses -> backward -> allreduce -> AdamW}; one
node-context = one sampled row of node_ids consumed by the encoder (B targets +
B*P pairs per step; the masked re-encode is extra work, not extra contexts).

Workload (every N, so that the 1/2/4/8-GPU series is ONE workload): BASELINE.json
configs[2], the synthetic 1M-node / 20M-edge item graph (1536-d + 768-d features,
4.6 GB of bf16 tables per GPU), default encoder (H = I = 128, 5 layers, 1 head,
L = 6, hops [16, 8, 4], P = 10), bf16 tensor-core GEMMs, 4096 targets (45,056
contexts) per GPU per step; weak scaling for N > 1 (per-GPU batch fixed, the global
batch of a step is 4096 x N distinct training nodes sharded by rank, one NCCL
allreduce of the flat gradient per step).  At N = 1 the line also carries
`config2_TG` (configs[1]: the TG-shaped graph on one B200), `cpu_baseline` (the CPU
port of the reference on the host cores) and `gpu_baseline` (the reference's model
step run eagerly with stock PyTorch ops on the same GPU).  `--workload TG|VG`
selects the other graphs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--workload", default="1M", choices=["VG", "TG", "1M"],
                    help="1M = BASELINE config 3 (1M nodes / 20M edges; default at every N so that the 1/2/4/8-GPU series is "
                         "one workload), TG = config 2, VG = config 1")
    ap.add_argument("--encoder", default="default", choices=["default", "wide"],
                    help="wide = BASELINE config 5: H=768, 12 layers, 12 heads, I=3072, 32 neighbours (L=33)")
    ap.add_argument("--batch", type=int, default=4096, help="targets per GPU per step")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="strong scaling (SURVEY 8(d) config 3: global B = 8192): targets per step over ALL ranks; each "
                         "rank takes global_batch / N of them and the line says \"scaling\": \"strong\"")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the config-2 (TG) block of the N = 1 line")
    ap.add_argument("--profile-out", default=None, help="write the per-kernel-family event profile to this JSON file")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last of them returned, its loss, as DIR/loss.npy "
                         "(float32); the inputs are seeded, so two builds run with the same arguments can be compared "
                         "output for output")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return a


def load_traffic(workload, batch):
    """Measured DRAM bytes per launch of each kernel family (ncu --set full captures, summarised in profiles/).
    File layout: {workload: {"targets_per_gpu_per_step": B, "traffic_bytes_per_launch": {family: bytes}}} (the
    round-1 single-workload layout is still understood)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return {}
    with open(p) as f:
        d = json.load(f)
    if workload in d and isinstance(d[workload], dict):
        d = d[workload]
    elif d.get("workload") != workload:
        return {}
    if d.get("targets_per_gpu_per_step") != batch:
        return {}
    return d.get("traffic_bytes_per_launch", {})


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d.get("bf16_tflops_sustained", d.get("bf16_tflops")), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1400.0, source="fallback")  # B200_PROFILING.md fallback


# ---------------------------------------------------------------------------
# reference arms: the oracle port on the host cores / eagerly on the GPU, each in a subprocess
# ---------------------------------------------------------------------------
def run_cpu_port(workload, steps, warmup, budget_s):
    """The reference's CPU path on the host cores, in a CUDA-free subprocess: the UNMODIFIED reference modules when they
    are available (the checkout oracle/ref_shim.py finds, or the copies oracle/build.py staged under oracle/_ref/ -- kind
    "reference"), else the oracle port (kind "port"), said on stderr."""
    from oracle import ref_shim
    use_ref = ref_shim.available() or ref_shim.staged_available()
    mod = "oracle.ref_baseline" if use_ref else "oracle.cpu_baseline"
    if not use_ref:
        print("bench: no upstream uoo723/PMGT reference (set PMGT_REFERENCE_ROOT, or stage it with build()); the CPU "
              "arm times the oracle port (kind \"port\")", file=sys.stderr)
    cmd = [sys.executable, "-m", mod, "--workload", workload, "--steps", str(steps), "--warmup", str(warmup),
           "--budget-s", str(budget_s)]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    if r.returncode != 0 and use_ref:  # never lose the line over the staged copy: fall back to the port, and say so
        print("bench: the reference's own modules failed; the CPU arm times the oracle port (kind \"port\"):\n"
              + r.stderr[-1000:], file=sys.stderr)
        cmd[2] = "oracle.cpu_baseline"
        r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    if r.returncode != 0:
        raise RuntimeError("cpu baseline failed: " + r.stderr[-2000:])
    d = json.loads(r.stdout.strip().splitlines()[-1])
    d.setdefault("kind", "port")
    return d


def run_gpu_eager(workload, batch, steps, warmup, device_index=0):
    """The reference's model step run eagerly on the GPU (oracle restatement, stock PyTorch ops, per-target loop)."""
    cmd = [sys.executable, "-m", "oracle.gpu_baseline", "--workload", workload, "--batch", str(batch), "--steps", str(steps),
           "--warmup", str(warmup)]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES=str(device_index))
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    if r.returncode != 0:
        raise RuntimeError("gpu eager baseline failed: " + r.stderr[-2000:])
    return json.loads(r.stdout.strip().splitlines()[-1])


def reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = "TG" if a.workload == "1M" else a.workload  # the fp32 host tables of the 1M graph (9.2 GB) are not built for a CPU run
    d = run_cpu_port(wl, a.steps, a.warmup, budget_s=150.0)
    how = ("the reference's own PMGTDataset in DataLoader worker processes + PMGT.forward (per-target loop) + "
           "DenseSparseAdamW" if d["kind"] == "reference" else "oracle port: sampler in a process pool, batched pair encode")
    sample = (f"{d['targets_per_step']} targets ({int(d['contexts'] / d['steps'])} contexts) per step x {d['steps']} steps on "
              f"the {wl} graph; {how}; {d['cores']} cores")
    line = {
        "impl": "reference", "metric": "pmgt_pretrain_node_contexts_per_s", "value": d["value"], "unit": "contexts/s",
        "n_gpus": a.gpus, "steps": d["steps"], "warmup": d["warmup"], "ms_per_step": d["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(wl, d["targets_per_step"], "cpu"),
        "cpu_baseline": {"value": d["value"], "unit": "contexts/s", "cores": d["cores"], "kind": d["kind"], "sample": sample,
                         "sampler_contexts_per_s": d["sampler_contexts_per_s"], "model_contexts_per_s": d["model_contexts_per_s"]},
        "e2e": {"value": d["value"], "unit": "contexts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def reference_gpu_arm(a):
    """`--impl reference-gpu`: stock-PyTorch eager execution of the reference's model step on one B200 (BASELINE.md
    section 4 item 5), at the reference's batch (256) and, when --batch differs, at that batch too."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = "TG" if a.workload == "1M" else a.workload
    steps, warmup = max(1, min(a.steps, 3)), max(1, min(a.warmup, 1))
    d = run_gpu_eager(wl, 256, steps, warmup)
    extra = None
    if a.batch != 256:
        extra = run_gpu_eager(wl, a.batch, 1, 0)
    line = {
        "impl": "reference-gpu", "metric": "pmgt_pretrain_node_contexts_per_s", "value": d["value"], "unit": "contexts/s",
        "n_gpus": 1, "steps": steps, "warmup": warmup, "ms_per_step": d["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(wl, 256, "gpu, stock PyTorch eager (oracle restatement of the reference model step; sampler excluded)"),
        "gpu_baseline": d, "gpu_baseline_at_batch": extra, "gpu_launches": 0,
        "e2e": {"value": d["value"], "unit": "contexts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


ENCODERS = {
    "default": (dict(), "default encoder H=128 I=128 5 layers 1 head, L=6"),
    "wide": (dict(hidden_size=768, intermediate_size=3072, num_hidden_layers=12, num_attention_heads=12, max_ctx_neigh=32),
             "wide encoder H=768 I=3072 12 layers 12 heads, L=33"),
}


def workload_config(wl, batch, where, encoder="default"):
    from pmgt_b200 import synthetic
    n, m, _, _ = synthetic.SHAPES[wl]
    return {"workload": f"PMGT pre-training step on synthetic {wl}-shaped item graph ({n} nodes / {m} edges, 1536-d visual + "
                        f"768-d text features), {ENCODERS[encoder][1]}, hops [16,8,4], 10 pairs/target",
            "targets_per_gpu_per_step": batch, "contexts_per_gpu_per_step": batch * 11, "where": where,
            "l2": "per-step working set (activations, several GB at the default batch) is >> the 126 MB L2; no explicit flush"}


# ---------------------------------------------------------------------------
# clocks sampling (nvidia-smi during the timed region)
# ---------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for nme, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        return {"sm_mhz": (sm[len(sm) // 2] if sm else None), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------
# kernel families of the encoder layers (SURVEY section 8(d) "K3": tensor-bound by definition, activations ideally on chip)
K3_FAMILIES = ("lt_qkvc_fwd", "attn_core_fwd", "lt_res_ln_fwd", "lt_gelu_fwd", "ffn_fwd", "ffn_bwd", "ln_bwd", "lt_dxdw_gelu",
               "lt_dxdw", "attn_core_bwd", "lt_dx_qkvc", "dw_tile", "gather_rows", "scatter_rows")
# widths the token-tile kernels do not cover (--encoder wide): the layers run on pmgt_gemm_bf16 + row-wise LayerNorm
# (the few non-layer GEMMs of a step -- projected feature tables, NFR heads -- carry their own tags or are < 1 % here)
K3_FAMILIES_WIDE = ("gemm_fwd", "gemm_dx", "gemm_dw", "res_ln_fwd", "res_ln_bwd", "attn_core_fwd", "attn_core_bwd", "colsum")
# SURVEY section 8(d) "K2": the multimodal feature path (gather + per-modality projection, then the fusion kernel)
K2_GATHER_FAMILIES = ("gemm_fwd_gather", "gemm_dw_gather")


def k3_flops_per_step(cfg_over, batch, L):
    """SURVEY section 8(d): per sequence and layer forward 8LH^2 + 6L^2H + 2LH^2 + 4LHI FLOPs, backward 2x; a training
    target costs 12 encoded sequences (target, 10 pairs, masked target)."""
    H = cfg_over.get("hidden_size", 128)
    inter = cfg_over.get("intermediate_size", 128)
    layers = cfg_over.get("num_hidden_layers", 5)
    per_seq_layer = 8 * L * H * H + 6 * L * L * H + 2 * L * H * H + 4 * L * H * inter
    return 3.0 * per_seq_layer * layers * 12 * batch


def measure(a, workload, steps, warmup, profile, rank, local_rank, ws, dev, dump_dir=None):
    """Builds the workload, runs the device-resident series (`value`), the end-to-end series (`e2e`) and, if asked,
    the per-kernel-family event profile.  Returns a dict of results (rank 0 carries the roofline).  With `dump_dir`,
    rank 0 writes there what the last step of the device-resident series returned, its loss.  The parameters and
    gradients that step leaves are not written: the backward pass sums gradients with floating-point atomics and AdamW
    amplifies the rounding differences, so after a few steps they differ from run to run by far more than rounding."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from pmgt_b200 import ops, trainer

    args = trainer.make_args(synthetic=workload, train_batch_size=a.batch, seed=0, **ENCODERS[a.encoder][0])
    args.device = dev
    trainer.set_seed(0)
    args.graph, args.feat_init_emb = trainer._load_graph_and_features(args)
    trainer.init_dataloader(args)
    trainer.init_model(args)
    tm = trainer.PMGTTrainerModel(args)
    ds = args.train_dataset
    B = a.batch
    n_train = len(ds)
    per_step = B * ws
    steps_per_epoch = max(1, n_train // per_step)
    perm_cache = {}

    def step_indices(step):
        # weak scaling: the global batch of a step is B * ws DISTINCT training nodes of a (seed, epoch)-derived
        # permutation, rank r takes its contiguous slice (trainer.shard_indices); only when the training split is
        # smaller than one global batch (TG beyond 2 GPUs) the permutation is tiled
        epoch, k = divmod(step, steps_per_epoch)
        perm = perm_cache.get(epoch)
        if perm is None:
            perm = trainer.epoch_permutation(n_train, 0, epoch)
            if n_train < per_step:
                perm = np.concatenate([perm] * ((per_step + n_train - 1) // n_train))
            perm_cache.clear()
            perm_cache[epoch] = perm
        return trainer.shard_indices(perm, k, B, rank, ws).astype(np.int64)

    total = warmup + steps
    idx_host = [torch.from_numpy(step_indices(s)).pin_memory() for s in range(total + steps)]
    idx_dev = [t.to(dev) for t in idx_host[:total]]

    def barrier():
        if ws > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_steps(src, first, n, read_loss=False, prefetch=True):
        """n consecutive steps; the batch of step k+1 (sampling + NFR corruption, and for host-resident indices their
        H2D copy) is prepared on the trainer's side stream while step k runs -- what a DataLoader's prefetch does."""
        loss = None
        for k in range(n):
            s = first + k
            loss = tm.train_on_indices(ds, src[s], epoch=s)
            if prefetch and k + 1 < n:
                tm.prefetch(ds, src[s + 1], epoch=s + 1)
            if read_loss:
                loss = tm.last_loss()  # D2H read of this step's loss (pinned buffer; waits for the forward pass only)
        return loss

    # ---- device-resident run: `value`
    run_steps(idx_dev, 0, warmup)
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    launches0 = ops.LAUNCHES[0]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last_loss = run_steps(idx_dev, warmup, steps)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ops.LAUNCHES[0] - launches0
    clk = clocks.stop() if rank == 0 else None
    if dump_dir and rank == 0:
        os.makedirs(dump_dir, exist_ok=True)
        np.save(os.path.join(dump_dir, "loss.npy"), last_loss.float().cpu().numpy())
    t = torch.tensor([ms], device=dev)
    if ws > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t)
    contexts_per_step = B * 11 * ws
    value = contexts_per_step * steps / (ms / 1e3)

    # ---- end-to-end run: host index batch (pinned) -> H2D -> step -> loss D2H, every step
    barrier()
    w0 = time.perf_counter()
    e0.record()
    loss_host = run_steps(idx_host, total, steps, read_loss=True)
    e1.record()
    barrier()
    ms_e2e = max(e0.elapsed_time(e1), (time.perf_counter() - w0) * 1e3)
    t = torch.tensor([ms_e2e], device=dev)
    if ws > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = contexts_per_step * steps / (float(t) / 1e3)
    res = {"value": value, "ms_per_step": ms / steps, "e2e_value": e2e_value, "launches": launches, "clocks": clk,
           "loss_last": loss_host, "roofline": None, "k3": None, "k2": None, "profile": None}

    # ---- per-kernel-family profile (CUDA events on the launching stream, inside real steps) -> roofline
    if profile:
        # every rank runs the profiled steps (they contain the gradient allreduce); only rank 0 records events
        n_prof = min(3, steps)
        if rank == 0:
            ops.PROFILE = []
        # (no side-stream prefetch and no programmatic dependent launch here: every kernel is timed alone)
        pdl_was = ops.set_pdl(False)
        run_steps(idx_dev, warmup, n_prof, prefetch=False)
        barrier()
        ops.set_pdl(pdl_was)
        if rank == 0:
            recs, ops.PROFILE = ops.PROFILE, None
            prof = ops.profile_summary(recs)
            tot = sum(d["ms"] for d in prof.values())
            for d in prof.values():
                d["ms_per_step"] = d["ms"] / n_prof
                d["share"] = d["ms"] / tot
                d["gbs"] = d["bytes"] / (d["ms"] * 1e-3) / 1e9 if d["ms"] > 0 else 0.0
                d["tflops"] = d["flops"] / (d["ms"] * 1e-3) / 1e12 if d["ms"] > 0 else 0.0
            top = max(prof, key=lambda k: prof[k]["ms"])
            peaks = load_peaks()
            d = prof[top]
            traffic = load_traffic(workload, B).get(top)
            note = None
            achieved = d["gbs"]
            if top == "sample_contexts":
                # The sampler is a dependent random-access chain (row pointers -> guide entry -> (cdf, id) pairs), not a
                # scan: SURVEY 8(d)'s linear-scan byte formula does not describe it.  Its HBM figure is the DRAM traffic
                # ncu measured for one launch of this workload (profiles/) over the live-timed duration; what bounds it is
                # the latency of ~4 dependent loads per draw x 3 hops, not bandwidth.
                achieved = (traffic / (1e3 * d["ms"] / d["calls"] * 1e-6) / 1e9) if traffic else None
                note = ("latency-bound dependent gather: achieved = ncu-measured DRAM bytes per launch / live duration"
                        if traffic else "latency-bound dependent gather; no DRAM-traffic capture for this workload: no HBM fraction quoted")
            frac = achieved / peaks["hbm_gbs"] if achieved else None
            if frac is not None and frac > 1.2:  # a byte model that beats the copy bandwidth by 20 % is not evidence
                note = f"byte model invalid for this kernel (would give {frac:.2f}); not quoted"
                frac, achieved = None, None
            roof = {"kernel": top, "bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": frac, "traffic": traffic,
                    # no algorithmic byte model for the sampler (see note): null, not 0
                    "algorithmic_bytes_per_launch": (d["bytes"] / d["calls"]) if d["bytes"] else None,
                    "peak_source": peaks["source"], "share_of_step": d["share"], "launches_per_step": d["calls"] / n_prof,
                    "avg_launch_us": 1e3 * d["ms"] / d["calls"], "tensor_tflops": d["tflops"], "note": note}
            # SURVEY 8(d) classifies the encoder layers (K3) as tensor-bound: FLOP-based fraction of the whole K3 chain
            fams = K3_FAMILIES_WIDE if a.encoder == "wide" else K3_FAMILIES
            k3_ms = sum(v["ms_per_step"] for k, v in prof.items() if k in fams)
            L = ENCODERS[a.encoder][0].get("max_ctx_neigh", 5) + 1
            k3_fl = k3_flops_per_step(ENCODERS[a.encoder][0], B, L)
            k3 = {"bound": "tensor", "flops_per_step": k3_fl, "ms_per_step": k3_ms,
                  "achieved": k3_fl / (k3_ms * 1e-3) / 1e12 if k3_ms > 0 else None, "peak": peaks["bf16_tflops"],
                  "unit": "TFLOP/s", "frac": (k3_fl / (k3_ms * 1e-3) / 1e12 / peaks["bf16_tflops"]) if k3_ms > 0 else None,
                  "note": "encoder-layer kernels summed (SURVEY 8(d) K3, FLOP model 3 x (8LH^2+6L^2H+2LH^2+4LHI) per sequence "
                          "and layer); the chain is HBM/issue-bound per kernel, see roofline and DESIGN.md section 4"}
            # K2 on graphs whose tables exceed L2: the gather-fused projection GEMMs, algorithmic bytes (every gathered
            # row + the operands / outputs once) over the live-timed duration, against the measured copy bandwidth
            k2 = None
            if any(k in prof for k in K2_GATHER_FAMILIES):
                k2 = {"bound": "hbm", "peak": peaks["hbm_gbs"], "unit": "GB/s", "kernels": {}}
                for k in K2_GATHER_FAMILIES:
                    if k in prof:
                        v = prof[k]
                        k2["kernels"][k] = {"achieved": v["gbs"], "frac": v["gbs"] / peaks["hbm_gbs"],
                                            "avg_launch_us": 1e3 * v["ms"] / v["calls"], "launches_per_step": v["calls"] / n_prof,
                                            "traffic": load_traffic(workload, B).get(k)}
            res["k2"] = k2
            res.update(roofline=roof, k3=k3,
                       profile={"per_kernel_family": prof, "steps_profiled": n_prof, "sum_ms_per_step": tot / n_prof,
                                "ms_per_step_timed": ms / steps})
    # release everything this workload holds on the device before a second workload is measured
    del tm, args, ds, idx_dev
    torch.cuda.empty_cache()
    return res


def resolve_batch(batch, global_batch, ws):
    """(targets per GPU per step, "weak" | "strong"): --batch fixes the per-GPU work (weak scaling); --global-batch fixes the
    total (SURVEY 8(d) config 3: one strong-scaling run at global B = 8192) and every rank takes its equal share."""
    if not global_batch:
        return batch, "weak"
    if global_batch < ws or global_batch % ws:
        raise SystemExit(f"--global-batch {global_batch} is not a positive multiple of the {ws} ranks")
    return global_batch // ws, "strong"


def ours(a):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    ws = int(os.environ.get("WORLD_SIZE", "1"))
    if ws != a.gpus:
        if ws == 1 and a.gpus > 1:
            raise SystemExit("launch multi-GPU runs with torch.distributed.run (one process per GPU)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: pmgt_b200 has no CPU fallback (use --impl reference for the CPU port)")
    a.batch, scaling = resolve_batch(a.batch, a.global_batch, ws)

    # baselines first (rank 0, N = 1 only), each in its own subprocess, so they never overlap the GPU timing
    cpu, gpu_eager = None, None
    if rank == 0 and ws == 1 and not a.no_cpu_baseline:
        wl = "TG" if a.workload == "1M" else a.workload
        d = run_cpu_port(wl, steps=2, warmup=0, budget_s=20.0)
        cpu = {"value": d["value"], "unit": "contexts/s", "cores": d["cores"], "kind": d["kind"],
               "sample": f"{d['targets_per_step']} targets x {d['steps']} steps of the {wl} workload (same encoder / hops / "
                         f"pairs; the graph only changes which rows are touched) "
                         f"(sampler in {d['cores']} worker processes: {d['sampler_contexts_per_s']:.0f} ctx/s; fp32 torch model "
                         f"{d['cores']} threads: {d['model_contexts_per_s']:.0f} ctx/s; "
                         + ("unmodified reference modules" if d["kind"] == "reference" else "oracle port") + ")"}
    if rank == 0 and ws == 1 and not a.no_gpu_baseline:
        try:
            g = run_gpu_eager("TG" if a.workload == "1M" else a.workload, 256, steps=2, warmup=1, device_index=local_rank)
            gpu_eager = {"value": g["value"], "unit": "contexts/s", "ms_per_step": g["ms_per_step"], "kind": "port-eager-on-gpu",
                         "targets_per_step": g["targets_per_step"], "dtype": "f32", "pair_encode": g["pair_encode"],
                         "sample": f"{g['steps']} steps of {g['targets_per_step']} targets (the reference's batch) on the "
                                   f"{g['workload']} graph, stock PyTorch ops on this GPU, sampler excluded"}
        except Exception as e:  # the baseline is a courtesy number; never lose the bench line over it
            gpu_eager = {"unavailable": str(e)[-300:]}

    torch.cuda.set_device(local_rank)
    if ws > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    main_res = measure(a, a.workload, a.steps, a.warmup, True, rank, local_rank, ws, dev, dump_dir=a.dump_outputs)
    if rank == 0 and a.profile_out and main_res["profile"]:
        with open(a.profile_out, "w") as f:
            json.dump(main_res["profile"], f, indent=1)

    second = None
    if ws == 1 and a.workload == "1M" and a.encoder == "default" and not a.no_secondary:
        # BASELINE config 2 (TG-shaped graph, one B200) beside the headline: tables fit in L2, projected-table mode
        r2 = measure(a, "TG", min(a.steps, 50), min(a.warmup, 5), False, rank, local_rank, ws, dev)
        second = {"config": workload_config("TG", a.batch, "gpu", a.encoder), "value": r2["value"], "unit": "contexts/s",
                  "ms_per_step": r2["ms_per_step"], "e2e": r2["e2e_value"], "gpu_launches": r2["launches"],
                  "loss_last": r2["loss_last"]}

    if rank == 0:
        B = a.batch
        line = {
            "metric": "pmgt_pretrain_node_contexts_per_s", "value": main_res["value"], "unit": "contexts/s", "n_gpus": ws,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": main_res["ms_per_step"], "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(a.workload, B, "gpu", a.encoder),
            "e2e": {"value": main_res["e2e_value"], "unit": "contexts/s", "h2d_bytes_per_step": B * 8, "d2h_bytes_per_step": 4,
                    "api": "pmgt_b200.trainer.PMGTTrainerModel.train_on_indices(pinned host index batch) + .last_loss() every step"},
            "gpu_launches": main_res["launches"], "clocks": main_res["clocks"], "roofline": main_res["roofline"],
            "roofline_k3": main_res["k3"], "roofline_k2": main_res["k2"], "cpu_baseline": cpu, "gpu_baseline": gpu_eager, "loss_last": main_res["loss_last"],
            "config2_TG": second,
        }
        print(json.dumps(line), flush=True)
    if ws > 1:
        dist.destroy_process_group()


def main():
    a = parse()
    if a.impl == "reference":
        reference_arm(a)
    elif a.impl == "reference-gpu":
        reference_gpu_arm(a)
    else:
        ours(a)


if __name__ == "__main__":
    main()
