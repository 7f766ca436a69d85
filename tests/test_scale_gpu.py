"""Parity at the sizes the benchmark runs (VERDICT round 1, "scale-parity"):

 * the whole pre-training step against the fp32 oracle on the same GPU at BASELINE config 2's full size (TG-shaped
   graph, 4096 targets = 49,152 encoded sequences = 2,304 token tiles: every persistent kernel wraps around its 148 CTAs
   ~16 times) and on the 1M-node graph (gather-fused projection GEMMs, out-of-L2 sampler);
 * the dual-softmax attention core at 60,000 sequences (its 148-CTA x 12/16-warp loop wraps ~25 times);
 * two NCCL ranks driving ``PMGTTrainerModel.train_on_indices``: parameters identical across ranks after the step and
   equal to one process that averages the two shard gradients (what DDP computes; SURVEY section 4 "distributed").

Tolerances are the ones stated in tests/test_model_gpu.py (bf16 operands / activations vs the fp32 reference).
"""
import math
import os
import socket

import numpy as np
import pytest
import torch

from oracle import model_ref

pytestmark = pytest.mark.gpu
BF16 = torch.bfloat16


def _check_grads(net, ref_grads, cos_min=0.995, norm_tol=0.05):
    for name, p in net.named_parameters():
        if not p.requires_grad:
            continue
        assert p.grad is not None, name
        want = ref_grads[name].float()
        got = p.grad.float()
        assert torch.isfinite(got).all(), name
        wn = float(want.norm())
        if wn < 1e-6:
            assert float(got.norm()) < 1e-4, (name, float(got.norm()))
            continue
        cos = float((got * want).sum() / (got.norm() * want.norm()).clamp_min(1e-20))
        assert cos >= cos_min, f"{name}: cosine {cos:.5f}"
        assert abs(float(got.norm()) / wn - 1) <= norm_tol, f"{name}: norm ratio {float(got.norm()) / wn:.4f}"


def _full_step_vs_oracle(graph, tables_dev, B, seed):
    """One training step of pmgt_b200.PMGT (dropout 0) on a sampled batch vs the fp32 oracle on the same device."""
    from pmgt_b200 import PMGT, PMGTConfig, PMGTDataset
    cfg = model_ref.default_cfg()
    node_size = graph.num_nodes
    sd = model_ref.init_state_dict(cfg, node_size, feats=[torch.zeros(1, 1536), torch.zeros(1, 768)], seed=seed, perturb=0.05)
    for m in range(2):
        del sd[f"feat_embeddings.{m}.weight"]
    net = PMGT(node_size, cfg["random_node_ratio"], cfg["mask_node_ratio"],
               PMGTConfig(hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0), feat_init_emb=tables_dev)
    missing, unexpected = net.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    net = net.cuda().train()
    ds = PMGTDataset(graph, seed=3)
    idx = torch.from_numpy(np.random.default_rng(seed).permutation(len(ds))[:B])
    batch = ds.sample_batch(idx, epoch=1)
    torch.manual_seed(5)
    masked = net.mask_nodes(batch[0]["node_ids"])
    out = net(*batch, masked_inputs=masked)
    out.loss.backward()

    sdc = {k: v.cuda() for k, v in sd.items()}
    for m in range(2):  # the oracle sees the same bf16-rounded feature rows the kernels gather
        sdc[f"feat_embeddings.{m}.weight"] = tables_dev[m].to(BF16).float()
    params = {k: v.requires_grad_(True) for k, v in sdc.items() if not k.startswith("feat_embeddings")}
    ref = model_ref.pretrain_forward(sdc, cfg, node_size, *batch, training=True, masked=masked)
    ref["loss"].backward()
    assert abs(float(out.loss) - float(ref["loss"])) <= 2e-2 * abs(float(ref["loss"])), (float(out.loss), float(ref["loss"]))
    assert float((out.prediction_logits - ref["prediction_logits"]).abs().max()) < 3e-2
    rh = ref["last_hidden_state"].detach()
    assert out.last_hidden_state.shape == rh.shape
    assert float((out.last_hidden_state - rh).abs().max()) < 3e-2 * float(rh.abs().max())
    _check_grads(net, {k: v.grad for k, v in params.items()})


def test_full_size_step_matches_oracle_config2():
    """BASELINE config 2 at the bench size: 4096 targets, 45,056 sampled contexts, 49,152 encoded sequences."""
    from pmgt_b200 import synthetic
    g = synthetic.make_item_graph("TG")
    feats = [torch.from_numpy(f).cuda() for f in synthetic.make_features(g.num_nodes, seed=1235)]
    _full_step_vs_oracle(g, feats, 4096, seed=1)


def test_step_matches_oracle_on_the_1m_graph():
    """BASELINE config 3's graph (1M nodes / 20M edges): gather-fused projection GEMMs (no projected tables), CSR + CDF
    far beyond L2.  1024 targets keep the fp32 oracle's activations small next to its 9.2 GB fp32 tables."""
    from pmgt_b200 import modeling_pmgt, synthetic
    g = synthetic.make_item_graph("1M")
    feats = synthetic.make_features_device(g.num_nodes, seed=1236, device="cuda")
    assert modeling_pmgt.PROJECTION_MODE == "auto"
    _full_step_vs_oracle(g, feats, 1024, seed=2)


def test_attention_core_at_60000_sequences():
    from pmgt_b200 import ops
    R, L, H, heads, beta = 60000, 6, 128, 1, 0.5
    T = R * L
    gen = torch.Generator(device="cuda").manual_seed(9)
    qkvc = (torch.randn(T, 4 * H, device="cuda", generator=gen) * 0.7).to(BF16)
    n_real = torch.randint(1, L, (R,), device="cuda", generator=gen)
    mask = (torch.arange(L, device="cuda")[None, :] <= n_real[:, None]).float()
    ctx = torch.empty(T, H, device="cuda", dtype=BF16)
    ops.attn_core_fwd(ops.attn_args(R, L, H, heads, beta, qkvc, mask, 0.0, 0, 0, ctx=ctx))
    x = qkvc.float().requires_grad_(True)
    q, k, v, c = [x[:, i * H:(i + 1) * H].view(R, L, heads, H).permute(0, 2, 1, 3) for i in range(4)]
    ext = (1.0 - mask[:, None, None, :]) * -10000.0
    n = torch.linalg.norm(c, dim=-1, keepdim=True)
    s1 = 1.0 - (c @ c.transpose(-1, -2)) / (n @ n.transpose(-1, -2)) + torch.eye(L, device="cuda")
    p1 = torch.softmax(s1 + ext, -1)
    p2 = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(H) + ext, -1)
    want = ((beta * p1 + (1 - beta) * p2) @ v).permute(0, 2, 1, 3).reshape(T, H)

    def close(got, ref, tol, name):
        scale = ref.abs().max().clamp_min(1e-6)
        assert torch.isfinite(got.float()).all(), name
        err = float((got.float() - ref).abs().max() / scale)
        assert err < tol, f"{name}: max scaled error {err:.4g}"

    close(ctx, want.detach(), 1e-2, "ctx")
    dctx = (torch.randn(T, H, device="cuda", generator=gen)).to(BF16)
    want.backward(dctx.float())
    dqkvc = torch.empty_like(qkvc)
    ops.attn_core_bwd(ops.attn_args(R, L, H, heads, beta, qkvc, mask, 0.0, 0, 0, dctx=dctx, dqkvc=dqkvc))
    for i, nm in enumerate("qkvc"):
        close(dqkvc[:, i * H:(i + 1) * H], x.grad[:, i * H:(i + 1) * H], 1.5e-2, "d" + nm)


# ---------------------------------------------------------------------------------------------------
# two NCCL ranks through the trainer
# ---------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _make_trainer(dev, B):
    from pmgt_b200 import trainer
    args = trainer.make_args(synthetic="VG", train_batch_size=B, seed=0, num_hidden_layers=2, hidden_dropout_prob=0.0,
                             attention_probs_dropout_prob=0.0, gradient_max_norm=1.0)
    args.device = dev
    trainer.set_seed(0)
    args.graph, args.feat_init_emb = trainer._load_graph_and_features(args)
    trainer.init_dataloader(args)
    trainer.init_model(args)
    return trainer, args, trainer.PMGTTrainerModel(args)


def _dp_worker(rank, ws, port, q, symm_reduce):
    import torch.distributed as dist
    try:
        os.environ["PMGT_SYMM_REDUCE"] = "1" if symm_reduce else "0"
        torch.cuda.set_device(rank)
        dev = torch.device("cuda", rank)
        B = 96
        # ---- reference: one process, the two shard gradients averaged (what DDP's mean-of-rank-losses computes)
        trainer, args, tm = _make_trainer(dev, B)
        ds = args.train_dataset
        perm = trainer.epoch_permutation(len(ds), 0, 0)
        shards = [trainer.shard_indices(perm, 0, B, r, ws) for r in range(ws)]
        tm.net.train()
        for r in range(ws):
            torch.manual_seed(100 + r)
            batch = ds.sample_batch(shards[r], epoch=0)
            masked = tm.net.mask_nodes(batch[0]["node_ids"], with_positions=True)
            tm.net(*batch, masked_inputs=masked)[0].backward()
        ref_grad = torch.cat([p.grad.reshape(-1) for p in tm.net.parameters() if p.requires_grad]).clone() / ws
        # ---- data-parallel step through the trainer
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=dev)
        trainer2, args2, tm2 = _make_trainer(dev, B)
        assert trainer2.world() == (rank, ws)
        p0 = torch.cat([p.detach().reshape(-1) for p in tm2.net.parameters() if p.requires_grad]).clone()
        torch.manual_seed(100 + rank)
        tm2.prefetch(args2.train_dataset, shards[rank], 0)
        loss = tm2.train_on_indices(args2.train_dataset, shards[rank], 0)
        torch.cuda.synchronize()
        assert torch.isfinite(loss)
        # which exchange ran: the in-place peer reduction over symmetric memory, or NCCL
        arena = tm2.net._flat()._step_arena
        assert (arena.symm is not None) == bool(symm_reduce), (arena.symm, symm_reduce)
        fv = tm2.optimizer.flat_views()
        dp_grad = fv[1].clone() / ws          # allreduced (sum) flat gradient
        p1 = torch.cat([p.detach().reshape(-1) for p in tm2.net.parameters() if p.requires_grad])
        # identical across ranks, bit for bit
        gathered = [torch.empty_like(p1) for _ in range(ws)]
        dist.all_gather(gathered, p1)
        assert all(torch.equal(gathered[0], g) for g in gathered), "replicas diverged"
        assert float((p1 - p0).abs().max()) > 1e-4, "the step did not move the parameters"
        # equal to the single-process average of the shard gradients (flat layouts: same parameter order)
        names = [n for n, p in tm2.net.named_parameters() if p.requires_grad]
        assert dp_grad.numel() >= ref_grad.numel()
        off_ok = 0
        fp = tm2.net._flat()
        for n, p in tm.net.named_parameters():
            if not p.requires_grad:
                continue
            o = fp.offsets[n]
            got = dp_grad[o: o + p.numel()]
            want = p.grad.reshape(-1) / ws
            wn = float(want.norm())
            if wn < 1e-7:
                continue
            cos = float((got * want).sum() / (got.norm() * want.norm()).clamp_min(1e-30))
            assert cos > 0.9995, (n, cos)
            assert abs(float(got.norm()) / wn - 1) < 1e-2, (n, float(got.norm()) / wn)
            off_ok += 1
        assert off_ok >= 40 and len(names) >= 40, (off_ok, len(names))
        q.put((rank, "ok"))
    except Exception as e:  # pragma: no cover
        import traceback
        q.put((rank, repr(e) + traceback.format_exc()[-1500:]))
    finally:
        try:
            import torch.distributed as dist
            if dist.is_initialized():
                dist.destroy_process_group()
        except Exception:
            pass


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("symm_reduce", [True, False])
def test_two_nccl_ranks_end_the_step_with_identical_parameters(symm_reduce):
    """Two ranks of the product end a step with bit-identical parameters equal to one GPU on the concatenated batch --
    through the symmetric-memory peer reduction (csrc/peer_reduce.cu) and through the NCCL all-reduce."""
    import torch.multiprocessing as mp
    ws = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, ws, port, q, symm_reduce)) for r in range(ws)]
    for p in procs:
        p.start()
    res = [q.get(timeout=600) for _ in range(ws)]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, "ok"), (1, "ok")], res
