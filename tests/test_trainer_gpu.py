"""End-to-end run of the trainer entry points (pmgt/pmgt/trainer.py:209-275, train.py:298-344) on a small synthetic
item graph: train with early-stopping bookkeeping and checkpoints, validation AUC, test, resume, and the embedding export
(bulk inference, BASELINE config 4's consumer format) with its downstream remap (pmgt/pmgt/utils.py:15-40)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _args(tmp_path, **over):
    from pmgt_b200 import trainer
    kw = dict(synthetic=(400, 3000), train_batch_size=64, test_batch_size=128, num_epochs=2, num_hidden_layers=2, seed=3,
              log_dir=str(tmp_path), lr=2e-3, early=5)
    kw.update(over)
    return trainer.make_args(**kw)


def test_train_validate_test_and_resume(tmp_path):
    from pmgt_b200 import trainer
    args = _args(tmp_path, gradient_max_norm=1.0)
    trainer.check_args(args)
    trainer.init_run(args)
    trainer.init_dataloader(args)
    trainer.init_model(args)
    best, tm = trainer.train(args)
    assert len(args.history) == 2
    for h in args.history:
        assert np.isfinite(h["loss/train"]) and np.isfinite(h["loss/val"]) and 0.0 <= h["val/auc"] <= 1.0
    assert args.history[-1]["loss/train"] < args.history[0]["loss/train"] + 0.05
    assert best == min(h["loss/val"] for h in args.history)
    assert args.best_model_path and os.path.exists(args.best_model_path)
    res = trainer.test(args, tm)
    assert 0.0 <= res["test/auc"] <= 1.0
    # the checkpoint carries the reference's key layout (Lightning prefixes everything with "net.")
    ckpt = torch.load(args.best_model_path, map_location="cpu", weights_only=False)
    keys = ckpt["state_dict"].keys() if "state_dict" in ckpt else ckpt.keys()
    assert any(k.endswith("bert.encoder.layer.0.attention.self.ctx_attention.weight") for k in keys)
    # a fresh trainer restored from it evaluates to the same validation loss (deterministic eval: same sampler keys)
    args2 = _args(tmp_path)
    trainer.init_run(args2)
    trainer.init_dataloader(args2)
    trainer.init_model(args2)
    tm2 = trainer.PMGTTrainerModel(args2)
    tm2.load_state_dict(ckpt)
    b = tm2.evaluate(args2.valid_dataset, 128)
    tm.load_state_dict(ckpt)  # `tm` holds the LAST epoch's weights until the best checkpoint is loaded back
    a = tm.evaluate(args.valid_dataset, 128)
    assert abs(a["loss"] - b["loss"]) <= 1e-5 * abs(a["loss"]) + 1e-6 and abs(a["auc"] - b["auc"]) <= 1e-6


def test_inference_export_and_downstream_remap(tmp_path):
    from pmgt_b200 import PMGTDataset, trainer
    from pmgt_b200.utils import remap_node_embeddings
    path = os.path.join(str(tmp_path), "emb", "node_emb.npy")
    args = _args(tmp_path, mode="inference", inference_result_path=path, test_batch_size=96)
    trainer.check_args(args)
    trainer.init_run(args)
    trainer.init_dataloader(args)
    trainer.init_model(args)
    emb = trainer.inference(args)
    n = len(args.graph)
    assert emb.shape == (n, args.hidden_size) and emb.dtype == np.float32 and np.isfinite(emb).all()
    assert np.array_equal(np.load(path), emb)                      # base_trainer.py:400-407: .npy in node order
    # row i is node id i + 2: recompute a few rows directly through the model
    ds = PMGTDataset(args.graph, is_training=False, is_inference=True, seed=args.seed)
    args.model.eval()
    with torch.no_grad():
        direct = args.model(ds.sample_batch(np.array([0, 7, n - 1])))[0][:, 0].cpu().numpy()
    assert np.allclose(direct, emb[[0, 7, n - 1]], rtol=0, atol=1e-6)
    # downstream loader: node order -> item order, N(0,1) rows for items outside the graph, unit rows
    node_classes = np.array([f"item{i}" for i in range(n)])
    item_classes = np.concatenate([node_classes[::-1][:50], np.array(["cold-start-item"])])
    out = remap_node_embeddings(item_classes, node_classes, emb, normalize=True)
    assert out.shape == (51, args.hidden_size)
    assert np.allclose(np.linalg.norm(out, axis=1), 1.0, atol=1e-5)
    want = emb[n - 1] / np.linalg.norm(emb[n - 1])
    assert np.allclose(out[0], want, atol=1e-6)


def test_prefetch_and_early_loss_readback(tmp_path):
    """`prefetch` (next batch sampled + corrupted on the side stream) must give the step the same batch it would have
    sampled itself, and `last_loss()` (pinned copy issued after the forward pass) the same number as float(loss)."""
    from pmgt_b200 import trainer
    losses = {}
    for use_prefetch in (False, True):
        args = _args(tmp_path, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
        trainer.init_run(args)
        trainer.init_dataloader(args)
        trainer.init_model(args)
        tm = trainer.PMGTTrainerModel(args)
        ds = args.train_dataset
        shards = [np.arange(s * 64, (s + 1) * 64) for s in range(4)]
        out = []
        for s in range(4):
            loss = tm.train_on_indices(ds, shards[s], epoch=7)
            if use_prefetch and s + 1 < 4:
                tm.prefetch(ds, shards[s + 1], epoch=7)
            host = tm.last_loss()
            assert host == float(loss)
            out.append(host)
        losses[use_prefetch] = out
    # no dropout; the NFR corruption consumes the torch generator once per step in the same order either way
    # -> the two runs are the same computation up to fp32 atomic ordering
    for a, b in zip(losses[False], losses[True]):
        assert abs(a - b) <= 1e-4 * abs(a), (losses[False], losses[True])


def test_resume_restores_optimizer_state_and_epoch(tmp_path):
    """Lightning's fit(ckpt_path=last.ckpt) semantics (base_trainer.py:324-332): weights, AdamW moments + step count,
    epoch counter and early-stopping bookkeeping come back, and training continues at the next epoch."""
    from pmgt_b200 import trainer
    args = _args(tmp_path, run_id="resume_me", num_epochs=2)
    trainer.check_args(args)
    trainer.init_run(args)
    trainer.init_dataloader(args)
    trainer.init_model(args)
    best, tm = trainer.train(args)
    last = os.path.join(str(tmp_path), "resume_me", "checkpoints", "last.ckpt")
    ckpt = torch.load(last, map_location="cpu", weights_only=False)
    assert ckpt["epoch"] == 2 and ckpt["global_step"] == tm.global_step > 0
    fl = tm.optimizer._flat
    m_saved, v_saved = fl["m"].clone(), fl["v"].clone()
    step_saved = tm.optimizer.state[fl["params"][0]]["step"]
    assert step_saved == tm.global_step and float(m_saved.abs().max()) > 0

    args2 = _args(tmp_path, run_id="resume_me", num_epochs=3)
    trainer.init_run(args2)
    trainer.init_dataloader(args2)
    trainer.init_model(args2)
    tm2 = trainer.PMGTTrainerModel(args2)
    tm2.load_state_dict(torch.load(last, map_location=args2.device, weights_only=False))
    assert tm2.epoch == 2 and tm2.global_step == tm.global_step and tm2.best == tm.best
    tm2.net.flat_parameters()                # parameters become views of the flat buffer (normally on the first forward)
    fv = tm2.optimizer.flat_views()          # rebuilds the flat moment buffers from the loaded per-parameter state
    assert fv is not None
    fl2 = tm2.optimizer._flat
    assert torch.equal(fl2["m"], m_saved) and torch.equal(fl2["v"], v_saved)
    assert tm2.optimizer.state[fl2["params"][0]]["step"] == step_saved
    # train() with the same run_id resumes: exactly ONE more epoch (epoch index 2) is run
    best3, tm3 = trainer.train(args2)
    assert [h["epoch"] for h in args2.history] == [2]
    assert tm3.global_step > tm.global_step and tm3.epoch == 3


def test_gradient_accumulation_and_rejected_flags(tmp_path):
    """--accumulation-step (base_trainer.py:315): the optimizer steps every k micro-batches on the mean gradient;
    --mp-enabled (fp16 autocast, base_trainer.py:312) is refused instead of being silently ignored."""
    from pmgt_b200 import trainer
    with pytest.raises(ValueError):
        trainer.check_args(_args(tmp_path, mp_enabled=True))
    args = _args(tmp_path, accumulation_step=2, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    trainer.check_args(args)
    trainer.init_run(args)
    trainer.init_dataloader(args)
    trainer.init_model(args)
    tm = trainer.PMGTTrainerModel(args)
    ds = args.train_dataset
    flat = lambda: torch.cat([p.detach().reshape(-1) for p in tm.net.parameters() if p.requires_grad]).clone()
    p0 = flat()
    tm.train_on_indices(ds, np.arange(0, 64), 0)
    assert tm.global_step == 0 and torch.equal(flat(), p0)          # first micro-batch: gradients only
    g1 = tm.optimizer.flat_views()[1].clone()
    tm.train_on_indices(ds, np.arange(64, 128), 0)
    assert tm.global_step == 1 and not torch.equal(flat(), p0)      # second one: the step
    g2 = tm.optimizer.flat_views()[1]
    assert float((g2 - g1).abs().max()) > 0 and float(g2.norm()) > 0.5 * float(g1.norm())   # accumulated, not replaced
    tm.train_on_indices(ds, np.arange(128, 192), 0)
    assert tm.global_step == 1                                      # gradients were reset, a new cycle started


def test_bench_times_exactly_steps_and_dumps_the_last_timed_loss(tmp_path, monkeypatch):
    """bench.py: after --warmup steps the device-resident series runs exactly --steps steps, and --dump-outputs writes
    the loss the last of them returned (float32 DIR/loss.npy)."""
    import importlib.util
    from pmgt_b200 import trainer
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(os.path.dirname(__file__)), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    dump = tmp_path / "dump"
    monkeypatch.setattr("sys.argv", ["bench.py", "--workload", "VG", "--batch", "64", "--steps", "3", "--warmup", "2",
                                     "--dump-outputs", str(dump)])
    a = bench.parse()
    calls = []
    step = trainer.PMGTTrainerModel.train_on_indices

    def counted(self, dataset, indices, epoch):
        loss = step(self, dataset, indices, epoch)
        calls.append((epoch, float(loss)))
        return loss

    monkeypatch.setattr(trainer.PMGTTrainerModel, "train_on_indices", counted)
    bench.measure(a, a.workload, a.steps, a.warmup, False, 0, 0, 1, torch.device("cuda", 0), dump_dir=a.dump_outputs)
    total = a.warmup + a.steps
    # warmup, the timed device-resident series, then the end-to-end series (as many steps again)
    assert [e for e, _ in calls] == list(range(total)) + list(range(total, total + a.steps))
    got = np.load(dump / "loss.npy")
    assert got.dtype == np.float32 and np.isfinite(got)
    assert float(got) == calls[total - 1][1]
