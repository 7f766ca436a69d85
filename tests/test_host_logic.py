"""CPU-only tests of the host-side mirror of the reference API: state-dict keys, config, collate,
ModelOutput indexing, synthetic inputs, graph ingestion, embedding remap."""
import os

import numpy as np
import pytest
import torch

from pmgt_b200 import PMGT, PMGTConfig, pmgt_collate_fn, synthetic
from pmgt_b200.graph import ItemGraph
from pmgt_b200.modeling_pmgt import FlatParams, PMGTForPreTrainingOutput, encoder_param_order
from pmgt_b200.utils import remap_node_embeddings


def test_state_dict_keys_match_reference_golden(golden_dir):
    g = torch.load(os.path.join(golden_dir, "model_golden.pt"), weights_only=False)["default"]
    net = PMGT(g["node_size"], config=PMGTConfig())
    trainable = {n for n, p in net.named_parameters() if p.requires_grad}
    assert trainable == set(g["grad_norms"].keys())            # the reference's 104 trainable tensors, same names
    sd = net.state_dict()
    assert {"feat_embeddings.0.weight", "feat_embeddings.1.weight", "bert.embeddings.position_ids",
            "bert.embeddings.role_ids"} <= set(sd)
    assert sum(p.numel() for p in net.parameters() if p.requires_grad) == 1_186_690
    assert not any(p.requires_grad for p in net.feat_embeddings.parameters())


@pytest.mark.parametrize("name", ["default", "multihead"])
def test_state_dict_layout_and_roundtrip_match_reference_golden(golden_dir, name):
    """The reference's state-dict layout as tests/golden/make_golden.py certified it: the reference loaded
    model_ref.init_state_dict(cfg) with strict=False (any shape mismatch raises) with no unexpected key and only the
    position_ids / role_ids buffers missing, and its named_parameters() order is the key order of grad_norms."""
    from oracle import model_ref
    g = torch.load(os.path.join(golden_dir, "model_golden.pt"), weights_only=False)[name]
    cfg = g["cfg"]
    ref_sd = model_ref.init_state_dict(cfg, g["node_size"], seed=g["weights_seed"], perturb=g["weights_perturb"])
    config = PMGTConfig(hidden_size=cfg["hidden_size"], feat_hidden_sizes=cfg["feat_hidden_sizes"],
                        num_hidden_layers=cfg["num_hidden_layers"], num_attention_heads=cfg["num_attention_heads"],
                        intermediate_size=cfg["intermediate_size"], beta=cfg["beta"])
    ours = PMGT(g["node_size"], cfg["random_node_ratio"], cfg["mask_node_ratio"], config,
                feat_init_emb=[ref_sd[f"feat_embeddings.{m}.weight"].numpy() for m in range(2)])
    assert [n for n, p in ours.named_parameters() if p.requires_grad] == list(g["grad_norms"])
    sd = ours.state_dict()
    assert set(sd) == set(ref_sd) | {"bert.embeddings.position_ids", "bert.embeddings.role_ids"}
    for k, v in ref_sd.items():
        assert sd[k].shape == v.shape and sd[k].dtype == v.dtype, (k, sd[k].shape, sd[k].dtype, v.shape, v.dtype)
    missing, unexpected = ours.load_state_dict(ref_sd, strict=False)   # reference checkpoint -> ours
    assert not unexpected and sorted(missing) == ["bert.embeddings.position_ids", "bert.embeddings.role_ids"]
    back = ours.state_dict()                                            # and back out, unchanged
    for k, v in ref_sd.items():
        assert torch.equal(back[k], v), k


@pytest.mark.needs_reference
def test_state_dict_roundtrip_with_live_reference():
    from oracle import ref_shim
    R = ref_shim.load()
    ref = R.PMGT(30, config=R.PMGTConfig(num_hidden_layers=2))
    ours = PMGT(30, config=PMGTConfig(num_hidden_layers=2))
    assert list(ref.state_dict().keys()) == list(ours.state_dict().keys())
    ours.load_state_dict(ref.state_dict())          # reference checkpoint -> ours
    ref.load_state_dict(ours.state_dict())          # and back
    for (k1, v1), (k2, v2) in zip(ref.state_dict().items(), ours.state_dict().items()):
        assert k1 == k2 and v1.shape == v2.shape and v1.dtype == v2.dtype


def test_config_defaults_and_validation():
    c = PMGTConfig()
    assert (c.hidden_size, c.feat_hidden_sizes, c.num_hidden_layers, c.num_attention_heads, c.intermediate_size) == \
        (128, [1536, 768], 5, 1, 128)
    assert (c.hidden_dropout_prob, c.attention_probs_dropout_prob, c.max_position_embeddings, c.layer_norm_eps, c.beta) == \
        (0.1, 0.1, 100, 1e-12, 0.5)
    assert c.use_return_dict and not c.output_attentions and c.chunk_size_feed_forward == 0
    with pytest.raises(ValueError, match="not a multiple of the number of attention"):
        PMGTConfig(hidden_size=100, num_attention_heads=3)


def test_flat_param_order_makes_qkvc_one_matrix():
    net = PMGT(10, config=PMGTConfig(hidden_size=32, intermediate_size=64, num_hidden_layers=2, num_attention_heads=2))
    order = encoder_param_order(net.bert, "bert.") + net.nfr_loss.param_order("nfr_loss.")
    fp = FlatParams(order)
    assert len(order) == sum(1 for p in net.parameters() if p.requires_grad)
    o = fp.offsets
    H = 32
    for i in range(2):
        p = f"bert.encoder.layer.{i}.attention.self."
        assert o[p + "key.weight"] - o[p + "query.weight"] == H * H
        assert o[p + "ctx_attention.weight"] - o[p + "query.weight"] == 3 * H * H
        assert o[p + "ctx_attention.bias"] - o[p + "query.bias"] == 3 * H
    assert all(v % 8 == 0 for v in o.values())


def test_model_output_indexing_like_transformers():
    out = PMGTForPreTrainingOutput(loss=None, prediction_logits=None, last_hidden_state=torch.zeros(2, 6, 4))
    assert out[0] is out.last_hidden_state                       # inference: net(x)[0] (trainer.py:153-154)
    out = PMGTForPreTrainingOutput(loss=torch.tensor(1.0), prediction_logits=torch.zeros(3), last_hidden_state=torch.zeros(1))
    assert out[0] is out.loss and out[1] is out.prediction_logits and out["loss"] is out.loss and len(out) == 3


def test_forward_asserts_like_the_reference():
    net = PMGT(10, config=PMGTConfig(num_hidden_layers=1))
    x = {"node_ids": torch.zeros(1, 6, dtype=torch.long), "attention_mask": torch.ones(1, 6)}
    with pytest.raises(AssertionError, match="labels must be passed"):
        net(x, x)
    with pytest.raises(AssertionError, match="num_pairs must be passed"):
        net(x, x, labels=torch.zeros(1))


def test_prepare_inputs_layout_matches_the_reference_order():
    """PMGT.prepare_inputs (what the trainer's prefetch builds on the side stream): the batched encoder input is
    [targets | pairs | masked targets] (models.py:104-162 encodes them in that order), the pair offsets are the running
    sum of num_pairs, and the NFR rows point at the masked positions inside the masked-target block of the compact
    hidden matrix [all target positions | position 0 of every pair | all masked-target positions]."""
    torch.manual_seed(3)
    B, L, P = 4, 6, 3
    net = PMGT(50, config=PMGTConfig(num_hidden_layers=1))
    t = {"node_ids": torch.randint(2, 52, (B, L)), "attention_mask": torch.ones(B, L)}
    num_pairs = torch.tensor([3, 1, 2, 3])
    SP = int(num_pairs.sum())
    p = {"node_ids": torch.randint(2, 52, (SP, L)), "attention_mask": torch.ones(SP, L)}
    masked = net.mask_nodes(t["node_ids"], with_positions=True)
    m_ids, m_mask, target_idx, m_pos = masked
    prep = net.prepare_inputs(t, p, num_pairs, masked)
    assert torch.equal(prep["ids_all"].view(-1, L), torch.cat([t["node_ids"], p["node_ids"], m_ids]))
    assert torch.equal(prep["mask_all"], torch.cat([t["attention_mask"], p["attention_mask"], t["attention_mask"]]))
    assert prep["pair_off"].tolist() == [0, 3, 4, 6, 9]
    assert torch.equal(prep["target_ids"], target_idx)
    # masked positions: row b, position 1 + j of the masked-target block that starts after B * L + SP compact rows
    rows = prep["nfr_rows"]
    assert rows.numel() == int(m_mask.sum()) == m_pos.shape[0]
    for k in range(rows.numel()):
        b, j = int(m_pos[k, 0]), int(m_pos[k, 1])
        assert int(rows[k]) == B * L + SP + b * L + 1 + j
        assert int(m_ids[b, 1 + j]) == 1                        # the <mask> index sits exactly there
    # without the precomputed positions (the 3-tuple the reference-style mask_nodes returns) the result is the same
    prep2 = net.prepare_inputs(t, p, num_pairs, masked[:3])
    assert all(torch.equal(prep[k], prep2[k]) for k in prep)


def test_collate_layout():
    L = 6
    item = lambda p: ((torch.arange(L), torch.ones(L)), (torch.zeros(p, L, dtype=torch.long), torch.ones(p, L)), torch.ones(p))
    t, p, n, lab = pmgt_collate_fn([item(10), item(7)])
    assert t["node_ids"].shape == (2, L) and p["node_ids"].shape == (17, L) and n.tolist() == [10, 7] and lab.shape == (17,)
    assert n.dtype == torch.int64
    inf = pmgt_collate_fn([((torch.arange(L), torch.ones(L)),)] * 3)
    assert set(inf) == {"node_ids", "attention_mask"} and inf["node_ids"].shape == (3, L)


def test_synthetic_graph_shapes_and_weights():
    g = synthetic.make_item_graph("VG")
    assert g.num_nodes == 7252 and g.num_edges_directed == 2 * 88606
    assert len(g.isolated_nodes()) == 0
    deg = np.diff(g.indptr)[2:]
    assert deg.max() > 20 * np.median(deg)                       # heavy tail
    assert g.weights.min() > 0 and np.all(g.cdf <= 1.0) and np.all(g.cdf > 0)
    # undirected: every (u, v) has its (v, u)
    rows = np.repeat(np.arange(len(g.indptr) - 1), np.diff(g.indptr))
    fwd = set(zip(rows[:2000].tolist(), g.indices[:2000].tolist()))
    allp = set(zip(rows.tolist(), g.indices.tolist()))
    assert all((v, u) in allp for u, v in fwd)
    f = synthetic.make_features(100, dims=(16, 8), seed=1)
    assert f[0].shape == (102, 16) and not f[0][:2].any() and abs(float(f[0][2:].std()) - 1) < 0.1


def test_item_graph_validation():
    with pytest.raises(ValueError):
        ItemGraph(3, np.array([0, 0, 1, 1, 1, 1]), np.array([3]), np.array([1.0]))   # row 1 (<mask>) not empty
    with pytest.raises(ValueError):
        ItemGraph(3, np.array([0, 0, 0, 1, 1, 1]), np.array([9]), np.array([1.0]))   # neighbour id out of range


def test_remap_node_embeddings_like_load_node_init_emb():
    emb = np.arange(12, dtype=np.float32).reshape(3, 4) + 1
    np.random.seed(0)
    out = remap_node_embeddings(["b", "zz", "a"], ["a", "b", "c"], emb, normalize=True)
    assert np.allclose(out[0], emb[1] / np.linalg.norm(emb[1])) and np.allclose(out[2], emb[0] / np.linalg.norm(emb[0]))
    assert np.isclose(np.linalg.norm(out[1]), 1.0)               # missing item: random row, normalised
    assert out.dtype == np.float32


def test_edge_list_duplicates_follow_networkx_semantics():
    """nx.Graph keeps one edge per unordered pair: a repeated (u, v) updates the weight in place (first position in the
    adjacency lists, last weight) -- ItemGraph.from_edge_list must build the same CSR (ADVICE r1)."""
    import networkx as nx
    import numpy as np
    from pmgt_b200.graph import ItemGraph
    edges = [(2, 3, 0.5), (3, 4, 1.0), (3, 2, 0.9), (4, 5, 0.2), (2, 3, 0.1), (5, 2, 0.7), (4, 3, 0.3)]
    g = nx.Graph()
    g.add_nodes_from(range(2, 6))
    g.add_weighted_edges_from(edges)
    a = ItemGraph.from_networkx(g)
    b = ItemGraph.from_edge_list(4, np.array([e[0] for e in edges]), np.array([e[1] for e in edges]),
                                 np.array([e[2] for e in edges]))
    assert np.array_equal(a.indptr, b.indptr) and np.array_equal(a.indices, b.indices)
    assert np.allclose(a.weights, b.weights) and np.array_equal(a.cdf, b.cdf)


def test_bench_batch_resolution_weak_and_strong():
    """bench.py: --batch is per GPU (weak scaling); --global-batch is the total of a step, split evenly (strong scaling,
    SURVEY 8(d) config 3)."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(os.path.dirname(__file__)), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    assert bench.resolve_batch(4096, 0, 8) == (4096, "weak")
    assert bench.resolve_batch(4096, 8192, 1) == (8192, "strong")
    assert bench.resolve_batch(4096, 8192, 8) == (1024, "strong")
    with pytest.raises(SystemExit):
        bench.resolve_batch(4096, 8190, 4)
    with pytest.raises(SystemExit):
        bench.resolve_batch(4096, 4, 8)


def test_bench_argument_checks(tmp_path, monkeypatch):
    """bench.py: --steps is the number of timed steps and must be at least 1; --dump-outputs belongs to --impl ours."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(os.path.dirname(__file__)), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    monkeypatch.setattr("sys.argv", ["bench.py", "--steps", "7", "--dump-outputs", str(tmp_path)])
    assert bench.parse().steps == 7
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        monkeypatch.setattr("sys.argv", ["bench.py", *argv])
        with pytest.raises(SystemExit):
            bench.parse()


@pytest.mark.parametrize("n,batch,ws", [(1000, 128, 1), (1000, 128, 4), (130, 64, 8), (64, 64, 2), (10, 64, 4)])
def test_epoch_batches_cover_every_target_once_and_keep_ranks_in_step(n, batch, ws):
    """trainer.epoch_batches: the reference's DataLoader keeps the partial last batch (shuffle=True, drop_last=False,
    trainer.py:90-103).  Over the ranks an epoch visits every training target, full global batches exactly once; every
    rank runs the same number of steps (the gradient exchange is collective); the shards of one step never overlap
    except for the one target a rank with an empty tail share repeats."""
    from pmgt_b200 import trainer
    perm = trainer.epoch_permutation(n, 0, 3)
    assert sorted(perm.tolist()) == list(range(n))
    per_rank = [trainer.epoch_batches(n, batch, r, ws, perm) for r in range(ws)]
    steps = {len(b) for b in per_rank}
    assert len(steps) == 1
    n_steps = steps.pop()
    full = n // (batch * ws)
    assert n_steps == full + (1 if n % (batch * ws) else 0)
    seen = []
    for step in range(n_steps):
        shards = [per_rank[r][step] for r in range(ws)]
        assert all(len(s) > 0 for s in shards)
        if step < full:
            assert all(len(s) == batch for s in shards)
            cat = np.concatenate(shards)
            assert len(set(cat.tolist())) == batch * ws
            np.testing.assert_array_equal(cat, perm[step * batch * ws:(step + 1) * batch * ws])
        seen.extend(np.concatenate(shards).tolist())
    assert set(seen) == set(range(n))
    # only the tail step may repeat a target (ranks without a share of a short tail)
    assert len(seen) - n <= max(0, ws - 1)


def test_trainer_check_args_error_behaviour_like_the_reference():
    """trainer.check_args (reference trainer.py:213-218 + base_trainer.py check_args): same refusals, plus the two flags
    this implementation cannot honour (fp16 autocast, LR schedulers) raise instead of being ignored; init_run refuses to
    train without a CUDA device (no CPU fallback)."""
    from pmgt_b200 import trainer
    trainer.check_args(trainer.make_args(synthetic="TG"))
    trainer.check_args(trainer.make_args(synthetic="TG", accumulation_step=4))
    for bad in (dict(early_criterion="ndcg"), dict(model_name="NCF"), dict(optim="sgd"), dict(scheduler_type="linear"),
                dict(mp_enabled=True), dict(accumulation_step=0)):
        with pytest.raises(ValueError):
            trainer.check_args(trainer.make_args(synthetic="TG", **bad))
    with pytest.raises(ValueError):
        trainer.check_args(trainer.make_args(dataset_name="Amazon"))
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            trainer.init_run(trainer.make_args(synthetic="TG"))
