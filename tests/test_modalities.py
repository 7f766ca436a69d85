"""CPU-only checks of one to four feature modalities: the configuration limit, the flat parameter order, the parameter
counts and state-dict layout against the oracle, and the C ABI of pmgt_embed_multi_args."""
import ctypes
import os
import re
import subprocess
import tempfile

import pytest
import torch

from oracle import model_ref

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def pretrain_forward(sd, cfg, node_size, target_inputs, pair_inputs, num_pairs, labels, training=True, masked=None):
    """The oracle's PMGT.forward (oracle/model_ref.pretrain_forward, models.py:56-176) for any number of modalities:
    the same building blocks, with every feature table of ``cfg["feat_hidden_sizes"]`` gathered.  Returns dict(loss,
    prediction_logits, last_hidden_state)."""
    n = len(cfg["feat_hidden_sizes"])
    t_ids, t_mask = target_inputs["node_ids"], target_inputs["attention_mask"]
    h_t = model_ref.encode(sd, model_ref.gather_feats(sd, t_ids, n), t_mask, cfg)
    h_p = model_ref.encode(sd, model_ref.gather_feats(sd, pair_inputs["node_ids"], n), pair_inputs["attention_mask"], cfg)
    losses, logits, bs = [], [], 0
    for i, k in enumerate(num_pairs.tolist()):
        l, lg = model_ref.gsr_loss(h_p[bs: bs + k, 0], h_t[i, 0], labels[bs: bs + k])
        losses.append(l)
        logits.append(lg)
        bs += k
    loss = torch.stack(losses).mean()
    if training:
        if masked is None:
            masked = model_ref.mask_nodes(t_ids, node_size, cfg["random_node_ratio"], cfg["mask_node_ratio"])
        m_ids, m_mask, target_idx = masked
        h_m = model_ref.encode(sd, model_ref.gather_feats(sd, m_ids, n), t_mask, cfg)
        loss = loss + model_ref.nfr_loss(sd, h_m[:, 1:][m_mask], model_ref.gather_feats(sd, target_idx, n))
    return {"loss": loss, "prediction_logits": torch.cat(logits), "last_hidden_state": h_t}


def test_multi_modality_oracle_is_the_oracle_at_two():
    """The helper above is model_ref.pretrain_forward where that one applies (two modalities)."""
    cfg = model_ref.default_cfg(num_hidden_layers=1, hidden_size=32, intermediate_size=32, feat_hidden_sizes=[24, 16],
                                mask_node_ratio=0.5)
    node_size, B, P, L = 30, 3, 4, 6
    sd = model_ref.init_state_dict(cfg, node_size, seed=3, perturb=0.1)
    g = torch.Generator().manual_seed(9)
    tgt = {"node_ids": torch.randint(2, node_size + 2, (B, L), generator=g), "attention_mask": torch.ones(B, L)}
    pair = {"node_ids": torch.randint(2, node_size + 2, (B * P, L), generator=g), "attention_mask": torch.ones(B * P, L)}
    num_pairs = torch.tensor([P] * B)
    labels = (torch.rand(B * P, generator=g) < 0.5).float()
    torch.manual_seed(1)
    want = model_ref.pretrain_forward(sd, cfg, node_size, tgt, pair, num_pairs, labels, training=True)
    torch.manual_seed(1)
    got = pretrain_forward(sd, cfg, node_size, tgt, pair, num_pairs, labels, training=True)
    for k in ("loss", "prediction_logits", "last_hidden_state"):
        assert torch.equal(got[k], want[k]), k


def _net(widths, node_size=40):
    from pmgt_b200 import PMGT, PMGTConfig
    cfg = model_ref.default_cfg(feat_hidden_sizes=list(widths))
    sd = model_ref.init_state_dict(cfg, node_size, seed=4, perturb=0.05)
    net = PMGT(node_size, config=PMGTConfig(feat_hidden_sizes=list(widths)),
               feat_init_emb=[sd[f"feat_embeddings.{m}.weight"].numpy() for m in range(len(widths))])
    return net, sd


@pytest.mark.parametrize("widths", [[1536], [1536, 768, 512], [64, 32, 16, 8]])
def test_config_accepts_one_to_four_modalities(widths):
    from pmgt_b200 import PMGTConfig
    assert PMGTConfig(feat_hidden_sizes=widths).feat_hidden_sizes == widths


@pytest.mark.parametrize("widths", [[], [8, 8, 8, 8, 8]])
def test_config_rejects_other_counts(widths):
    from pmgt_b200 import PMGTConfig
    with pytest.raises(ValueError, match="1 to 4"):
        PMGTConfig(feat_hidden_sizes=widths)


def test_limit_matches_the_header():
    from pmgt_b200 import _lib, configuration_pmgt
    src = open(os.path.join(ROOT, "include", "pmgt_b200.h")).read()
    (n,) = re.findall(r"#define\s+PMGT_MAX_MODALITIES\s+(\d+)", src)
    assert int(n) == configuration_pmgt.MAX_MODALITIES == _lib.MAX_MODALITIES


def test_two_modality_flat_order_is_unchanged():
    from pmgt_b200 import PMGTConfig
    from pmgt_b200.modeling_pmgt import PMGTModel, encoder_param_order
    names = [n for n, _ in encoder_param_order(PMGTModel(PMGTConfig(num_hidden_layers=1)))]
    assert names[:10] == [
        "embeddings.feat_linear.0.weight", "embeddings.feat_linear.1.weight",
        "embeddings.feat_linear.0.bias", "embeddings.feat_linear.1.bias",
        "embeddings.attention.1.weight", "embeddings.attention.1.bias",
        "embeddings.position_embeddings.weight", "embeddings.role_embeddings.weight",
        "embeddings.LayerNorm.weight", "embeddings.LayerNorm.bias",
    ]


def test_three_modality_flat_order():
    from pmgt_b200 import PMGTConfig
    from pmgt_b200.modeling_pmgt import PMGTModel, encoder_param_order
    names = [n for n, _ in encoder_param_order(PMGTModel(PMGTConfig(num_hidden_layers=1, feat_hidden_sizes=[16, 8, 4])))]
    assert names[:6] == [f"embeddings.feat_linear.{m}.weight" for m in range(3)] + \
        [f"embeddings.feat_linear.{m}.bias" for m in range(3)]


@pytest.mark.parametrize("widths,n_tensors,n_params", [
    ([1536, 768], 104, 1_186_690),
    ([1536, 768, 512], 108, 1_319_043),
    ([1536], 100, 988_801),
])
def test_parameter_counts_and_state_dict_layout(widths, n_tensors, n_params):
    import warnings
    warnings.filterwarnings("ignore", message=".*use_return_dict.*")
    net, sd = _net(widths)
    trainable = [p for p in net.parameters() if p.requires_grad]
    assert len(trainable) == n_tensors
    assert sum(p.numel() for p in trainable) == n_params
    mine = {k: v for k, v in net.state_dict().items() if not k.endswith(("position_ids", "role_ids"))}
    assert set(mine) == set(sd)
    assert all(tuple(mine[k].shape) == tuple(sd[k].shape) for k in sd)
    # both ways: the oracle's dict loads into the model, and the model's dict reproduces it
    missing, unexpected = net.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.endswith(("position_ids", "role_ids")) for k in missing)
    back = net.state_dict()
    assert all(torch.equal(back[k], sd[k]) for k in sd)
    net2, _ = _net(widths)
    net2.load_state_dict(back)
    assert all(torch.equal(net2.state_dict()[k], back[k]) for k in back)


def test_embed_multi_struct_matches_the_header():
    from pmgt_b200 import _lib
    prog = r'''
#include <stdio.h>
#include <stddef.h>
#include "pmgt_b200.h"
int main(void){printf("%zu %zu %zu %zu %d\n", sizeof(pmgt_embed_multi_args), offsetof(pmgt_embed_multi_args, de),
  offsetof(pmgt_embed_multi_args, de_acc), offsetof(pmgt_embed_multi_args, skip_row0), PMGT_MAX_MODALITIES); return 0;}
'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(prog)
        exe = os.path.join(d, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        size, off_de, off_acc, off_skip, n = [int(x) for x in subprocess.check_output([exe]).split()]
    S = _lib.EmbedMultiArgs
    assert ctypes.sizeof(S) == size
    assert (S.de.offset, S.de_acc.offset, S.skip_row0.offset) == (off_de, off_acc, off_skip)
    assert n == _lib.MAX_MODALITIES


def test_embed_multi_argument_validation_without_a_gpu():
    """Out-of-range modality counts and missing or misaligned operands are refused before any CUDA call."""
    from pmgt_b200 import _lib, build
    build.build()
    lib = _lib.lib()
    a = _lib.EmbedMultiArgs()
    a.rows, a.L, a.H = 4, 6, 128
    for n in (0, 5):
        a.n_mod = n
        assert lib.pmgt_embed_multi_fwd(ctypes.byref(a), None) == -1
        assert b"n_mod" in lib.pmgt_last_error()
    a.n_mod = 3
    assert lib.pmgt_embed_multi_fwd(ctypes.byref(a), None) == -1
    assert b"null" in lib.pmgt_last_error()
    for f in ("w_att", "b_att", "pos", "role", "ln_g", "ln_b", "x_out"):
        setattr(a, f, 256)
    a.e[0], a.e[1] = 256, 512
    assert lib.pmgt_embed_multi_fwd(ctypes.byref(a), None) == -1
    assert b"e[2]" in lib.pmgt_last_error()
    a.e[2] = 520  # 8-byte aligned only
    assert lib.pmgt_embed_multi_fwd(ctypes.byref(a), None) == -1
    assert b"aligned" in lib.pmgt_last_error()
    a.e[2], a.H = 768, 36
    assert lib.pmgt_embed_multi_fwd(ctypes.byref(a), None) == -1
    assert b"multiple of 8" in lib.pmgt_last_error()
    a.H = 128
    assert lib.pmgt_embed_multi_bwd(ctypes.byref(a), None) == -1  # no gradient outputs
    assert b"null" in lib.pmgt_last_error()


@pytest.mark.needs_reference
@pytest.mark.parametrize("widths", [[48], [48, 40, 24]])
def test_oracle_matches_live_reference_at_other_modality_counts(widths):
    from oracle import ref_shim
    R = ref_shim.load()
    cfg = model_ref.default_cfg(num_hidden_layers=2, mask_node_ratio=0.5, feat_hidden_sizes=widths)
    node_size = 30
    sd = model_ref.init_state_dict(cfg, node_size, seed=3, perturb=0.1)
    rcfg = R.PMGTConfig(num_hidden_layers=2, feat_hidden_sizes=widths, hidden_dropout_prob=0.0,
                        attention_probs_dropout_prob=0.0)
    net = R.PMGT(node_size, cfg["random_node_ratio"], cfg["mask_node_ratio"], rcfg,
                 feat_init_emb=[sd[f"feat_embeddings.{m}.weight"].numpy() for m in range(len(widths))])
    net.load_state_dict(sd, strict=False)
    net.train()
    g = torch.Generator().manual_seed(9)
    B, P, L = 3, 4, 6
    tgt = {"node_ids": torch.randint(2, node_size + 2, (B, L), generator=g), "attention_mask": torch.ones(B, L)}
    pair = {"node_ids": torch.randint(2, node_size + 2, (B * P, L), generator=g), "attention_mask": torch.ones(B * P, L)}
    pair["attention_mask"][:, -2:] = 0
    pair["node_ids"][:, -2:] = 0
    num_pairs = torch.tensor([4, 4, 4])
    labels = (torch.rand(B * P, generator=g) < 0.5).float()
    torch.manual_seed(1)
    ref = net(tgt, pair, num_pairs, labels)
    torch.manual_seed(1)
    ours = pretrain_forward(sd, cfg, node_size, tgt, pair, num_pairs, labels, training=True)
    assert torch.allclose(ours["loss"], ref.loss, rtol=1e-5)
    assert torch.allclose(ours["prediction_logits"], ref.prediction_logits, rtol=1e-4, atol=1e-5)
