"""Context lengths the model accepts, checked on the host: a context of L tokens needs L rows of the position table
and an attention core that covers L (at most 128 tokens).  Both checks run before any device work."""
import pytest
import torch


def _encode(cfg, L, R=2):
    from pmgt_b200.modeling_pmgt import PMGTModel
    net = PMGTModel(cfg)
    src = [torch.zeros(R * L, d, dtype=torch.bfloat16) for d in cfg.feat_hidden_sizes]
    return net.encode(src, None, torch.ones(R, L), R, L)


def test_encode_refuses_a_context_longer_than_the_position_table():
    from pmgt_b200 import PMGTConfig
    cfg = PMGTConfig(num_hidden_layers=1, feat_hidden_sizes=[16, 8])
    with pytest.raises(ValueError, match=r"101 tokens.*max_position_embeddings is 100"):
        _encode(cfg, 101)


def test_encode_refuses_a_context_longer_than_the_attention_core_limit():
    from pmgt_b200 import PMGTConfig
    from pmgt_b200.modeling_pmgt import MAX_CONTEXT_LEN
    assert MAX_CONTEXT_LEN == 128
    cfg = PMGTConfig(num_hidden_layers=1, feat_hidden_sizes=[16, 8], max_position_embeddings=200)
    with pytest.raises(ValueError, match=r"129 tokens.*attention core's limit of 128"):
        _encode(cfg, 129)


def test_check_args_bounds_max_ctx_neigh_by_the_default_position_table():
    from pmgt_b200 import trainer
    trainer.check_args(trainer.make_args(max_ctx_neigh=99))
    with pytest.raises(ValueError, match=r"max_ctx_neigh must be <= 99"):
        trainer.check_args(trainer.make_args(max_ctx_neigh=100))
