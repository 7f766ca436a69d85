"""CPU-only: per-layer hidden states and attention maps (output_hidden_states / output_attentions) -- the flag rules,
the tuple layout, head_mask still refused, the C-ABI argument checks of pmgt_attn_maps_fwd, and the fp32 reference
(``encode_with_outputs``) the GPU tests compare against, pinned here to the oracle's own encoder."""
import ctypes

import pytest
import torch

from oracle import model_ref


# ---------------------------------------------------------------------------------------------------------------------
# reference: oracle/model_ref's encoder with transformers' output_hidden_states / output_attentions
# ---------------------------------------------------------------------------------------------------------------------
def attention_probs(sd, prefix, x, ext_mask, heads, beta):
    """The matrix PMGTSelfAttention.forward multiplies the values with (modeling_pmgt.py:519-526), dropout = identity:
    beta * P1 + (1 - beta) * P2 as ``[R, heads, L, L]`` -- model_ref.self_attention up to that point."""
    R, L, H = x.shape
    dh = H // heads

    def split(t):
        return t.view(R, L, heads, dh).permute(0, 2, 1, 3)

    q = split(model_ref._linear(x, sd, prefix + "query"))
    k = split(model_ref._linear(x, sd, prefix + "key"))
    c = split(model_ref._linear(x, sd, prefix + "ctx_attention"))
    n = torch.linalg.norm(c, dim=-1, keepdim=True)
    s1 = 1.0 - (c @ c.transpose(-1, -2)) / (n @ n.transpose(-1, -2)) + torch.eye(L, device=x.device, dtype=x.dtype)
    p1 = torch.softmax(s1 + ext_mask, dim=-1)
    p2 = torch.softmax((q @ k.transpose(-1, -2)) / dh ** 0.5 + ext_mask, dim=-1)
    return beta * p1 + (1.0 - beta) * p2


def encode_with_outputs(sd, feats, attention_mask, cfg):
    """model_ref.encode with per-layer outputs: (hidden_states, attentions) -- ``num_hidden_layers + 1`` tensors
    ``[R, L, H]`` (embedding output, then every layer's output; the last is model_ref.encode's result) and
    ``num_hidden_layers`` tensors ``[R, heads, L, L]``.  Differentiable."""
    ext = (1.0 - attention_mask[:, None, None, :].to(feats[0].dtype)) * -10000.0
    x = model_ref.embeddings(sd, feats, cfg["layer_norm_eps"])
    hidden_states, attentions = [x], []
    for i in range(cfg["num_hidden_layers"]):
        attentions.append(attention_probs(sd, f"bert.encoder.layer.{i}.attention.self.", x, ext,
                                          cfg["num_attention_heads"], cfg["beta"]))
        x = model_ref.layer(sd, i, x, ext, cfg["num_attention_heads"], cfg["beta"], cfg["layer_norm_eps"])
        hidden_states.append(x)
    return tuple(hidden_states), tuple(attentions)


def test_reference_outputs_are_the_oracle_encoder():
    """The last hidden state is model_ref.encode's, and A V of every layer is model_ref.self_attention's context."""
    cfg = model_ref.default_cfg(num_hidden_layers=3, hidden_size=32, intermediate_size=48, num_attention_heads=2,
                                feat_hidden_sizes=[24, 16])
    sd = model_ref.init_state_dict(cfg, 20, seed=4, perturb=0.1)
    g = torch.Generator().manual_seed(1)
    R, L = 3, 7
    ids = torch.randint(2, 22, (R, L), generator=g)
    mask = torch.ones(R, L)
    mask[1, 4:] = 0
    feats = model_ref.gather_feats(sd, ids)
    hs, att = encode_with_outputs(sd, feats, mask, cfg)
    assert len(hs) == 4 and len(att) == 3
    assert all(h.shape == (R, L, 32) for h in hs) and all(a.shape == (R, 2, L, L) for a in att)
    torch.testing.assert_close(hs[-1], model_ref.encode(sd, feats, mask, cfg), rtol=0, atol=0)
    torch.testing.assert_close(att[0].sum(-1), torch.ones(R, 2, L), rtol=1e-5, atol=1e-5)
    ext = (1.0 - mask[:, None, None, :]) * -10000.0
    for i, a in enumerate(att):
        p = f"bert.encoder.layer.{i}.attention.self."
        v = model_ref._linear(hs[i], sd, p + "value").view(R, L, 2, 16).permute(0, 2, 1, 3)
        ctx = (a @ v).permute(0, 2, 1, 3).reshape(R, L, 32)
        torch.testing.assert_close(ctx, model_ref.self_attention(sd, p, hs[i], ext, 2, cfg["beta"]))
    assert float(att[1][1, :, :, 4:].abs().max()) < 1e-30  # padded keys get no weight


# ---------------------------------------------------------------------------------------------------------------------
# host logic
# ---------------------------------------------------------------------------------------------------------------------
def test_output_flags_follow_arguments_then_config():
    from pmgt_b200 import PMGTConfig
    from pmgt_b200.modeling_pmgt import resolve_output_flags
    assert resolve_output_flags(PMGTConfig(), None, None) == (False, False)
    c = PMGTConfig(output_attentions=True, output_hidden_states=True)
    assert resolve_output_flags(c, None, None) == (True, True)
    assert resolve_output_flags(c, False, None) == (False, True)
    assert resolve_output_flags(c, None, False) == (True, False)
    assert resolve_output_flags(PMGTConfig(), True, False) == (True, False)
    assert resolve_output_flags(PMGTConfig(), None, True) == (False, True)


def test_tuple_tail_holds_only_what_was_requested():
    from pmgt_b200.modeling_pmgt import output_tuple
    hs, att = (torch.zeros(1),), (torch.ones(1),)
    assert output_tuple(None, None) == ()
    assert output_tuple(hs, None) == (hs,)
    assert output_tuple(None, att) == (att,)
    assert output_tuple(hs, att) == (hs, att)


def test_head_mask_still_raises_and_flags_are_accepted():
    """head_mask is refused before anything else; the output flags are not (a CPU call then fails for lack of CUDA)."""
    from pmgt_b200 import PMGTConfig, PMGTModel, _lib
    cfg = PMGTConfig(hidden_size=32, intermediate_size=32, num_hidden_layers=1, num_attention_heads=2,
                     feat_hidden_sizes=[8, 8])
    m = PMGTModel(cfg)
    x = [torch.zeros(2, 6, 8), torch.zeros(2, 6, 8)]
    with pytest.raises(NotImplementedError, match="head_mask"):
        m(*x, head_mask=torch.ones(1, 2))
    with pytest.raises(_lib.PMGTError, match="CUDA"):
        m(*x, output_attentions=True, output_hidden_states=True)


def test_pmgt_accepts_output_flags():
    from pmgt_b200 import PMGT, PMGTConfig, _lib
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        net = PMGT(50, config=PMGTConfig(num_hidden_layers=1, output_attentions=True, output_hidden_states=True))
    x = {"node_ids": torch.randint(2, 52, (2, 6)), "attention_mask": torch.ones(2, 6)}
    with pytest.raises(_lib.PMGTError):
        net(x)


# ---------------------------------------------------------------------------------------------------------------------
# C ABI
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from pmgt_b200 import _lib, build
    build.build()
    return _lib.lib()


def test_maps_entry_is_exported(lib):
    from pmgt_b200 import _lib
    assert hasattr(lib, "pmgt_attn_maps_fwd") and "pmgt_attn_maps_fwd" in _lib.SIGNATURES
    assert lib.pmgt_abi_version() == _lib.ABI_VERSION == 14


def test_maps_argument_validation_without_a_gpu(lib):
    """A null maps pointer, a misaligned qkvc or maps, or a shape the core refuses return PMGT_ERR_INVALID with a
    message, before any CUDA call.  The pointers are fake, so this only runs where no device could be reached."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from pmgt_b200 import _lib
    a = _lib.AttnArgs()
    a.rows, a.L, a.H, a.heads, a.beta = 4, 33, 64, 1, 0.5
    a.qkvc, a.mask = 16, 16
    a.dropout_p = 0.1
    assert lib.pmgt_attn_maps_fwd(ctypes.byref(a), None, None) == -1
    assert b"pmgt_attn_maps_fwd: null argument" in lib.pmgt_last_error()
    a.qkvc = 24
    assert lib.pmgt_attn_maps_fwd(ctypes.byref(a), 16, None) == -1
    assert b"pmgt_attn_maps_fwd: qkvc must be 16-byte aligned" in lib.pmgt_last_error()
    a.qkvc = 16
    assert lib.pmgt_attn_maps_fwd(ctypes.byref(a), 8, None) == -1
    assert b"pmgt_attn_maps_fwd: maps must be 16-byte aligned" in lib.pmgt_last_error()
    a.L = 129
    assert lib.pmgt_attn_maps_fwd(ctypes.byref(a), 16, None) == -1
    assert b"L must be in [1,128]" in lib.pmgt_last_error()
    a.L, a.H = 33, 66
    a.heads = 2  # head size 33: odd
    assert lib.pmgt_attn_maps_fwd(ctypes.byref(a), 16, None) == -1
    assert b"head size must be even" in lib.pmgt_last_error()
    a.mask = None
    assert lib.pmgt_attn_maps_fwd(ctypes.byref(a), 16, None) == -1
    assert b"pmgt_attn_maps_fwd: null argument" in lib.pmgt_last_error()
