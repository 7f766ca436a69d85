"""Host-side mirror of ``pmgt/pmgt/modeling_pmgt.py``.

Same class names, constructor arguments, forward signatures and state-dict keys
as the reference; the computation underneath is ``libpmgt_b200.so`` (sm_100a
CUDA through the C ABI).  ``nn.Linear`` / ``nn.Embedding`` / ``nn.LayerNorm``
objects are used purely as *parameter containers* so that
``state_dict()`` / ``load_state_dict()`` interchange with reference checkpoints
both ways; their ``forward`` is never called.

Numerics: parameters are fp32 (master copy); every GEMM runs on tcgen05 tensor
cores with bf16 operands and fp32 accumulation; activations are stored in
bf16; softmax / LayerNorm / losses are computed in fp32.

There is no CPU path: calling ``forward`` with CPU tensors raises.
"""
from dataclasses import dataclass, fields
from typing import List, Optional, Tuple

import torch
import torch.nn as nn

from . import ops
from ._lib import PMGTError
from .configuration_pmgt import PMGTConfig

BF16 = torch.bfloat16
_ALIGN = 8  # elements: 16-byte alignment of every bf16 tensor (TMA / vector loads); tensors whose numel is a
# multiple of 8 are packed back to back, which the [4H, H] "span" views over q/k/v/ctx rely on


# ---------------------------------------------------------------------------
# outputs (modeling_pmgt.py:572-579, transformers ModelOutput semantics)
# ---------------------------------------------------------------------------
class _ModelOutput:
    """Minimal ``transformers.file_utils.ModelOutput``: attribute + key access,
    and integer indexing over the non-``None`` fields (which is why the
    reference's ``net(x)[0]`` is the loss in training and ``last_hidden_state``
    at inference, trainer.py:153-157)."""

    def to_tuple(self):
        return tuple(getattr(self, f.name) for f in fields(self) if getattr(self, f.name) is not None)

    def __getitem__(self, k):
        if isinstance(k, str):
            v = getattr(self, k)
            if v is None:
                raise KeyError(k)
            return v
        return self.to_tuple()[k]

    def __iter__(self):
        return iter(self.to_tuple())

    def __len__(self):
        return len(self.to_tuple())

    def keys(self):
        return [f.name for f in fields(self) if getattr(self, f.name) is not None]


@dataclass
class BaseModelOutputWithPooling(_ModelOutput):
    last_hidden_state: torch.Tensor = None
    pooler_output: Optional[torch.Tensor] = None
    hidden_states: Optional[Tuple[torch.Tensor]] = None
    attentions: Optional[Tuple[torch.Tensor]] = None


@dataclass
class PMGTForPreTrainingOutput(_ModelOutput):
    loss: Optional[torch.Tensor] = None
    prediction_logits: Optional[torch.Tensor] = None
    last_hidden_state: torch.Tensor = None
    pooler_output: Optional[torch.Tensor] = None
    hidden_states: Optional[Tuple[torch.Tensor]] = None
    attentions: Optional[Tuple[torch.Tensor]] = None


# ---------------------------------------------------------------------------
# parameter containers (names == reference state-dict keys)
# ---------------------------------------------------------------------------
class PMGTEmbeddings(nn.Module):
    """modeling_pmgt.py:155-187."""

    def __init__(self, config):
        super().__init__()
        H = config.hidden_size
        self.position_embeddings = nn.Embedding(config.max_position_embeddings, H)
        self.role_embeddings = nn.Embedding(2, H)
        self.feat_linear = nn.ModuleList(nn.Linear(d, H) for d in config.feat_hidden_sizes)
        n = len(config.feat_hidden_sizes)
        self.attention = nn.Sequential(nn.Tanh(), nn.Linear(n * H, n), nn.Softmax(dim=-1))
        self.LayerNorm = nn.LayerNorm(H, eps=config.layer_norm_eps)
        self.dropout = nn.Dropout(config.hidden_dropout_prob)
        self.register_buffer("position_ids", torch.arange(config.max_position_embeddings).unsqueeze(0))
        self.register_buffer("role_ids", torch.LongTensor([0] + [1] * (config.max_position_embeddings - 1)).unsqueeze(0))


class PMGTSelfAttention(nn.Module):
    """modeling_pmgt.py:378-399."""

    def __init__(self, config):
        super().__init__()
        if config.hidden_size % config.num_attention_heads != 0:
            raise ValueError(
                f"The hidden size ({config.hidden_size}) is not a multiple of the number of attention "
                f"heads ({config.num_attention_heads})")
        H = config.hidden_size
        self.num_attention_heads = config.num_attention_heads
        self.attention_head_size = H // config.num_attention_heads
        self.all_head_size = H
        self.beta = config.beta
        self.query = nn.Linear(H, H)
        self.key = nn.Linear(H, H)
        self.value = nn.Linear(H, H)
        self.ctx_attention = nn.Linear(H, H)
        self.dropout = nn.Dropout(config.attention_probs_dropout_prob)


class _DenseLN(nn.Module):
    """BertSelfOutput / BertOutput parameter layout: ``dense`` + ``LayerNorm``."""

    def __init__(self, in_f, out_f, eps, p):
        super().__init__()
        self.dense = nn.Linear(in_f, out_f)
        self.LayerNorm = nn.LayerNorm(out_f, eps=eps)
        self.dropout = nn.Dropout(p)


class _Dense(nn.Module):
    """BertIntermediate parameter layout: ``dense``."""

    def __init__(self, in_f, out_f):
        super().__init__()
        self.dense = nn.Linear(in_f, out_f)


class PMGTAttention(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.self = PMGTSelfAttention(config)
        self.output = _DenseLN(config.hidden_size, config.hidden_size, config.layer_norm_eps, config.hidden_dropout_prob)


class PMGTLayer(nn.Module):
    """modeling_pmgt.py:287-295."""

    def __init__(self, config):
        super().__init__()
        self.attention = PMGTAttention(config)
        self.intermediate = _Dense(config.hidden_size, config.intermediate_size)
        self.output = _DenseLN(config.intermediate_size, config.hidden_size, config.layer_norm_eps,
                               config.hidden_dropout_prob)


class PMGTEncoder(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.config = config
        self.layer = nn.ModuleList([PMGTLayer(config) for _ in range(config.num_hidden_layers)])
        self.gradient_checkpointing = False


# ---------------------------------------------------------------------------
# flat parameter storage
# ---------------------------------------------------------------------------
class FlatParams:
    """All trainable parameters of a root module as views into ONE fp32 buffer
    (so the bf16 shadow cast, the gradient allreduce and AdamW are single
    launches), in an order that makes [Wq;Wk;Wv;Wc] one [4H, H] matrix."""

    def __init__(self, named_params: List[Tuple[str, nn.Parameter]]):
        self.names = [n for n, _ in named_params]
        self.params = [p for _, p in named_params]
        self.offsets = {}
        self.shapes = {}
        off = 0
        for n, p in named_params:
            self.offsets[n] = off
            self.shapes[n] = tuple(p.shape)
            off += (p.numel() + _ALIGN - 1) // _ALIGN * _ALIGN
        self.total = off
        self.flat = None
        self.flat_bf16 = None
        # called as hook(arena) from the encoder backward once every gradient EXCEPT those of the embedding block is
        # final (data-parallel training starts the allreduce of that part here, overlapping the embedding backward)
        self.after_layers_hook = None
        self._views32 = {}
        self._views16 = {}

    def ensure(self):
        """(Re)attach parameters to the flat buffer if ``.to()`` / ``.cuda()`` moved them."""
        p0 = self.params[0]
        # fast path (every step): the first and the last parameter still sit where the flat buffer put them.  A move of
        # the module (.to / .cuda) relocates all of them; anything subtler is caught by the full check below, which
        # runs whenever either pointer changed.
        if self.flat is not None:
            base = self.flat.data_ptr()
            pl = self.params[-1]
            if (p0.data_ptr() == base + 4 * self.offsets[self.names[0]]
                    and pl.data_ptr() == base + 4 * self.offsets[self.names[-1]]):
                return self
        dev = p0.device
        if dev.type != "cuda":
            raise PMGTError("pmgt_b200 modules must live on a CUDA device (no CPU fallback); call .cuda() first")
        ok = self.flat is not None and self.flat.device == dev
        if ok:
            base = self.flat.data_ptr()
            for n, p in zip(self.names, self.params):
                if p.data_ptr() != base + 4 * self.offsets[n] or p.dtype != torch.float32:
                    ok = False
                    break
        if not ok:
            flat = torch.zeros(self.total, dtype=torch.float32, device=dev)
            with torch.no_grad():
                for n, p in zip(self.names, self.params):
                    v = flat[self.offsets[n]: self.offsets[n] + p.numel()].view(p.shape)
                    v.copy_(p.data.to(torch.float32))
                    p.data = v
            self.flat = flat
            self.flat_bf16 = torch.empty(self.total, dtype=BF16, device=dev)
            self._views32, self._views16 = {}, {}
        return self

    def refresh_bf16(self):
        ops.cast_f32_bf16(self.flat, self.flat_bf16)

    def _view(self, buf, cache, name, span=None):
        key = (name, span)
        v = cache.get(key)
        if v is None:
            off = self.offsets[name]
            shape = self.shapes[name]
            if span is not None:  # `span` consecutive same-shaped tensors as one matrix / vector
                shape = (shape[0] * span,) + shape[1:]
            n = 1
            for s in shape:
                n *= s
            v = buf[off: off + n].view(shape)
            cache[key] = v
        return v

    def f32(self, name, span=None):
        return self._view(self.flat, self._views32, name, span)

    def step_arena(self) -> "GradArena":
        """The persistent gradient arena of this parameter set (one per flat buffer), zeroed for a new step."""
        a = getattr(self, "_step_arena", None)
        if a is None or a.buf is None or a.buf.device != self.flat.device or a.buf.numel() != self.total:
            a = GradArena(self, persistent=True, symm_group=getattr(self, "symm_group", None))
            a.get()
            self._step_arena = a
            return a
        return a.reset()

    def bf16(self, name, span=None):
        return self._view(self.flat_bf16, self._views16, name, span)


class GradArena:
    """One fp32 buffer per backward pass holding every parameter gradient in
    FlatParams order; autograd receives views of it."""

    def __init__(self, fp: FlatParams, persistent: bool = False, symm_group=None):
        self.fp = fp
        self.buf = None
        self.persistent = persistent  # the same buffer every step (zeroed by `reset`): what a launch plan needs
        # data parallel: allocate the buffer in symmetric memory of this process group, so that the ranks can sum their
        # gradients through peer pointers (trainer.train_on_indices, csrc/peer_reduce.cu); `symm` = the handle
        self.symm_group = symm_group
        self.symm = None

    def reset(self):
        if self.buf is not None:
            self.buf.zero_()
        return self

    def get(self):
        if self.buf is None:
            dev = self.fp.flat.device
            if self.symm_group is not None:
                import torch.distributed._symmetric_memory as symm_mem
                self.buf = symm_mem.empty(self.fp.total, dtype=torch.float32, device=dev)
                self.buf.zero_()
                self.symm = symm_mem.rendezvous(self.buf, self.symm_group)   # collective: every rank allocates here
            else:
                self.buf = torch.zeros(self.fp.total, dtype=torch.float32, device=dev)
        return self.buf

    def view(self, name, span=None):
        fp = self.fp
        off = fp.offsets[name]
        shape = fp.shapes[name]
        if span is not None:
            shape = (shape[0] * span,) + shape[1:]
        # one as_strided instead of slice + view: this runs ~100 times per backward pass (host-bound small batches)
        strides = fp.__dict__.setdefault("_strides", {}).get(shape)
        if strides is None:
            st, acc = [], 1
            for d in reversed(shape):
                st.append(acc)
                acc *= d
            strides = fp._strides[shape] = tuple(reversed(st))
        return torch.as_strided(self.get(), shape, strides, off)


MAX_CONTEXT_LEN = 128  # the attention core's longest sequence (pmgt_attn_core_fwd / _bwd)


def check_context_len(config, L: int) -> None:
    """A context of ``L`` tokens needs ``L`` rows of the position table and an attention core that covers ``L``."""
    if L > config.max_position_embeddings:
        raise ValueError(f"context of {L} tokens exceeds the position table: max_position_embeddings is "
                         f"{config.max_position_embeddings}")
    if L > MAX_CONTEXT_LEN:
        raise ValueError(f"context of {L} tokens exceeds the attention core's limit of {MAX_CONTEXT_LEN} tokens")


def encoder_param_order(bert: "PMGTModel", prefix: str = "") -> List[Tuple[str, nn.Parameter]]:
    """Flat order of the encoder's trainable parameters (names carry ``prefix``)."""
    e = bert.embeddings
    # every feature projection's weight, then every bias (the flat buffer layout of the two-modality model)
    out = [(f"embeddings.feat_linear.{m}.weight", l.weight) for m, l in enumerate(e.feat_linear)]
    out += [(f"embeddings.feat_linear.{m}.bias", l.bias) for m, l in enumerate(e.feat_linear)]
    out += [
        ("embeddings.attention.1.weight", e.attention[1].weight),
        ("embeddings.attention.1.bias", e.attention[1].bias),
        ("embeddings.position_embeddings.weight", e.position_embeddings.weight),
        ("embeddings.role_embeddings.weight", e.role_embeddings.weight),
        ("embeddings.LayerNorm.weight", e.LayerNorm.weight),
        ("embeddings.LayerNorm.bias", e.LayerNorm.bias),
    ]
    for i, l in enumerate(bert.encoder.layer):
        p = f"encoder.layer.{i}."
        s = l.attention.self
        out += [(p + f"attention.self.{n}.weight", getattr(s, n).weight) for n in ("query", "key", "value", "ctx_attention")]
        out += [(p + f"attention.self.{n}.bias", getattr(s, n).bias) for n in ("query", "key", "value", "ctx_attention")]
        out += [
            (p + "attention.output.dense.weight", l.attention.output.dense.weight),
            (p + "attention.output.dense.bias", l.attention.output.dense.bias),
            (p + "attention.output.LayerNorm.weight", l.attention.output.LayerNorm.weight),
            (p + "attention.output.LayerNorm.bias", l.attention.output.LayerNorm.bias),
            (p + "intermediate.dense.weight", l.intermediate.dense.weight),
            (p + "intermediate.dense.bias", l.intermediate.dense.bias),
            (p + "output.dense.weight", l.output.dense.weight),
            (p + "output.dense.bias", l.output.dense.bias),
            (p + "output.LayerNorm.weight", l.output.LayerNorm.weight),
            (p + "output.LayerNorm.bias", l.output.LayerNorm.bias),
        ]
    return [(prefix + n, p) for n, p in out]


# ---------------------------------------------------------------------------
# encoder forward / backward orchestration
# ---------------------------------------------------------------------------
class _BufPool:
    """Shape-keyed free list for the backward pass of a launch plan: a buffer released after its last reader was
    enqueued is handed to a later allocation of the same shape (everything runs on one stream, so stream order makes
    the reuse safe).  Without it a recorded backward pass would pin every temporary of every layer."""

    def __init__(self, device):
        self.device = device
        self.free = {}
        self.owned = []

    def get(self, shape, dtype):
        key = (tuple(shape), dtype)
        lst = self.free.get(key)
        if lst:
            return lst.pop()
        t = torch.empty(shape, dtype=dtype, device=self.device)
        self.owned.append(t)
        return t

    def release(self, *ts):
        seen = set()
        for t in ts:
            if t is None or id(t) in seen:
                continue
            seen.add(id(t))
            self.free.setdefault((tuple(t.shape), t.dtype), []).append(t)


class _EncoderPlan:
    """The launch sequence of one encoder pass at fixed shapes, recorded on the first step and re-issued afterwards.

    Everything the recorded argument blocks point at is owned by the plan (inputs are copied into ``rows_idx`` /
    ``mask``; activations, temporaries, ``hidden`` and ``d_hidden`` stay allocated), so a replay is ~170 ctypes calls
    with ready-made arguments; only the dropout seed is patched.  Outputs are valid until the next pass through the
    same plan -- which is why plans are opt-in (``PMGTModel.use_launch_plans``; the trainer's step loop turns them on).
    """

    def __init__(self, key, R, L, H, device, n_last=0):
        self.key, self.R, self.L, self.T, self.H = key, R, L, R * L, H
        self.device = device
        self.rows_idx = torch.empty(R * L, dtype=torch.int64, device=device)
        self.mask = torch.empty(R, L, dtype=torch.float32, device=device)
        self.last_rows = torch.empty(n_last, dtype=torch.int64, device=device) if n_last else None
        self.fwd_tape, self.bwd_tape = None, None
        self.fwd_seeds, self.bwd_seeds = [], []
        self.hidden, self.run, self.d_hidden = None, None, None
        self.pool = _BufPool(device)
        self.pending_backward = False

    def grad_buffer(self) -> torch.Tensor:
        """fp32 [T, H] buffer the caller may build d(loss)/d(hidden) in (saves the copy in ``backward``)."""
        if self.d_hidden is None:
            n = self.last_rows.numel() if self.last_rows is not None else self.T
            self.d_hidden = torch.empty(n, self.H, dtype=torch.float32, device=self.device)
        return self.d_hidden

    def forward(self, fp, pre, cfg, src, rows_idx, mask, training, seed, keep, last_rows=None):
        self.rows_idx.copy_(rows_idx.reshape(-1))
        self.mask.copy_(mask)
        if self.last_rows is not None:
            self.last_rows.copy_(last_rows)
        if self.fwd_tape is None:
            tape = []
            ops.TAPE = tape
            try:
                self.held = []
                self.hidden, self.run = _encode_forward(fp, pre, cfg, src, self.rows_idx, self.R, self.L, self.mask,
                                                        training, seed, keep, hold=self.held, last_rows=self.last_rows)
            finally:
                ops.TAPE = None
            self.fwd_tape, self.fwd_seeds = tape, ops.tape_seed_blocks(tape)
        else:
            for a in self.fwd_seeds:
                a.dropout_seed = seed
            if self.run is not None:
                self.run.seed = seed
            ops.replay(self.fwd_tape)
        self.pending_backward = keep
        return self.hidden.view(self.hidden.shape)  # a fresh tensor object over the plan-owned buffer

    def backward(self, fp, pre, cfg, d_hidden, arena):
        buf = self.grad_buffer()
        if d_hidden.data_ptr() != buf.data_ptr():
            buf.copy_(d_hidden.reshape(-1, self.H))
        if self.bwd_tape is None:
            tape = []
            ops.TAPE = tape
            try:
                _encode_backward(fp, pre, cfg, self.run, buf, arena, pool=self.pool)
            finally:
                ops.TAPE = None
            self.bwd_tape, self.bwd_seeds = tape, ops.tape_seed_blocks(tape)
        else:
            for a in self.bwd_seeds:
                a.dropout_seed = self.run.seed
            ops.replay(self.bwd_tape)
        self.pending_backward = False


class _EncoderOutputs:
    """What an encoder pass collects besides its final hidden state (``output_hidden_states`` /
    ``output_attentions``): ``layers`` = the bf16 ``[T, H]`` inputs of layers 0 .. n-1 (the embedding output, then the
    outputs of layers 1 .. n-1), ``maps`` = per layer the fp32 ``[map_rows, heads, L, L]`` matrices its attention core
    multiplied V with, for the first ``map_rows`` sequences."""
    __slots__ = ("hidden", "attentions", "map_rows", "layers", "maps")

    def __init__(self, hidden: bool, attentions: bool, map_rows: int):
        self.hidden, self.attentions, self.map_rows = hidden, attentions, map_rows
        self.layers, self.maps = [], []


class _EncoderRun:
    """Activations of one encoder pass kept for the backward pass."""
    __slots__ = ("R", "L", "T", "mask", "rows_idx", "src", "src_rows", "proj", "x0", "layers", "seed", "p_hid",
                 "p_att", "hidden_f32", "tile", "dense_tables", "last_rows")


# dX kernels of the 128 x 128 Linears also produce dW / dbias (one pass over dY); False: separate pmgt_dw_tile launches
FUSED_DW = True
# dW of the fused Q/K/V/C projection: one batched launch for all layers at the end of the backward pass (False: per layer)
BATCH_DW_QKVC = True

# "auto": projected tables when 4 * table rows <= tokens, else the gather-fused GEMM; "table" / "gather" force a mode
PROJECTION_MODE = "auto"


def _tile_path(H: int, I: int) -> bool:
    """The persistent token-tile kernels cover the default encoder (H = I = 128); other sizes use pmgt_gemm_bf16."""
    return (ops.linear_tile_supported(H, 4 * H, False, ops.LT_BIAS) and ops.linear_tile_supported(H, H, False, ops.LT_RES_LN)
            and ops.linear_tile_supported(H, I, False, ops.LT_GELU) and ops.linear_tile_supported(I, H, False, ops.LT_RES_LN)
            and ops.linear_tile_supported(4 * H, H, True, ops.LT_PLAIN) and ops.linear_tile_supported(I, H, True, ops.LT_PLAIN)
            and ops.linear_tile_supported(H, I, True, ops.LT_GELU_BWD) and ops.dw_tile_supported(4 * H, H)
            and ops.dw_tile_supported(H, I) and ops.dw_tile_supported(I, H) and H == 128)


def _encode_forward(fp: FlatParams, pre: str, cfg: PMGTConfig, src: List[torch.Tensor], rows_idx, R: int, L: int,
                    mask: torch.Tensor, training: bool, seed: int, keep: bool, hold: Optional[list] = None,
                    last_rows: Optional[torch.Tensor] = None, outs: Optional[_EncoderOutputs] = None):
    """PMGTModel.forward (modeling_pmgt.py:80-152) on ``R`` sequences of length ``L``.

    ``src``: per modality either the bf16 feature table (``rows_idx`` = flat int64
    node ids, fused gather) or a dense bf16 ``[T, D]`` matrix (``rows_idx`` None).
    Returns (hidden_f32 [R, L, H], run-or-None).

    ``last_rows`` (token-tile path only): sorted unique token indices whose final hidden state the caller consumes.
    Rows are independent after the attention core, so the LAST layer runs its post-attention half (output projection +
    LayerNorm, FFN, LayerNorm -- and their whole backward) only on those rows; the result is then the compact
    ``[len(last_rows), H]`` matrix.  In pre-training that is ~30 % of the tokens (all positions of the target and the
    masked-target rows, position 0 of the pair rows).

    ``outs`` (opt-in): collect the per-layer hidden states and attention maps there (see ``_EncoderOutputs``).  The maps
    come from pmgt_attn_maps_fwd with each layer's own attention arguments (same seed and site), right after its
    attention core, so they carry the dropout mask that core applied.
    """
    H, I, heads = cfg.hidden_size, cfg.intermediate_size, cfg.num_attention_heads
    T = R * L
    dev = mask.device
    p_hid = float(cfg.hidden_dropout_prob) if training else 0.0
    p_att = float(cfg.attention_probs_dropout_prob) if training else 0.0
    E = pre + "embeddings."

    def new(*shape, dtype=BF16):
        t = torch.empty(shape, dtype=dtype, device=dev)
        if hold is not None:  # a launch plan keeps every buffer its recorded launches point at
            hold.append(t)
        return t

    # K2: per-modality projections on tensor cores, then the fusion kernel.  Two modes:
    #  * gather-fused GEMM: rows of the feature tables are fetched inside the GEMM, one projection per TOKEN
    #    (large graphs: most table rows are never touched in a step);
    #  * projected tables: when the tables are small next to the token count (VG / TG: ~10^4 rows vs 3*10^5
    #    tokens) every table row is projected ONCE and tokens gather the projected H-vectors instead.
    dense_tables = rows_idx is not None and (PROJECTION_MODE == "table" or
                                             (PROJECTION_MODE == "auto" and 4 * src[0].shape[0] <= T))
    proj = []
    for m in range(len(src)):
        if dense_tables:
            out = new(src[m].shape[0], H)
            ops.linear_fwd(src[m], fp.bf16(f"{E}feat_linear.{m}.weight"), fp.f32(f"{E}feat_linear.{m}.bias"), out,
                           tag="gemm_fwd_table")
        else:
            out = new(T, H)
            ops.linear_fwd(src[m], fp.bf16(f"{E}feat_linear.{m}.weight"), fp.f32(f"{E}feat_linear.{m}.bias"), out,
                           rows=rows_idx, src_rows=(src[m].shape[0] if rows_idx is not None else 0))
        proj.append(out)
    x = new(T, H)
    ea = ops.embed_multi_args(R, L, H, proj, fp.f32(E + "attention.1.weight"), fp.f32(E + "attention.1.bias"),
                              fp.f32(E + "position_embeddings.weight"), fp.f32(E + "role_embeddings.weight"),
                              fp.f32(E + "LayerNorm.weight"), fp.f32(E + "LayerNorm.bias"), cfg.layer_norm_eps, p_hid, seed,
                              0, x_out=x, row_idx=(rows_idx if dense_tables else None))
    ops.embed_multi_fwd(ea)
    if outs is not None and outs.hidden and cfg.num_hidden_layers > 0:  # with no layers, x is the final state
        outs.layers.append(x)

    def collect_maps(i, qkvc):  # right after layer i's attention core, with its arguments
        if outs is not None and outs.attentions:
            maps = torch.empty(outs.map_rows, heads, L, L, dtype=torch.float32, device=dev)
            ops.attn_maps_fwd(ops.attn_args(outs.map_rows, L, H, heads, float(cfg.beta), qkvc, mask, p_att, seed,
                                            10 * (i + 1)), maps)
            outs.maps.append(maps)

    run = None
    if keep:
        run = _EncoderRun()
        run.R, run.L, run.T, run.mask, run.rows_idx = R, L, T, mask, rows_idx
        run.src, run.src_rows = src, [s.shape[0] for s in src]
        run.proj, run.x0, run.layers = proj, x, []
        run.seed, run.p_hid, run.p_att = seed, p_hid, p_att
        run.dense_tables = dense_tables

    n_layers = cfg.num_hidden_layers
    tile = _tile_path(H, I)
    compact = last_rows is not None and tile and n_layers > 0
    Tc = int(last_rows.numel()) if compact else T
    hidden_f32 = new(Tc, H, dtype=torch.float32)
    if keep:
        run.tile = tile
        run.last_rows = last_rows if compact else None
    for i in range(n_layers if tile else 0):
        # ---- fast path: persistent tcgen05 token-tile kernels, element-wise work fused into the epilogues
        P = f"{pre}encoder.layer.{i}."
        site = 10 * (i + 1)
        last = i == n_layers - 1
        qkvc = new(T, 4 * H)
        ops.linear_tile(x, fp.bf16(P + "attention.self.query.weight", 4), qkvc, ops.LT_BIAS,
                        bias=fp.f32(P + "attention.self.query.bias", 4), tag="lt_qkvc_fwd")
        ctx = new(T, H)
        ops.attn_core_fwd(ops.attn_args(R, L, H, heads, float(cfg.beta), qkvc, mask, p_att, seed, site, ctx=ctx))
        collect_maps(i, qkvc)
        Tl, x_res = T, x
        if last and compact:  # the rest of the last layer only for the rows somebody reads
            Tl = Tc
            ctx_c, x_res = new(Tc, H), new(Tc, H)
            ops.gather_rows(ctx, last_rows, ctx_c)
            ops.gather_rows(x, last_rows, x_res)
            ctx = ctx_c
        a, z1 = new(Tl, H), new(Tl, H)
        ops.linear_tile(ctx, fp.bf16(P + "attention.output.dense.weight"), a, ops.LT_RES_LN,
                        bias=fp.f32(P + "attention.output.dense.bias"), aux_out=z1, e_in=x_res,
                        ln_g=fp.f32(P + "attention.output.LayerNorm.weight"), ln_b=fp.f32(P + "attention.output.LayerNorm.bias"),
                        ln_eps=cfg.layer_norm_eps, p=p_hid, seed=seed, site=site + 3, tag="lt_res_ln_fwd")
        h_pre, h = new(Tl, I), new(Tl, I)
        ops.linear_tile(a, fp.bf16(P + "intermediate.dense.weight"), h, ops.LT_GELU,
                        bias=fp.f32(P + "intermediate.dense.bias"), aux_out=h_pre, tag="lt_gelu_fwd")
        y, z2 = new(Tl, H), new(Tl, H)
        ops.linear_tile(h, fp.bf16(P + "output.dense.weight"), y, ops.LT_RES_LN, bias=fp.f32(P + "output.dense.bias"),
                        aux_out=z2, e_in=a, ln_g=fp.f32(P + "output.LayerNorm.weight"),
                        ln_b=fp.f32(P + "output.LayerNorm.bias"), ln_eps=cfg.layer_norm_eps, p=p_hid, seed=seed,
                        site=site + 4, out_f32=(hidden_f32 if last else None), tag="lt_res_ln_fwd")
        if keep:
            run.layers.append((x, qkvc, ctx, z1, a, h_pre, h, z2))
        if outs is not None and outs.hidden and not last:
            outs.layers.append(y)
        x = y
    for i in range(0 if tile else n_layers):
        P = f"{pre}encoder.layer.{i}."
        site = 10 * (i + 1)
        qkvc = new(T, 4 * H)
        ops.linear_fwd(x, fp.bf16(P + "attention.self.query.weight", 4), fp.f32(P + "attention.self.query.bias", 4), qkvc)
        ctx = new(T, H)
        ops.attn_core_fwd(ops.attn_args(R, L, H, heads, float(cfg.beta), qkvc, mask, p_att, seed, site, ctx=ctx))
        collect_maps(i, qkvc)
        o1 = new(T, H)
        ops.linear_fwd(ctx, fp.bf16(P + "attention.output.dense.weight"), fp.f32(P + "attention.output.dense.bias"), o1)
        a = new(T, H)
        ops.res_ln_fwd(ops.resln_args(T, H, o1, x, fp.f32(P + "attention.output.LayerNorm.weight"),
                                      fp.f32(P + "attention.output.LayerNorm.bias"), cfg.layer_norm_eps, p_hid, seed,
                                      site + 3, y=a))
        h_pre = new(T, I)
        h = new(T, I)
        ops.linear_fwd(a, fp.bf16(P + "intermediate.dense.weight"), fp.f32(P + "intermediate.dense.bias"), h,
                       gelu_aux=h_pre)
        o2 = new(T, H)
        ops.linear_fwd(h, fp.bf16(P + "output.dense.weight"), fp.f32(P + "output.dense.bias"), o2)
        y = new(T, H)
        last = i == n_layers - 1
        ops.res_ln_fwd(ops.resln_args(T, H, o2, a, fp.f32(P + "output.LayerNorm.weight"),
                                      fp.f32(P + "output.LayerNorm.bias"), cfg.layer_norm_eps, p_hid, seed, site + 4,
                                      y=y, y_f32=(hidden_f32 if last else None)))
        if keep:
            run.layers.append((x, qkvc, ctx, o1, a, h_pre, h, o2))
        if outs is not None and outs.hidden and not last:
            outs.layers.append(y)
        x = y
    if n_layers == 0:
        hidden_f32 = x.float()
    return (hidden_f32 if compact else hidden_f32.view(R, L, H)), run


def _encode_backward(fp: FlatParams, pre: str, cfg: PMGTConfig, run: _EncoderRun, d_hidden: torch.Tensor,
                     arena: GradArena, pool: Optional[_BufPool] = None, d_layers: Optional[list] = None):
    """Reverse of ``_encode_forward``; parameter gradients are accumulated into ``arena``.  ``pool`` (launch plans)
    recycles the per-layer temporaries instead of leaving that to torch's allocator.

    ``d_layers`` (optional): fp32 ``[T, H]`` gradients (or None) of the inputs of layers 0 .. n-1, i.e. of the
    ``_EncoderOutputs.layers`` hidden states.  The gradient of layer k's input joins the backward pass where layer k-1's
    output LayerNorm reads its incoming gradient (its fp32 addend, otherwise unused there); that of the embedding output
    is added to the gradient the embedding backward reads."""
    H, I, heads = cfg.hidden_size, cfg.intermediate_size, cfg.num_attention_heads
    R, L, T = run.R, run.L, run.T
    dev = d_hidden.device
    seed, p_hid, p_att = run.seed, run.p_hid, run.p_att

    def new(*shape, dtype=BF16):
        if pool is not None:
            return pool.get(shape, dtype)
        return torch.empty(shape, dtype=dtype, device=dev)

    def done(*ts):
        if pool is not None:
            pool.release(*ts)

    G = arena.view
    last_rows = run.last_rows
    dy_f32 = d_hidden.contiguous().view(-1, H)
    top = cfg.num_hidden_layers - 1
    dy = None
    dy_b = None  # second gradient term of the layer input (the LayerNorm residual branch), tile path only
    deferred_dw = []
    for i in reversed(range(cfg.num_hidden_layers if run.tile else 0)):
        P = f"{pre}encoder.layer.{i}."
        site = 10 * (i + 1)
        x, qkvc, ctx, z1, a, h_pre, h, z2 = run.layers[i]
        # the last layer's post-attention half ran on the compact row set (ctx is then the gathered [Tc, H] matrix)
        compact = i == top and last_rows is not None
        Tl = int(last_rows.numel()) if compact else T
        # ---- BertOutput: LayerNorm(dropout(dense(h)) + a)
        dz2 = new(Tl, H)
        do2 = new(Tl, H) if p_hid > 0 else dz2
        ops.ln_bwd(Tl, H, z2, fp.f32(P + "output.LayerNorm.weight"), cfg.layer_norm_eps, p_hid, seed, site + 4, dz2, do2,
                   G(P + "output.LayerNorm.weight"), G(P + "output.LayerNorm.bias"), dy_a=dy, dy_b=dy_b, dy_f32=dy_f32)
        dy_f32 = None
        # each dX kernel of a 128 x 128 Linear also forms that Linear's dW / dbias from the dY tile it already holds
        fused = FUSED_DW and H == 128 and I == 128
        dh_pre = new(Tl, I)
        if fused:
            ops.linear_tile(do2, fp.bf16(P + "output.dense.weight"), dh_pre, ops.LT_GELU_BWD, w_mn=True, e_in=h_pre,
                            dw_x=h, dw=G(P + "output.dense.weight"), dbias=G(P + "output.dense.bias"), tag="lt_dxdw_gelu")
        else:
            ops.dw_tile(do2, h, G(P + "output.dense.weight"), G(P + "output.dense.bias"))
            ops.linear_tile(do2, fp.bf16(P + "output.dense.weight"), dh_pre, ops.LT_GELU_BWD, w_mn=True, e_in=h_pre,
                            tag="lt_dx_gelu")
        # ---- BertIntermediate
        da = new(Tl, H)
        if fused:
            ops.linear_tile(dh_pre, fp.bf16(P + "intermediate.dense.weight"), da, ops.LT_PLAIN, w_mn=True, dw_x=a,
                            dw=G(P + "intermediate.dense.weight"), dbias=G(P + "intermediate.dense.bias"), tag="lt_dxdw")
        else:
            ops.dw_tile(dh_pre, a, G(P + "intermediate.dense.weight"), G(P + "intermediate.dense.bias"))
            ops.linear_tile(dh_pre, fp.bf16(P + "intermediate.dense.weight"), da, ops.LT_PLAIN, w_mn=True, tag="lt_dx")
        # ---- BertSelfOutput: LayerNorm(dropout(dense(ctx)) + x); d a = da (FFN branch) + dz2 (residual branch)
        dz1 = new(Tl, H)
        do1 = new(Tl, H) if p_hid > 0 else dz1
        ops.ln_bwd(Tl, H, z1, fp.f32(P + "attention.output.LayerNorm.weight"), cfg.layer_norm_eps, p_hid, seed, site + 3,
                   dz1, do1, G(P + "attention.output.LayerNorm.weight"), G(P + "attention.output.LayerNorm.bias"),
                   dy_a=da, dy_b=dz2)
        dctx = new(Tl, H)
        if fused:
            ops.linear_tile(do1, fp.bf16(P + "attention.output.dense.weight"), dctx, ops.LT_PLAIN, w_mn=True, dw_x=ctx,
                            dw=G(P + "attention.output.dense.weight"), dbias=G(P + "attention.output.dense.bias"),
                            tag="lt_dxdw")
        else:
            ops.dw_tile(do1, ctx, G(P + "attention.output.dense.weight"), G(P + "attention.output.dense.bias"))
            ops.linear_tile(do1, fp.bf16(P + "attention.output.dense.weight"), dctx, ops.LT_PLAIN, w_mn=True, tag="lt_dx")
        if compact:
            # back to the full token set: rows outside `last_rows` carry no gradient from this layer's second half
            dctx_c, dz1_c = dctx, dz1
            dctx, dz1 = new(T, H), new(T, H)
            ops.zero_(dctx)
            ops.zero_(dz1)
            ops.scatter_rows(dctx_c, last_rows, dctx)
            ops.scatter_rows(dz1_c, last_rows, dz1)
            done(dctx_c, dz1_c)  # their last readers (the scatters; the dX kernel that read do1) are enqueued
            if do1 is dz1_c:
                do1 = dz1  # no dropout: do1 aliased the compact dz1, which has just been released
        # ---- dual-softmax attention core, then the fused Q/K/V/C projection
        dqkvc = new(T, 4 * H)
        ops.attn_core_bwd(ops.attn_args(R, L, H, heads, float(cfg.beta), qkvc, run.mask, p_att, seed, site, dctx=dctx,
                                        dqkvc=dqkvc))
        if BATCH_DW_QKVC:
            # the Q/K/V/C weight gradient is not needed before the optimizer: all layers share ONE launch at the end
            deferred_dw.append((dqkvc, x, G(P + "attention.self.query.weight", 4), G(P + "attention.self.query.bias", 4)))
        else:
            ops.dw_tile(dqkvc, x, G(P + "attention.self.query.weight", 4), G(P + "attention.self.query.bias", 4))
        dx = new(T, H)
        ops.linear_tile(dqkvc, fp.bf16(P + "attention.self.query.weight", 4), dx, ops.LT_PLAIN, w_mn=True, tag="lt_dx_qkvc")
        done(dy, dy_b, dz2, do2, dh_pre, da, dctx, *((do1,) if do1 is not dz1 else ()),
             *(() if BATCH_DW_QKVC else (dqkvc,)))
        dy, dy_b = dx, dz1  # d x = dx (projection branch) + dz1 (residual branch): summed by the consumer
        if d_layers is not None and i > 0:
            dy_f32 = d_layers[i]  # a loss on the hidden state between layers i - 1 and i
    if deferred_dw:
        ops.dw_tile_batch(deferred_dw)
        done(*(d[0] for d in deferred_dw))
    for i in reversed(range(0 if run.tile else cfg.num_hidden_layers)):
        P = f"{pre}encoder.layer.{i}."
        site = 10 * (i + 1)
        x, qkvc, ctx, o1, a, h_pre, h, o2 = run.layers[i]
        # ---- BertOutput: LayerNorm(dropout(dense(h)) + a)
        dz2 = new(T, H)
        do2 = new(T, H) if p_hid > 0 else dz2
        ops.res_ln_bwd(ops.resln_args(T, H, o2, a, fp.f32(P + "output.LayerNorm.weight"), None, cfg.layer_norm_eps,
                                      p_hid, seed, site + 4, dy=dy, dy_f32=dy_f32, dz=dz2, d_o=do2,
                                      d_g=G(P + "output.LayerNorm.weight"), d_b=G(P + "output.LayerNorm.bias"),
                                      d_bias=G(P + "output.dense.bias")))
        dy_f32 = None
        ops.linear_dw(do2, h, G(P + "output.dense.weight"))
        dh_pre = new(T, I)
        ops.linear_dx(do2, fp.bf16(P + "output.dense.weight"), dh_pre, gelu_bwd_aux=h_pre)
        # ---- BertIntermediate
        ops.colsum(dh_pre, G(P + "intermediate.dense.bias"))
        ops.linear_dw(dh_pre, a, G(P + "intermediate.dense.weight"))
        da = new(T, H)
        ops.linear_dx(dh_pre, fp.bf16(P + "intermediate.dense.weight"), da, addend=dz2)
        # ---- BertSelfOutput: LayerNorm(dropout(dense(ctx)) + x)
        dz1 = new(T, H)
        do1 = new(T, H) if p_hid > 0 else dz1
        ops.res_ln_bwd(ops.resln_args(T, H, o1, x, fp.f32(P + "attention.output.LayerNorm.weight"), None,
                                      cfg.layer_norm_eps, p_hid, seed, site + 3, dy=da, dz=dz1, d_o=do1,
                                      d_g=G(P + "attention.output.LayerNorm.weight"),
                                      d_b=G(P + "attention.output.LayerNorm.bias"),
                                      d_bias=G(P + "attention.output.dense.bias")))
        ops.linear_dw(do1, ctx, G(P + "attention.output.dense.weight"))
        dctx = new(T, H)
        ops.linear_dx(do1, fp.bf16(P + "attention.output.dense.weight"), dctx)
        # ---- dual-softmax attention core
        dqkvc = new(T, 4 * H)
        ops.attn_core_bwd(ops.attn_args(R, L, H, heads, float(cfg.beta), qkvc, run.mask, p_att, seed, site, dctx=dctx,
                                        dqkvc=dqkvc, d_bias_qkvc=G(P + "attention.self.query.bias", 4)))
        ops.linear_dw(dqkvc, x, G(P + "attention.self.query.weight", 4))
        dx = new(T, H)
        ops.linear_dx(dqkvc, fp.bf16(P + "attention.self.query.weight", 4), dx, addend=dz1)
        dy = dx
        if d_layers is not None and i > 0:
            dy_f32 = d_layers[i]  # a loss on the hidden state between layers i - 1 and i
    if dy is None:  # zero layers
        dy = dy_f32.to(BF16)
        dy_b = None
    elif d_layers is not None and d_layers[0] is not None:  # a loss on the embedding output
        if dy_b is None:
            dy_b = new(T, H)
            ops.cast_f32_bf16(d_layers[0], dy_b)
        else:
            dy_b = (dy_b.float() + d_layers[0].view(T, H)).to(BF16)
    if fp.after_layers_hook is not None:
        ops.host_hook(fp.after_layers_hook, arena)
    # ---- embeddings
    E = pre + "embeddings."
    n_mod = len(run.src)
    common = dict(dx=dy, dx_b=dy_b, d_w_att=G(E + "attention.1.weight"), d_b_att=G(E + "attention.1.bias"),
                  d_pos=G(E + "position_embeddings.weight"), d_role=G(E + "role_embeddings.weight"),
                  d_ln_g=G(E + "LayerNorm.weight"), d_ln_b=G(E + "LayerNorm.bias"),
                  d_bias=[G(f"{E}feat_linear.{m}.bias") for m in range(n_mod)])
    eargs = (R, L, H, run.proj, fp.f32(E + "attention.1.weight"), fp.f32(E + "attention.1.bias"),
             fp.f32(E + "position_embeddings.weight"), fp.f32(E + "role_embeddings.weight"),
             fp.f32(E + "LayerNorm.weight"), fp.f32(E + "LayerNorm.bias"), cfg.layer_norm_eps, p_hid, seed, 0)
    if run.dense_tables:
        # per-table-row gradient of the projected rows (fp32 red.add), then ONE dense dW GEMM per modality
        accs = [new(n, H, dtype=torch.float32) for n in run.src_rows]
        for acc in accs:
            ops.zero_(acc)
        skip0 = int(all(getattr(t, "_pmgt_row0_zero", False) for t in run.src))
        ops.embed_multi_bwd(ops.embed_multi_args(*eargs, row_idx=run.rows_idx, de_acc=accs, skip_row0=skip0, **common))
        for m in range(n_mod):
            d16 = new(run.src_rows[m], H)
            ops.cast_f32_bf16(accs[m].view(-1), d16.view(-1))
            ops.linear_dw(d16, run.src[m], G(f"{E}feat_linear.{m}.weight"), tag="gemm_dw_table")
    else:
        des = [new(T, H) for _ in range(n_mod)]
        ops.embed_multi_bwd(ops.embed_multi_args(*eargs, de=des, **common))
        for m, d in enumerate(des):
            ops.linear_dw(d, run.src[m], G(f"{E}feat_linear.{m}.weight"), rows=run.rows_idx,
                          src_rows=(run.src_rows[m] if run.rows_idx is not None else 0), x_cols=run.src[m].shape[1])


class _EncodeFn(torch.autograd.Function):
    """Autograd node for one batched encoder pass.  ``params`` are passed only so
    that autograd routes their gradients; the data is read from ``fp``.

    With ``outs`` (per-layer outputs requested) the pass is never planned, and the fp32 ``[T, H]`` copies of
    ``outs.layers`` are further outputs of the node, so their gradients reach the backward pass."""

    @staticmethod
    def forward(ctx, host, src, rows_idx, mask, R, L, training, seed, arena, keep, last_rows, outs, *params):
        fp, pre, cfg = host._fp, host._fp_prefix, host.config
        plan = host._plan_for(fp, src, rows_idx, R, L, training, keep, arena, last_rows) if outs is None else None
        host._active_plan = plan
        if plan is not None:
            hidden, run = plan.forward(fp, pre, cfg, src, rows_idx, mask, training, seed, keep, last_rows), None
        else:
            hidden, run = _encode_forward(fp, pre, cfg, src, rows_idx, R, L, mask, training, seed, keep,
                                          last_rows=last_rows, outs=outs)
        ctx.host, ctx.run, ctx.arena, ctx.n_params, ctx.plan, ctx.keep = host, run, arena, len(params), plan, keep
        ctx.hidden_shape = hidden.shape
        if outs is None or not outs.hidden:
            return hidden
        ctx.set_materialize_grads(False)  # an output nobody differentiates arrives as None, not as zeros
        return (hidden,) + tuple(x.float() for x in outs.layers)

    @staticmethod
    def backward(ctx, d_hidden, *d_layers):
        host, run, arena, plan = ctx.host, ctx.run, ctx.arena, ctx.plan
        fp, pre, cfg = host._fp, host._fp_prefix, host.config
        if d_layers:
            if d_hidden is None:
                d_hidden = torch.zeros(ctx.hidden_shape, dtype=torch.float32, device=arena.fp.flat.device)
            d_layers = [None if d is None else d.to(torch.float32).contiguous() for d in d_layers]
            if all(d is None for d in d_layers):
                d_layers = None
        else:
            d_layers = None
        if plan is not None:
            if not ctx.keep or not plan.pending_backward:
                raise PMGTError("encoder backward called but the launch plan holds no activations for it")
            plan.backward(fp, pre, cfg, d_hidden, arena)
        else:
            if run is None:
                raise PMGTError("encoder backward called but activations were not kept")
            _encode_backward(fp, pre, cfg, run, d_hidden, arena, d_layers=d_layers)
            ctx.run = None
        grads = tuple(arena.view(n) for n in host._encoder_param_names)
        return (None,) * 12 + grads


class _AttentionMapFn(torch.autograd.Function):
    """Identity on an attention map that puts it into the autograd graph of the encoder pass (``anchor``) only to
    refuse a backward pass through it: its gradient would need a new input to the backward kernel of every attention
    family.  Without this node such a gradient would silently be dropped."""

    @staticmethod
    def forward(ctx, maps, anchor):
        return maps.view_as(maps)

    @staticmethod
    def backward(ctx, g, _g_anchor=None):
        raise NotImplementedError("attention maps (output_attentions) are not differentiable; detach them before "
                                  "using them in a loss")


class PMGTPretrainedModel(nn.Module):
    """Weight init of modeling_pmgt.py:34-62 (N(0, initializer_range) for Linear /
    Embedding weights, zeros for biases, ones/zeros for LayerNorm)."""

    config_class = PMGTConfig
    base_model_prefix = "pmgt"
    supports_gradient_checkpointing = True

    def __init__(self, config):
        super().__init__()
        self.config = config

    def _init_weights(self, module):
        if isinstance(module, nn.Linear):
            module.weight.data.normal_(mean=0.0, std=self.config.initializer_range)
            if module.bias is not None:
                module.bias.data.zero_()
        elif isinstance(module, nn.Embedding):
            module.weight.data.normal_(mean=0.0, std=self.config.initializer_range)
            if module.padding_idx is not None:
                module.weight.data[module.padding_idx].zero_()
        elif isinstance(module, nn.LayerNorm):
            module.bias.data.zero_()
            module.weight.data.fill_(1.0)

    def init_weights(self):
        self.apply(self._init_weights)

    @property
    def dtype(self):
        return torch.float32


def resolve_output_flags(config, output_attentions, output_hidden_states):
    """transformers' rule: an explicit argument wins, otherwise the config's flag (False by default)."""
    oa = output_attentions if output_attentions is not None else getattr(config, "output_attentions", False)
    oh = output_hidden_states if output_hidden_states is not None else getattr(config, "output_hidden_states", False)
    return bool(oa), bool(oh)


def output_tuple(hidden_states, attentions) -> tuple:
    """The optional tail of a ``return_dict=False`` tuple: ``hidden_states``, then ``attentions``, each if requested."""
    return tuple(t for t in (hidden_states, attentions) if t is not None)


_seed_counter = [0]


def next_dropout_seed() -> int:
    """A fresh 64-bit Philox seed per forward pass, derived from torch's seed."""
    _seed_counter[0] += 1
    return (torch.initial_seed() * 0x9E3779B97F4A7C15 + _seed_counter[0] * 0xD1342543DE82EF95) & 0xFFFFFFFFFFFFFFFF


class PMGTModel(PMGTPretrainedModel):
    """modeling_pmgt.py:65-152.  ``forward(*input_feat_embeds, attention_mask=...)``
    keeps the reference signature (dense per-modality features); the fused
    gather path used by ``PMGT`` is ``encode_ids``."""

    def __init__(self, config, add_pooling_layer=False):
        super().__init__(config)
        if add_pooling_layer:
            raise ValueError("the reference never enables the pooler (modeling_pmgt.py:66-72); not implemented")
        self.embeddings = PMGTEmbeddings(config)
        self.encoder = PMGTEncoder(config)
        self.pooler = None
        self.init_weights()
        self._fp = None
        self._fp_prefix = ""
        self._encoder_param_names = [n for n, _ in encoder_param_order(self)]
        self.use_launch_plans = False  # opt-in: outputs of a planned pass alias plan-owned buffers (see _EncoderPlan)
        self._plans = {}
        self._active_plan = None

    def _plan_for(self, fp, src, rows_idx, R, L, training, keep, arena, last_rows=None) -> Optional["_EncoderPlan"]:
        """The launch plan for this call, or None when plans are off or the call is not plannable (dense inputs,
        a transient gradient arena, or a forward whose backward is still outstanding on the same plan)."""
        if not self.use_launch_plans or rows_idx is None or (keep and not getattr(arena, "persistent", False)):
            return None
        cfg = self.config
        key = (R, L, bool(training), bool(keep), float(cfg.hidden_dropout_prob), float(cfg.attention_probs_dropout_prob),
               tuple((t.data_ptr(), tuple(t.shape)) for t in src), fp.flat.data_ptr(), fp.flat_bf16.data_ptr(),
               arena.get().data_ptr() if keep else 0, ops.cur_stream(), PROJECTION_MODE,
               int(last_rows.numel()) if last_rows is not None else -1)
        plan = self._plans.get(key)
        if plan is None:
            if len(self._plans) >= 4:  # e.g. full batch, tail batch, eval batch; drop the oldest beyond that
                self._plans.pop(next(iter(self._plans)))
            plan = _EncoderPlan(key, R, L, cfg.hidden_size, rows_idx.device,
                                n_last=int(last_rows.numel()) if last_rows is not None else 0)
            self._plans[key] = plan
        elif plan.pending_backward:
            return None
        return plan

    # -- flat storage: standalone use owns its own FlatParams; inside PMGT the parent's is shared
    def _attach(self, fp: FlatParams, prefix: str):
        self._fp, self._fp_prefix = fp, prefix
        self._encoder_param_names = [prefix + n for n, _ in encoder_param_order(self)]

    def _flat(self) -> FlatParams:
        if self._fp is None:
            self._fp = FlatParams(encoder_param_order(self))
        return self._fp.ensure()

    def _encoder_params(self):
        ps = self.__dict__.get("_encoder_params_cache")
        if ps is None:  # Parameter objects keep their identity across .to() / load_state_dict
            ps = [p for _, p in encoder_param_order(self)]
            self.__dict__["_encoder_params_cache"] = ps
        return ps

    def encode(self, src, rows_idx, mask, R, L, arena=None, refresh=True, last_rows=None, *,
               output_hidden_states=False, output_attentions=False, output_rows=None):
        """``src``: one bf16 source per modality (feature tables gathered through ``rows_idx``, or dense ``[R * L, D]``
        matrices when ``rows_idx`` is None).  ``last_rows`` (sorted unique token indices): return only those rows of
        the final hidden state, as a ``[len(last_rows), H]`` matrix; on the token-tile path the last layer's
        post-attention half is then computed for those rows only (see ``_encode_forward``).

        ``output_hidden_states`` / ``output_attentions``: return ``(hidden, hidden_states, attentions)`` instead, for
        the first ``output_rows`` sequences (default all ``R``).  ``hidden_states`` is a tuple of
        ``num_hidden_layers`` fp32 ``[output_rows, L, H]`` tensors, the embedding output and the outputs of layers
        1 .. n-1 (bf16 activations widened to fp32; the last layer's output is ``hidden``), and is differentiable.
        ``attentions`` is a tuple of ``num_hidden_layers`` fp32 ``[output_rows, heads, L, L]`` tensors, the matrices
        each layer multiplied V with (with this pass's dropout mask); a backward pass through one raises
        ``NotImplementedError``.  Either is None when not requested.  Such a call never uses a launch plan.

        Raises ``ValueError``, before any device work, for a context longer than the position table or than the
        attention core's limit (MAX_CONTEXT_LEN tokens)."""
        check_context_len(self.config, L)
        fp = self._flat()
        if refresh:
            fp.refresh_bf16()
        if arena is None:
            arena = GradArena(fp)
        seed = next_dropout_seed()
        mask = mask.to(torch.float32).contiguous()
        params = self._encoder_params()
        keep = torch.is_grad_enabled() and any(p.requires_grad for p in params)
        cfg = self.config
        in_kernel = (last_rows is not None and cfg.num_hidden_layers > 0
                     and _tile_path(cfg.hidden_size, cfg.intermediate_size))
        src = tuple(src)
        if len(src) != len(cfg.feat_hidden_sizes):
            raise PMGTError(f"encode: {len(src)} feature sources for {len(cfg.feat_hidden_sizes)} modalities")
        want = bool(output_hidden_states or output_attentions)
        n_out = R if output_rows is None else int(output_rows)
        outs = _EncoderOutputs(bool(output_hidden_states), bool(output_attentions), n_out) if want else None
        out = _EncodeFn.apply(self, src, rows_idx, mask, R, L, self.training, seed, arena, keep,
                              last_rows if in_kernel else None, outs, *params)
        layers = ()
        if isinstance(out, tuple):
            out, *layers = out
        if last_rows is not None and not in_kernel:  # other widths: encode everything, then pick the rows
            self._active_plan = None  # the gradient of the picked rows does not line up with the plan's buffer
            out = out.reshape(R * L, -1).index_select(0, last_rows)
        if not want:
            return out
        hidden_states = tuple(h.view(R, L, -1)[:n_out] for h in layers) if output_hidden_states else None
        attentions = None
        if output_attentions:
            attentions = tuple(_AttentionMapFn.apply(m, out) if out.requires_grad else m for m in outs.maps)
        return out, hidden_states, attentions

    def forward(self, *input_feat_embeds, attention_mask=None, head_mask=None, output_attentions=None,
                output_hidden_states=None, return_dict=None):
        """modeling_pmgt.py:80-152.  ``output_hidden_states`` / ``output_attentions`` (default: the config's) follow
        transformers:

        * ``hidden_states``: ``num_hidden_layers + 1`` fp32 ``[R, L, H]`` tensors, the embedding output and the output
          of every layer; the last is ``last_hidden_state`` itself.  The others are the bf16 activations the encoder
          keeps, widened to fp32.  They are differentiable: a loss on entry k reaches the parameters through the
          backward pass of the layers below it.
        * ``attentions``: ``num_hidden_layers`` fp32 ``[R, heads, L, L]`` tensors.  Entry k is the matrix layer k
          multiplies the values with, ``beta * dropout(P1) + (1 - beta) * dropout(P2)`` (P1 the cosine softmax of the
          context projections, P2 the scaled dot-product softmax, both with the -10000 key mask): rows sum to 1 in
          eval mode, and in training they carry the dropout mask this pass applied.  They are not differentiable; a
          backward pass through one raises ``NotImplementedError``.  They take ``4 * heads * L^2`` bytes per sequence
          and layer (335 MB for 1,024 sequences of 128 tokens and 5 layers).

        With ``return_dict=False`` they are appended to the tuple, ``hidden_states`` first, only when requested.  A call
        that requests either never uses a launch plan.  ``head_mask`` is not supported."""
        assert len(input_feat_embeds) == len(self.config.feat_hidden_sizes), \
            f"# of multi-modal features must be {len(self.config.feat_hidden_sizes)}"
        first = input_feat_embeds[0]
        assert all(first.size()[:-1] == f.size()[:-1] for f in input_feat_embeds[1:]), \
            "All features are same dim except last one"
        if head_mask is not None:
            raise NotImplementedError("head_mask is not supported by the fused attention kernels (the reference's "
                                      "trainer never passes one)")
        output_attentions, output_hidden_states = resolve_output_flags(self.config, output_attentions,
                                                                       output_hidden_states)
        if not first.is_cuda:
            raise PMGTError("PMGTModel.forward needs CUDA tensors: pmgt_b200 has no CPU fallback")
        R, L = first.shape[:2]
        return_dict = return_dict if return_dict is not None else self.config.use_return_dict
        if attention_mask is None:
            attention_mask = torch.ones(R, L, device=first.device)
        dense = [f.reshape(R * L, f.shape[-1]).to(BF16).contiguous() for f in input_feat_embeds]
        hidden_states = attentions = None
        if output_attentions or output_hidden_states:
            seq, inner, attentions = self.encode(dense, None, attention_mask, R, L,
                                                 output_hidden_states=output_hidden_states,
                                                 output_attentions=output_attentions)
            if output_hidden_states:
                hidden_states = inner + (seq,)
        else:
            seq = self.encode(dense, None, attention_mask, R, L)
        if not return_dict:
            return (seq, None) + output_tuple(hidden_states, attentions)
        return BaseModelOutputWithPooling(last_hidden_state=seq, pooler_output=None, hidden_states=hidden_states,
                                          attentions=attentions)


# ---------------------------------------------------------------------------
# losses
# ---------------------------------------------------------------------------
class _GsrFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, tgt_h0, pair_h0, pair_off, labels):
        B, H = tgt_h0.shape
        SP = pair_h0.shape[0]
        dev = tgt_h0.device
        tgt_h0 = tgt_h0 if tgt_h0.stride(1) == 1 else tgt_h0.contiguous()
        pair_h0 = pair_h0 if pair_h0.stride(1) == 1 else pair_h0.contiguous()
        logits = torch.empty(SP, dtype=torch.float32, device=dev)
        loss = torch.zeros((), dtype=torch.float32, device=dev)
        ops.gsr(True, B, SP, H, tgt_h0, tgt_h0.stride(0), pair_h0, pair_h0.stride(0), pair_off, labels, logits=logits,
                loss_out=loss)
        ctx.save_for_backward(tgt_h0, pair_h0, pair_off, labels)
        ctx.mark_non_differentiable(logits)
        return loss, logits

    @staticmethod
    def backward(ctx, g_loss, _g_logits):
        tgt_h0, pair_h0, pair_off, labels = ctx.saved_tensors
        B, H = tgt_h0.shape
        SP = pair_h0.shape[0]
        d_t = torch.empty(B, H, dtype=torch.float32, device=tgt_h0.device)
        d_p = torch.zeros(SP, H, dtype=torch.float32, device=tgt_h0.device)
        g = g_loss.to(torch.float32).contiguous()
        ops.gsr(False, B, SP, H, tgt_h0, tgt_h0.stride(0), pair_h0, pair_h0.stride(0), pair_off, labels, grad_out=g,
                d_tgt=d_t, d_pair=d_p)
        return d_t, d_p, None, None


class PMGTGraphConstructLoss(nn.Module):
    """modeling_pmgt.py:537-546.  ``forward(hidden_states, other_hidden_states,
    labels)`` keeps the reference's per-target signature; ``batched`` is the
    whole-batch form PMGT uses (one launch instead of a Python loop with a
    device sync per target, models.py:111-124)."""

    def __init__(self, config=None):
        super().__init__()

    def forward(self, hidden_states, other_hidden_states, labels):
        off = torch.tensor([0, hidden_states.shape[0]], dtype=torch.int64, device=hidden_states.device)
        loss, logits = _GsrFn.apply(other_hidden_states.reshape(1, -1).float(), hidden_states.float(), off,
                                    labels.float().contiguous())
        return loss, logits

    @staticmethod
    def batched(tgt_h0, pair_h0, pair_off, labels):
        return _GsrFn.apply(tgt_h0, pair_h0, pair_off, labels)


class _NfrFn(torch.autograd.Function):
    """Projections (tensor-core GEMM) + MSE against gathered table rows, both modalities."""

    @staticmethod
    def forward(ctx, host, h_masked, target_ids, tables, arena, *params):
        fp, pre = host._fp, host._fp_prefix
        Mm, H = h_masked.shape
        dev = h_masked.device
        loss = torch.zeros((), dtype=torch.float32, device=dev)
        hb = h_masked.to(BF16).contiguous()
        projs = []
        n_mod = len(tables)
        for m, table in enumerate(tables):
            D = table.shape[1]
            proj = torch.empty(Mm, D, dtype=BF16, device=dev)
            if Mm > 0:
                ops.linear_fwd(hb, fp.bf16(f"{pre}projections.{m}.weight"), fp.f32(f"{pre}projections.{m}.bias"), proj)
            ops.nfr_mse(True, Mm, D, proj, table, target_ids, 1.0 / n_mod, loss_out=loss)
            projs.append(proj)
        ctx.host, ctx.arena, ctx.tables, ctx.n_params = host, arena, tables, len(params)
        ctx.save_for_backward(hb, target_ids, *projs)
        return loss

    @staticmethod
    def backward(ctx, g_loss):
        host, arena, tables = ctx.host, ctx.arena, ctx.tables
        fp, pre = host._fp, host._fp_prefix
        hb, target_ids, *projs = ctx.saved_tensors
        Mm, H = hb.shape
        dev = hb.device
        g = g_loss.to(torch.float32).contiguous()
        dh = None
        n_mod = len(tables)
        for m, table in enumerate(tables):
            D = table.shape[1]
            if Mm == 0:
                continue
            dproj = torch.empty(Mm, D, dtype=BF16, device=dev)
            ops.nfr_mse(False, Mm, D, projs[m], table, target_ids, 1.0 / n_mod, grad_out=g, dproj=dproj)
            ops.colsum(dproj, arena.view(f"{pre}projections.{m}.bias"))
            ops.linear_dw(dproj, hb, arena.view(f"{pre}projections.{m}.weight"))
            out = torch.empty(Mm, H, dtype=BF16, device=dev)
            ops.linear_dx(dproj, fp.bf16(f"{pre}projections.{m}.weight"), out, addend=dh)
            dh = out
        d_h = dh.float() if dh is not None else torch.zeros(Mm, H, dtype=torch.float32, device=dev)
        grads = tuple(arena.view(n) for n in host._param_names)
        return (None, d_h, None, None, None) + grads


class PMGTNodeConstructLoss(nn.Module):
    """modeling_pmgt.py:549-569."""

    def __init__(self, config):
        super().__init__()
        self.projections = nn.ModuleList([nn.Linear(config.hidden_size, d) for d in config.feat_hidden_sizes])
        self._fp = None
        self._fp_prefix = ""
        self._param_names = [n for n, _ in self.param_order()]

    def param_order(self, prefix: str = ""):
        out = []
        for m, l in enumerate(self.projections):
            out += [(f"{prefix}projections.{m}.weight", l.weight), (f"{prefix}projections.{m}.bias", l.bias)]
        return out

    def _attach(self, fp: FlatParams, prefix: str):
        self._fp, self._fp_prefix = fp, prefix
        self._param_names = [n for n, _ in self.param_order(prefix)]

    def from_ids(self, h_masked, target_ids, tables_bf16, arena=None):
        if self._fp is None:
            self._fp = FlatParams(self.param_order())
        fp = self._fp.ensure()
        if arena is None:
            fp.refresh_bf16()
            arena = GradArena(fp)
        return _NfrFn.apply(self, h_masked, target_ids, tables_bf16, arena, *[p for _, p in self.param_order()])

    def forward(self, inputs, targets):
        """Reference signature: ``targets`` are the already-gathered feature rows."""
        assert len(targets) == len(self.projections), f"# of multi-modal features must be {len(self.projections)}"
        ids = torch.arange(inputs.shape[0], dtype=torch.int64, device=inputs.device)
        tables = [t.to(BF16).contiguous() for t in targets]
        return self.from_ids(inputs, ids, tables)
