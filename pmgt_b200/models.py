"""Host-side mirror of ``pmgt/pmgt/models.py``: the ``PMGT`` pre-training module.

Same constructor / ``forward`` signature, outputs and state-dict keys as the
reference.  What changed underneath:

* the reference encodes the pair contexts in a Python loop over targets with a
  device->host sync per target (models.py:111-124) and runs three separate
  encoder calls; here targets, all pairs and the masked targets go through ONE
  batched encoder pass (rows are independent, so the math is identical);
* feature rows are gathered inside the projection GEMM from bf16 copies of the
  frozen tables instead of being materialised by ``nn.Embedding``;
* both losses are fused reduction kernels.

The NFR corruption (models.py:131-151) stays host PyTorch code issued in the
reference's order, so the same ``torch.manual_seed`` corrupts the same nodes.
"""
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.nn as nn

from ._lib import PMGTError
from .configuration_pmgt import PMGTConfig
from .modeling_pmgt import (BF16, FlatParams, GradArena, PMGTForPreTrainingOutput, PMGTGraphConstructLoss, PMGTModel,
                            PMGTNodeConstructLoss, PMGTPretrainedModel, encoder_param_order, output_tuple,
                            resolve_output_flags)
from .utils import get_input_feat_embeds  # noqa: F401  (re-exported like the reference module)


class _PretrainLossFn(torch.autograd.Function):
    """GSR + NFR losses of one batch straight from the encoder's compact hidden-state matrix, and their gradient
    written straight into the buffer the encoder's backward pass reads.

    ``hidden`` is ``[B*L + SP (+ B*L), H]`` fp32: every position of the targets, position 0 of the pairs, (training)
    every position of the masked targets.  The GSR kernel reads the target / pair rows through strides (no gather),
    NFR gathers its ~0.16 * B * (L - 1) masked rows; backward zeroes the gradient buffer once, the GSR kernel writes
    its rows through the same strides and the NFR rows are copied in.  This replaces an index_select of ~48k rows,
    three slice-backward zero-fills / adds and an index_copy per step with two small gathers (models.py:104-162)."""

    @staticmethod
    def forward(ctx, host, hidden, B, SP, L, pair_off, labels, nfr_rows, target_idx, tables, arena, grad_buf, *params):
        from . import ops
        H = hidden.shape[1]
        dev = hidden.device
        hidden = hidden if hidden.is_contiguous() else hidden.contiguous()
        tgt = hidden[: B * L].view(B, L, H)[:, 0]            # stride L * H
        pair = hidden[B * L: B * L + SP]
        logits = torch.empty(SP, dtype=torch.float32, device=dev)
        loss = torch.zeros((), dtype=torch.float32, device=dev)
        ops.gsr(True, B, SP, H, tgt, tgt.stride(0), pair, pair.stride(0), pair_off, labels, logits=logits, loss_out=loss)
        saved = [hidden, pair_off, labels]
        ctx.n_mod = 0
        if nfr_rows is not None:
            nfr = host.nfr_loss
            fp, pre = nfr._fp, nfr._fp_prefix
            Mm = int(nfr_rows.numel())
            hb = hidden.index_select(0, nfr_rows).to(BF16) if Mm > 0 else torch.empty(0, H, dtype=BF16, device=dev)
            projs = []
            for m, table in enumerate(tables):
                D = table.shape[1]
                proj = torch.empty(Mm, D, dtype=BF16, device=dev)
                if Mm > 0:
                    ops.linear_fwd(hb, fp.bf16(f"{pre}projections.{m}.weight"), fp.f32(f"{pre}projections.{m}.bias"), proj)
                ops.nfr_mse(True, Mm, D, proj, table, target_idx, 1.0 / len(tables), loss_out=loss)   # adds into `loss`
                projs.append(proj)
            saved += [nfr_rows, target_idx, hb, *projs]
            ctx.n_mod = len(tables)
        ctx.save_for_backward(*saved)
        ctx.host, ctx.arena, ctx.tables, ctx.grad_buf, ctx.dims = host, arena, tables, grad_buf, (B, SP, L, H)
        ctx.n_params = len(params)
        ctx.mark_non_differentiable(logits)
        return loss, logits

    @staticmethod
    def backward(ctx, g_loss, _g_logits):
        from . import ops
        host, arena, tables = ctx.host, ctx.arena, ctx.tables
        B, SP, L, H = ctx.dims
        hidden, pair_off, labels, *rest = ctx.saved_tensors
        out = ctx.grad_buf
        if out is not None and out.shape == hidden.shape and out.dtype == torch.float32:
            out.zero_()
        else:
            out = torch.zeros_like(hidden)
        g = g_loss.to(torch.float32).contiguous()
        tgt = hidden[: B * L].view(B, L, H)[:, 0]
        pair = hidden[B * L: B * L + SP]
        d_t = out[: B * L].view(B, L, H)[:, 0]
        d_p = out[B * L: B * L + SP]
        ops.gsr(False, B, SP, H, tgt, tgt.stride(0), pair, pair.stride(0), pair_off, labels, grad_out=g, d_tgt=d_t, d_pair=d_p)
        grads = (None,) * ctx.n_params
        if ctx.n_mod:
            nfr = host.nfr_loss
            fp, pre = nfr._fp, nfr._fp_prefix
            nfr_rows, target_idx, hb, *projs = rest
            Mm = hb.shape[0]
            dh = None
            for m, table in enumerate(tables):
                if Mm == 0:
                    continue
                D = table.shape[1]
                dproj = torch.empty(Mm, D, dtype=BF16, device=hb.device)
                ops.nfr_mse(False, Mm, D, projs[m], table, target_idx, 1.0 / len(tables), grad_out=g, dproj=dproj)
                ops.colsum(dproj, arena.view(f"{pre}projections.{m}.bias"))
                ops.linear_dw(dproj, hb, arena.view(f"{pre}projections.{m}.weight"))
                o = torch.empty(Mm, H, dtype=BF16, device=hb.device)
                ops.linear_dx(dproj, fp.bf16(f"{pre}projections.{m}.weight"), o, addend=dh)
                dh = o
            if dh is not None:
                out.index_copy_(0, nfr_rows, dh.float())     # masked rows: disjoint from the rows GSR wrote
            grads = tuple(arena.view(n) for n in nfr._param_names)
        return (None, out) + (None,) * 10 + grads


class PMGT(PMGTPretrainedModel):
    def __init__(
        self,
        node_size: int,
        random_node_ratio: float = 0.2 * 0.1,
        mask_node_ratio: float = 0.2 * 0.8,
        config: PMGTConfig = None,
        feat_init_emb: Optional[List[np.ndarray]] = None,
    ) -> None:
        config = config if config is not None else PMGTConfig()
        super().__init__(config)
        if feat_init_emb is None:
            # the reference would TRAIN randomly initialised tables in this case (models.py:49-54 freezes them only when
            # feat_init_emb is given); the bf16 gather path here treats the tables as a frozen feature store
            import warnings
            warnings.warn("PMGT(feat_init_emb=None): feature tables are randomly initialised and stay frozen; the "
                          "reference would train them. Pass the visual / textual feature matrices.", stacklevel=2)
        self.node_size = node_size
        self.random_node_ratio = random_node_ratio
        self.mask_node_ratio = mask_node_ratio
        self.config = config
        self.bert = PMGTModel(config)
        self.gsr_loss = PMGTGraphConstructLoss(config)
        self.nfr_loss = PMGTNodeConstructLoss(config)

        # idx 0 is <pad>, idx 1 is <mask> (models.py:40-47).  The tables are frozen
        # feature stores; torch tensors (any device / dtype) are adopted without a copy.
        tables = []
        for m, d in enumerate(config.feat_hidden_sizes):
            if feat_init_emb is not None and isinstance(feat_init_emb[m], torch.Tensor):
                w = feat_init_emb[m]
                assert tuple(w.shape) == (node_size + 2, d), f"feature table {m} must be {(node_size + 2, d)}"
                emb = nn.Embedding(1, 1, padding_idx=0)
                emb.num_embeddings, emb.embedding_dim = node_size + 2, d
                emb.weight = nn.Parameter(w, requires_grad=False)
            else:
                emb = nn.Embedding(node_size + 2, d, padding_idx=0)
                if feat_init_emb is not None:
                    with torch.no_grad():
                        emb.weight.copy_(torch.from_numpy(np.asarray(feat_init_emb[m])))
            emb.requires_grad_(False)
            tables.append(emb)
        if feat_init_emb is not None:
            assert len(feat_init_emb) == len(tables)
        self.feat_embeddings = nn.ModuleList(tables)

        self._root_fp = None
        self._tables_bf16 = None
        self._tables_key = None

    # ------------------------------------------------------------------
    def _flat(self) -> FlatParams:
        if self._root_fp is None:
            order = encoder_param_order(self.bert, "bert.") + self.nfr_loss.param_order("nfr_loss.")
            self._root_fp = FlatParams(order)
            self.bert._attach(self._root_fp, "bert.")
            self.nfr_loss._attach(self._root_fp, "nfr_loss.")
        return self._root_fp.ensure()

    def flat_parameters(self) -> torch.Tensor:
        """All trainable parameters as one fp32 vector (views, FlatParams order)."""
        return self._flat().flat

    def flat_decay_mask(self, no_decay=("bias", "LayerNorm.weight")) -> torch.Tensor:
        """uint8 per element: 1 where weight decay applies (base_trainer.py:35-59)."""
        fp = self._flat()
        mask = torch.zeros(fp.total, dtype=torch.uint8)
        for n, p in zip(fp.names, fp.params):
            if not any(nd in n for nd in no_decay):
                mask[fp.offsets[n]: fp.offsets[n] + p.numel()] = 1
        return mask.to(fp.flat.device)

    def feature_tables_bf16(self) -> List[torch.Tensor]:
        """bf16 device copies of the frozen feature tables (built once, rebuilt if the tables change)."""
        key = tuple((e.weight.data_ptr(), e.weight._version, str(e.weight.device)) for e in self.feat_embeddings)
        if self._tables_bf16 is None or key != self._tables_key:
            out = []
            for e in self.feat_embeddings:
                w = e.weight.data
                if not w.is_cuda:
                    raise PMGTError("PMGT must be moved to a CUDA device before forward (no CPU fallback)")
                t = w if w.dtype == BF16 else w.to(BF16).contiguous()
                # <pad> row all zero (the reference's tables, notebook cell 30): its gradient rows are never needed
                t._pmgt_row0_zero = bool((t[0] == 0).all())
                out.append(t)
            self._tables_bf16, self._tables_key = out, key
        return self._tables_bf16

    def _last_rows(self, B: int, SP: int, L: int, with_masked: bool, dev) -> torch.Tensor:
        """Token indices (in the batched [targets | pairs | masked targets] order) whose final state is consumed."""
        key = (B, SP, L, with_masked, str(dev))
        cache = self.__dict__.setdefault("_last_rows_cache", {})
        sel = cache.get(key)
        if sel is None:
            parts = [torch.arange(B * L, device=dev), B * L + torch.arange(SP, device=dev) * L]
            if with_masked:
                parts.append((B + SP) * L + torch.arange(B * L, device=dev))
            sel = torch.cat(parts).contiguous()
            if len(cache) > 8:
                cache.clear()
            cache[key] = sel
        return sel

    def mask_nodes(self, node_ids: torch.Tensor, with_positions: bool = False):
        """models.py:131-151, same RNG consumption order (rand, randint, rand).  ``with_positions`` appends the
        (row, position-1) index pairs of the masked slots, so that ``forward`` needs no host sync of its own."""
        device = node_ids.device
        masked_input_ids = node_ids.clone()
        shape = masked_input_ids.size()
        rand = torch.rand(shape[0], shape[1] - 1, device=device)
        mask = (rand < self.random_node_ratio) * (masked_input_ids[:, 1:] != 0)
        masked_input_ids[:, 1:][mask] = torch.randint(2, self.node_size + 2, (int(mask.sum()),), device=device)
        rand = torch.rand(shape[0], shape[1] - 1, device=device)
        mask = (rand < self.mask_node_ratio) * (masked_input_ids[:, 1:] != 0)
        target_idx = masked_input_ids[:, 1:][mask]
        masked_input_ids[:, 1:][mask] = 1  # Fill mask index
        if with_positions:
            return masked_input_ids, mask, target_idx, mask.nonzero(as_tuple=False)
        return masked_input_ids, mask, target_idx

    @torch.no_grad()
    def item_embeddings(self, target_node_inputs: Dict[str, torch.Tensor]) -> torch.Tensor:
        """``self(inputs)[0][:, 0]`` -- the item embedding the downstream recommenders load (trainer.py:153-154,
        base_trainer.py:400-407) -- as a ``[B, H]`` fp32 matrix, with the last encoder layer's post-attention half run
        on position 0 only (rows are independent after the attention core; results are identical row for row)."""
        ids, mask = target_node_inputs["node_ids"], target_node_inputs["attention_mask"]
        if not ids.is_cuda:
            raise PMGTError("PMGT.item_embeddings needs CUDA tensors: pmgt_b200 has no CPU fallback")
        B, L = ids.shape
        fp = self._flat()
        fp.refresh_bf16()
        tables = self.feature_tables_bf16()
        key = ("emb", B, L, str(ids.device))
        cache = self.__dict__.setdefault("_last_rows_cache", {})
        sel = cache.get(key)
        if sel is None:
            if len(cache) > 8:
                cache.clear()
            sel = cache[key] = (torch.arange(B, device=ids.device) * L).contiguous()
        return self.bert.encode(tables, ids.reshape(-1).contiguous(), mask, B, L, refresh=False, last_rows=sel)

    def prepare_inputs(self, target_node_inputs, pair_node_inputs, num_pairs, masked_inputs) -> Dict[str, torch.Tensor]:
        """Everything ``forward`` derives from the batch alone (training with pairs): the concatenated
        [targets | pairs | masked targets] ids / masks, the pair offsets and the compact row numbers of the masked
        positions.  ``forward`` computes it itself when not handed in; the trainer's prefetch builds it on the side
        stream as the fifth element of ``masked_inputs``."""
        t_ids, t_mask = target_node_inputs["node_ids"], target_node_inputs["attention_mask"]
        p_ids, p_mask = pair_node_inputs["node_ids"], pair_node_inputs["attention_mask"]
        B, L = t_ids.shape
        SP = p_ids.shape[0]
        dev = t_ids.device
        m_ids, m_mask = masked_inputs[0], masked_inputs[1]
        m_pos = masked_inputs[3] if len(masked_inputs) > 3 else m_mask.nonzero(as_tuple=False)  # (Mm, 2): row, position-1
        pair_off = torch.zeros(B + 1, dtype=torch.int64, device=dev)
        torch.cumsum(num_pairs.to(dev), 0, out=pair_off[1:])
        return {
            "ids_all": torch.cat([t_ids, p_ids, m_ids], dim=0).reshape(-1),
            "mask_all": torch.cat([t_mask, p_mask, t_mask], dim=0),
            "pair_off": pair_off,
            # compact row numbers of the masked positions (inside the masked-target block of the encoder's output)
            "nfr_rows": B * L + SP + m_pos[:, 0] * L + m_pos[:, 1] + 1,
            "target_ids": masked_inputs[2].contiguous(),
        }

    # ------------------------------------------------------------------
    def forward(
        self,
        target_node_inputs: Dict[str, torch.Tensor],
        pair_node_inputs: Optional[Dict[str, torch.Tensor]] = None,
        num_pairs: torch.LongTensor = None,
        labels: Optional[torch.FloatTensor] = None,
        output_attentions: Optional[bool] = None,
        output_hidden_states: Optional[bool] = None,
        return_dict: Optional[bool] = None,
        masked_inputs=None,
    ):
        """models.py:56-176.  ``output_hidden_states`` / ``output_attentions`` (default: the config's) describe the
        encoding of the TARGET contexts only (the pass whose ``last_hidden_state`` is returned), not the pairs or the
        masked targets: ``hidden_states`` = ``num_hidden_layers + 1`` fp32 ``[B, L, H]`` tensors ending with
        ``last_hidden_state``, ``attentions`` = ``num_hidden_layers`` fp32 ``[B, heads, L, L]`` tensors, with the
        semantics, gradients and memory cost documented at ``PMGTModel.forward``.  With ``return_dict=False`` they are
        appended to the tuple, ``hidden_states`` first, only when requested."""
        if pair_node_inputs is not None:
            assert labels is not None, "labels must be passed, when set pair_node_inputs"
            assert num_pairs is not None, "num_pairs must be passed, when set pair_node_inputs"
        output_attentions, output_hidden_states = resolve_output_flags(self.config, output_attentions,
                                                                       output_hidden_states)
        want = output_attentions or output_hidden_states
        return_dict = return_dict if return_dict is not None else self.config.use_return_dict

        t_ids = target_node_inputs["node_ids"]
        t_mask = target_node_inputs["attention_mask"]
        if not t_ids.is_cuda:
            raise PMGTError("PMGT.forward needs CUDA tensors: pmgt_b200 has no CPU fallback")
        B, L = t_ids.shape
        fp = self._flat()
        fp.refresh_bf16()
        tables = self.feature_tables_bf16()
        # launch plans need the gradients of every step at the same address; the persistent arena is only safe while
        # no gradient of an earlier step is still attached (zero_grad(set_to_none=True) between steps)
        # (a call that asks for per-layer outputs is never planned: it keeps the plans' arena out of it too)
        if (self.bert.use_launch_plans and not want and torch.is_grad_enabled() and all(p.grad is None for p in fp.params)
                and not any(pl.pending_backward for pl in self.bert._plans.values())):
            arena = fp.step_arena()
        else:
            arena = GradArena(fp)

        SP = 0
        nfr_on = False
        prep = None
        if pair_node_inputs is not None:
            SP = pair_node_inputs["node_ids"].shape[0]
            if self.training:
                nfr_on = True
                if masked_inputs is None:
                    masked_inputs = self.mask_nodes(t_ids)
                # data-dependent shapes (nonzero() of the mask) are resolved HERE, before the encoder is enqueued: a sync
                # after the encoder launch would drain the whole launch pipeline
                prep = masked_inputs[4] if len(masked_inputs) > 4 else \
                    self.prepare_inputs(target_node_inputs, pair_node_inputs, num_pairs, masked_inputs)
                ids_flat, mask_all = prep["ids_all"], prep["mask_all"]
            else:
                ids_flat = torch.cat([t_ids, pair_node_inputs["node_ids"]], dim=0).reshape(-1)
                mask_all = torch.cat([t_mask, pair_node_inputs["attention_mask"]], dim=0)
        else:
            ids_flat, mask_all = t_ids.reshape(-1), t_mask
        ids_flat = ids_flat.contiguous()
        R = mask_all.shape[0]
        # the targets are the first B sequences of the batched pass: per-layer outputs are taken for those only
        extra = dict(output_hidden_states=output_hidden_states, output_attentions=output_attentions,
                     output_rows=B) if want else {}
        inner = attentions = None
        if pair_node_inputs is None:
            hidden = self.bert.encode(tables, ids_flat, mask_all, R, L,
                                      arena=arena, refresh=False, **extra)  # (R, L, H) fp32
            if want:
                hidden, inner, attentions = hidden
            H = hidden.shape[-1]
            last_hidden_state = hidden[:B]
        else:
            # Only these token rows of the final hidden state are consumed: every position of the targets (returned as
            # last_hidden_state), position 0 of the pairs (GSR), every position of the masked targets (NFR reads the
            # masked ones).  The encoder prunes its last layer to them and returns the compact [Tc, H] matrix.
            dev = t_ids.device
            sel = self._last_rows(B, SP, L, nfr_on, dev)
            hidden = self.bert.encode(tables, ids_flat, mask_all, R, L,
                                      arena=arena, refresh=False, last_rows=sel, **extra)  # (Tc, H) fp32
            if want:
                hidden, inner, attentions = hidden
            H = hidden.shape[-1]
            last_hidden_state = hidden[:B * L].view(B, L, H)
        hidden_states = inner + (last_hidden_state,) if output_hidden_states else None

        loss = None
        prediction_logits = None
        if pair_node_inputs is not None:
            plan = self.bert._active_plan
            nfr_rows = None
            target_ids = None
            if nfr_on:
                pair_off, nfr_rows, target_ids = prep["pair_off"], prep["nfr_rows"], prep["target_ids"]
            else:
                pair_off = torch.zeros(B + 1, dtype=torch.int64, device=dev)
                torch.cumsum(num_pairs.to(dev), 0, out=pair_off[1:])
            nfr_params = [p for _, p in self.nfr_loss.param_order()] if nfr_on else []
            loss, prediction_logits = _PretrainLossFn.apply(
                self, hidden, B, SP, L, pair_off, labels.to(torch.float32).contiguous(), nfr_rows, target_ids, tables, arena,
                plan.grad_buffer() if plan is not None and hidden.requires_grad else None, *nfr_params)

        if not return_dict:
            return (loss, prediction_logits, last_hidden_state, None) + output_tuple(hidden_states, attentions)
        return PMGTForPreTrainingOutput(loss=loss, prediction_logits=prediction_logits,
                                        last_hidden_state=last_hidden_state, hidden_states=hidden_states,
                                        attentions=attentions)
