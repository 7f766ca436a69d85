"""Host-side mirror of ``pmgt/pmgt/trainer.py`` (+ the parts of
``pmgt/base_trainer.py`` the PMGT path uses), re-hosted on a plain loop.

The reference drives everything through pytorch-lightning / mlflow / optuna
(absent here and out of scope); this module keeps the reference's entry
functions -- ``check_args``, ``init_run``, ``init_dataloader``, ``init_model``,
``train``, ``test``, ``inference`` -- with the same ``args`` fields
(train.py:18-70,223-288), and ``PMGTTrainerModel`` with the same step methods.

What is different by design:
 * batches come from ``PMGTDataset.sample_batch`` (GPU sampler) instead of
   DataLoader worker processes; a "dataloader" here is an index-batch iterator;
 * data parallelism is explicit: one process per GPU, targets sharded by rank,
   ONE NCCL allreduce of the flat gradient buffer per step (the reference gets
   bucketed DDP implicitly from Lightning, base_trainer.py:309-322);
 * optimizer = fused ``DenseSparseAdamW`` over the flat parameter buffer with
   the reference's two parameter groups (base_trainer.py:35-59) and optional
   ``clip_grad_norm_`` (``gradient_max_norm``, base_trainer.py:314).
"""
import os
import pickle
import time
from typing import Dict, Iterator, List, Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist

from . import ops
from .configuration_pmgt import PMGTConfig
from .datasets import PMGTDataset
from .graph import ItemGraph
from .models import PMGT
from .optimizers import DenseSparseAdamW
from .utils import set_seed


class AttrDict(dict):
    """Minimal ``attrdict.AttrDict``: attribute access over a dict; missing keys read as None."""

    def __getattr__(self, k):
        return self.get(k)

    def __setattr__(self, k, v):
        self[k] = v


DEFAULTS = dict(  # train.py:18-70 (shared flags) and 223-288 (PMGT flags)
    mode="train", seed=0, model_name="PMGT", dataset_name="VG", data_dir="./data", log_dir="./logs",
    num_epochs=20, train_batch_size=256, test_batch_size=256, no_cuda=False, num_workers=8, lr=1e-3, decay=1e-2,
    optim="adamw", early=10, early_criterion="loss", valid_size=0.2, mp_enabled=False, gradient_max_norm=None,
    accumulation_step=1, scheduler_type=None, run_id=None, inference_result_path=None,
    max_ctx_neigh=5, hop_sampling_sizes=[16, 8, 4], max_total_samples=10, min_neg_samples=5,
    hidden_size=128, intermediate_size=128, num_hidden_layers=5, num_attention_heads=1, beta=0.5,
    random_node_ratio=0.2 * 0.1, mask_node_ratio=0.2 * 0.8, synthetic=None,
)


def make_args(**over) -> AttrDict:
    a = AttrDict(DEFAULTS)
    a.update(over)
    return a


# ---------------------------------------------------------------------------
# distributed helpers
# ---------------------------------------------------------------------------
def world() -> Tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_indices(perm: np.ndarray, step: int, batch_per_rank: int, rank: int, world_size: int) -> np.ndarray:
    """Targets of ``rank`` at ``step``: perm[step*B*W + rank*B : ... + B]  (SURVEY section 8e)."""
    lo = step * batch_per_rank * world_size + rank * batch_per_rank
    return perm[lo: lo + batch_per_rank]


def epoch_permutation(n: int, seed: int, epoch: int) -> np.ndarray:
    """Same permutation on every rank, derived from (seed, epoch)."""
    return np.random.default_rng([int(seed), int(epoch)]).permutation(n)


# ---------------------------------------------------------------------------
# reference entry points
# ---------------------------------------------------------------------------
def check_args(args: AttrDict) -> None:
    """trainer.py:213-218 / base_trainer.py check_args."""
    if args.early_criterion not in ["loss", "auc"]:
        raise ValueError(f"early_criterion must be one of ['loss', 'auc'], got {args.early_criterion}")
    if args.model_name not in ["PMGT"]:
        raise ValueError(f"model_name must be one of ['PMGT'], got {args.model_name}")
    if args.dataset_name not in ["VG", "TG"] and not args.synthetic:
        raise ValueError(f"dataset_name must be one of ['VG', 'TG'], got {args.dataset_name}")
    if args.optim != "adamw":
        raise ValueError(f"Optimizer {args.optim} is not supported")
    if args.scheduler_type is not None:
        raise ValueError("LR schedulers are not wired in the reference's PMGT path (base_trainer.py:71-90 recurses)")
    if args.mp_enabled:
        # the reference's --mp-enabled is fp16 autocast + GradScaler (base_trainer.py:312); this implementation always
        # computes in bf16 with fp32 accumulation / statistics, there is no fp16 path to switch on
        raise ValueError("mp_enabled (fp16 autocast) is not supported: pmgt_b200 always runs bf16 tensor-core math with "
                         "fp32 accumulation")
    if args.accumulation_step is not None and int(args.accumulation_step) < 1:
        raise ValueError("accumulation_step must be >= 1")
    # init_model builds the config with the default position table: a context is max_ctx_neigh + 1 tokens
    max_pos = PMGTConfig().max_position_embeddings
    if int(args.max_ctx_neigh) + 1 > max_pos:
        raise ValueError(f"max_ctx_neigh must be <= {max_pos - 1}: a context of max_ctx_neigh + 1 tokens needs that "
                         f"many rows of the {max_pos}-row position table")


def init_run(args: AttrDict) -> None:
    """base_trainer.py:194-200."""
    set_seed(args.seed)
    if not torch.cuda.is_available() or args.no_cuda:
        raise RuntimeError("pmgt_b200 trains on CUDA devices only (no CPU fallback)")
    args.device = torch.device("cuda", torch.cuda.current_device())
    args.num_gpus = world()[1]


def _load_graph_and_features(args: AttrDict):
    """trainer.py:30-41,112-116; ``args.synthetic`` substitutes seeded synthetic inputs."""
    if args.synthetic:
        from . import synthetic

        name = args.synthetic
        big = isinstance(name, str) and name in synthetic.SHAPES and synthetic.SHAPES[name][0] > 200_000
        # large graphs are ingested on the device (edge list -> CSR + CDF + lookup tables by kernels)
        graph = synthetic.make_item_graph(name, device=args.device if (big and args.device is not None) else None)
        seed = synthetic.SHAPES[name][3] if isinstance(name, str) and name in synthetic.SHAPES else 1234
        if graph.num_nodes > 200_000:
            feats = synthetic.make_features_device(graph.num_nodes, seed=seed, device=args.device)
        else:
            feats = synthetic.make_features(graph.num_nodes, seed=seed)
        return graph, feats
    import joblib
    import networkx as nx

    data_dir = os.path.join(args.data_dir, args.dataset_name)
    node_encoder = joblib.load(os.path.join(data_dir, "node_encoder"))
    with open(os.path.join(data_dir, "graph.gpickle"), "rb") as f:  # nx.read_gpickle (networkx 2.6) == pickle.load
        g = pickle.load(f)
    # idx 0 is <pad>, idx 1 is <mask>
    mapping = {label: i + 2 for i, label in enumerate(node_encoder.classes_)}
    g = nx.relabel_nodes(g, mapping)
    feats = [np.load(os.path.join(data_dir, "visual_init_emb.npy")), np.load(os.path.join(data_dir, "textual_init_emb.npy"))]
    return ItemGraph.from_networkx(g), feats


def _split(n_nodes: int, valid_size: float, seed: int):
    """sklearn.model_selection.train_test_split(np.arange(2, N+2), test_size, random_state) (trainer.py:45-52)."""
    from sklearn.model_selection import train_test_split

    return train_test_split(np.arange(start=2, stop=n_nodes + 2), test_size=valid_size, random_state=seed)


def init_dataloader(args: AttrDict) -> None:
    if args.graph is None:
        args.graph, args.feat_init_emb = _load_graph_and_features(args)
    train_nodes, valid_nodes = _split(len(args.graph), args.valid_size, args.seed)
    args.train_dataset = PMGTDataset(args.graph, train_nodes, args.max_ctx_neigh, args.hop_sampling_sizes,
                                     args.max_total_samples, args.min_neg_samples, seed=args.seed)
    args.valid_dataset = PMGTDataset(args.graph, valid_nodes, args.max_ctx_neigh, args.hop_sampling_sizes,
                                     is_training=False, seed=args.seed + 1)
    args.test_dataset = args.valid_dataset  # trainer.py:71 returns the validation set twice


def init_model(args: AttrDict) -> None:
    if args.graph is None:
        args.graph, args.feat_init_emb = _load_graph_and_features(args)
    feats = args.feat_init_emb
    config = PMGTConfig(hidden_size=args.hidden_size, feat_hidden_sizes=[int(f.shape[-1]) for f in feats],
                        intermediate_size=args.intermediate_size, num_hidden_layers=args.num_hidden_layers,
                        num_attention_heads=args.num_attention_heads, beta=args.beta,
                        **({"hidden_dropout_prob": args.hidden_dropout_prob} if args.hidden_dropout_prob is not None else {}),
                        **({"attention_probs_dropout_prob": args.attention_probs_dropout_prob}
                           if args.attention_probs_dropout_prob is not None else {}))
    model = PMGT(node_size=len(args.graph), random_node_ratio=args.random_node_ratio,
                 mask_node_ratio=args.mask_node_ratio, config=config, feat_init_emb=feats)
    args.model = model.to(args.device)


def get_optimizer(args: AttrDict) -> DenseSparseAdamW:
    """base_trainer.py:35-68: no weight decay for names containing "bias" or "LayerNorm.weight"."""
    no_decay = ["bias", "LayerNorm.weight"]
    named = [(n, p) for n, p in args.model.named_parameters() if p.requires_grad]
    groups = [
        {"params": [p for n, p in named if not any(nd in n for nd in no_decay)], "weight_decay": args.decay, "lr": args.lr},
        {"params": [p for n, p in named if any(nd in n for nd in no_decay)], "weight_decay": 0.0, "lr": args.lr},
    ]
    return DenseSparseAdamW(groups)


class PMGTTrainerModel:
    """trainer.py:150-206 without Lightning: holds the net + optimizer and implements the step methods."""

    def __init__(self, args: AttrDict):
        self.args = args
        self.net: PMGT = args.model
        self.optimizer = get_optimizer(args)
        # PMGT_SYMM_REDUCE=1: data parallel on one NVSwitch domain without NCCL in the step -- gradients live in symmetric
        # memory and are summed in place by peer_reduce (csrc/peer_reduce.cu).  Off by default: measured on 4 GPUs it is
        # 1.5 % slower (6.47 vs 6.37 ms/step) than the NCCL all-reduce started from inside the backward pass, whose
        # transfer hides behind the embedding backward while the peer reduction's two barriers + kernel are exposed.
        if (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1 and dist.get_world_size() <= 8
                and dist.get_backend() == "nccl" and os.environ.get("PMGT_SYMM_REDUCE", "0") == "1"):
            self.net._flat().symm_group = dist.group.WORLD
        self.global_step = 0
        self._sumsq = None
        self._side = None        # high-priority stream the next step's batch is prepared on
        self._prefetched = None  # (dataset, indices, epoch, batch, masked, ready-event)
        self._loss_pin = None    # pinned host scalar the step's loss is copied into right after the forward pass
        self._loss_event = None
        self._work = None        # in-flight allreduce of the encoder-layer gradients (started inside the backward pass)
        self._work_buf = None
        self.max_run_ahead = 1   # the host enqueues at most this many steps beyond the one whose forward pass is running
        self._micro = 0          # micro-batches accumulated since the last optimizer step
        self.epoch = 0           # next epoch to train (saved in checkpoints; Lightning's current_epoch)
        self.best, self.bad_epochs, self.best_path = None, 0, None

    # -- inference: net(x)[0][:, 0] (trainer.py:153-154)
    def forward(self, x):
        return self.net(x)[0][:, 0].cpu().numpy()

    __call__ = forward

    def training_step(self, batch, batch_idx: int = 0) -> torch.Tensor:
        return self.net(*batch)[0]

    def _validation_and_test_step(self, batch):
        outputs = self.net(*batch)
        loss, logits, labels = outputs[0], outputs[1], batch[-1]
        return loss, logits.sigmoid().cpu().numpy(), labels.cpu().numpy()

    # -- the batch of a LATER step, prepared while the current step is still running on the device
    def prefetch(self, dataset: PMGTDataset, indices, epoch: int) -> None:
        """Sample the contexts of ``indices`` and draw their NFR corruption on a side stream.

        The corruption (models.py:131-151) has data-dependent shapes, i.e. host syncs; issued here they wait for the
        small side stream only, while the main stream still holds the queued kernels of the current step.  The next
        ``train_on_indices`` call with the same ``(dataset, indices, epoch)`` picks the result up; anything else
        discards it.  The torch generator is consumed once per step in the reference's order either way.
        """
        dev = self.args.device
        if self._side is None:
            self._side = torch.cuda.Stream(device=dev, priority=int(os.environ.get("PMGT_SIDE_PRIORITY", "-1")))
        # No wait on the main stream's tail (that would serialise us behind the very step we want to overlap): host indices
        # are copied on the side stream; device-resident indices must already be complete.  The side stream does wait for
        # the END OF THE RUNNING STEP'S FORWARD PASS (its loss event): the encoder's persistent kernels leave a sampler CTA
        # no room, so sampling beside them only displaces them, while the loss kernels and the head of the backward pass
        # that follow (~0.35 ms of small grids) leave most SMs free (PMGT_PREFETCH_AFTER_FWD=0: start immediately).
        if self._loss_event is not None and os.environ.get("PMGT_PREFETCH_AFTER_FWD", "1") != "0":
            self._side.wait_event(self._loss_event)
        with torch.cuda.stream(self._side):
            idx = indices if isinstance(indices, torch.Tensor) else torch.as_tensor(np.asarray(indices))
            idx = idx.to(dev, non_blocking=True)
            batch = dataset.sample_batch(idx, epoch=epoch)
            masked = None
            if dataset.is_training:
                masked = self.net.mask_nodes(batch[0]["node_ids"], with_positions=True)
                # the concatenated [targets | pairs | masked targets] inputs and the loss indices depend on the batch
                # only: built here, they cost the main stream nothing
                masked = masked + (self.net.prepare_inputs(batch[0], batch[1], batch[2], masked),)
            ready = torch.cuda.Event()
            ready.record(self._side)
        self._prefetched = (dataset, indices, epoch, batch, masked, ready)

    def _take_prefetched(self, dataset, indices, epoch):
        pf, self._prefetched = self._prefetched, None
        if pf is None or pf[0] is not dataset or pf[1] is not indices or pf[2] != epoch:
            return None
        _, _, _, batch, masked, ready = pf
        main = torch.cuda.current_stream(self.args.device)
        main.wait_event(ready)
        tensors = [batch[0]["node_ids"], batch[0]["attention_mask"], batch[1]["node_ids"], batch[1]["attention_mask"],
                   batch[2], batch[3]]
        for m in (masked or ()):
            tensors.extend(m.values() if isinstance(m, dict) else [m])
        for t in tensors:
            if isinstance(t, torch.Tensor):
                t.record_stream(main)  # allocated on the side stream, consumed on the main one
        return batch, masked

    # -- one optimisation step on a sampled batch (sample -> fwd -> bwd -> allreduce -> AdamW)
    def train_on_indices(self, dataset: PMGTDataset, indices, epoch: int) -> torch.Tensor:
        """One micro-batch: forward + backward, and -- every ``accumulation_step`` calls (pl.Trainer's
        ``accumulate_grad_batches``, base_trainer.py:315) -- gradient allreduce, clipping and the AdamW step."""
        args = self.args
        if not self.net.training:
            self.net.train()
        accum = max(1, int(args.accumulation_step or 1))
        # Bound the host's run-ahead: wait until the PREVIOUS step's forward pass has finished (its loss event) before
        # enqueueing this step.  An unthrottled loop queues several steps of side-stream sampling next to the main
        # stream's kernels, which measurably slows both (round 1: the loop that read the loss every step was faster).
        if self.max_run_ahead and self._loss_event is not None:
            self._loss_event.synchronize()
        # fixed-shape steps: record the encoder's launch list once, then replay.  Launch plans write the gradients of
        # every pass into the same arena, so with gradient accumulation (which must ADD passes) they stay off.
        self.net.bert.use_launch_plans = accum == 1
        pf = self._take_prefetched(dataset, indices, epoch)
        if self._micro == 0:
            self.optimizer.zero_grad(set_to_none=True)
        if pf is not None:
            batch, masked = pf
            loss = self.net(*batch, masked_inputs=masked)[0]
        else:
            batch = dataset.sample_batch(indices, epoch=epoch)
            loss = self.training_step(batch)
        # the loss is final once the forward pass is: copy it out NOW (pinned buffer + event), so that reading it on the
        # host (`last_loss`) waits for the forward kernels only, not for the backward pass and the optimizer behind them
        if self._loss_pin is None:
            self._loss_pin = torch.empty((), dtype=torch.float32).pin_memory()
            self._loss_event = torch.cuda.Event()
        self._loss_pin.copy_(loss.detach(), non_blocking=True)
        self._loss_event.record()
        rank, ws = world()
        fp = self.net._flat()
        arena = getattr(fp, "_step_arena", None)
        symm = arena.symm if (arena is not None and ws > 1 and accum == 1) else None
        # NCCL path: the encoder-layer gradients are reduced from inside the backward pass; symmetric-memory path: one
        # in-place peer reduction after it (below)
        fp.after_layers_hook = self._reduce_layers_early if (ws > 1 and symm is None and self._micro + 1 >= accum) else None
        self._work = None
        loss.backward()
        self._micro += 1
        if self._micro < accum:
            return loss.detach()
        self._micro = 0
        scale = 1.0 / accum
        fv = self.optimizer.flat_views()
        if ws > 1:
            if fv is None or fv[1] is None:
                raise RuntimeError("data-parallel training needs the flat gradient buffer")
            if symm is not None and fv[1].data_ptr() == arena.buf.data_ptr():
                # every rank's gradient is complete -> each rank sums its slice over all copies through peer pointers
                # and writes it back to all of them -> every slice is in place (two device-side barriers, one kernel)
                symm.barrier(channel=0)
                ops.peer_reduce(symm.buffer_ptrs, rank, fv[1].numel())
                symm.barrier(channel=1)
            elif self._work is not None:
                # the encoder-layer (+ NFR) part of the flat gradient has been in flight since the middle of the backward
                # pass; only the embedding block -- whose backward ran meanwhile -- is reduced here
                if fv[1].data_ptr() != self._work_buf.data_ptr():
                    raise RuntimeError("the gradient that was reduced early is not the buffer the optimizer steps with")
                self._work.wait()
                dist.all_reduce(fv[1][: self._layers_lo(fp)])
                self._work = None
            else:
                dist.all_reduce(fv[1])  # ONE allreduce of the flat gradient (sum); mean folded into the step
            scale = scale / ws
        scale_dev = None
        if args.gradient_max_norm:
            # torch.nn.utils.clip_grad_norm_: coef = min(1, max_norm / (norm + 1e-6)), on the averaged gradient; one small
            # kernel folds it with the gradient scale and resets the accumulator for the next step
            if self._sumsq is None:
                self._sumsq = torch.zeros(1, dtype=torch.float32, device=loss.device)
                self._coef = torch.empty(1, dtype=torch.float32, device=loss.device)
            if fv is not None and fv[1] is not None:
                ops.sumsq(fv[1], self._sumsq)
            else:
                for p in self.net.parameters():
                    if p.grad is not None:
                        ops.sumsq(p.grad.contiguous().view(-1), self._sumsq)
            ops.clip_coef(self._sumsq, scale, float(args.gradient_max_norm), self._coef)
            scale_dev = self._coef
        # step with exactly the buffer that was reduced / measured above (it is a temporary when the gradients are not
        # zero-copy views of the arena: a second flat_views() call would rebuild it from the un-reduced p.grad)
        self.optimizer.step(grad_scale=scale, grad_scale_dev=scale_dev,
                            flat_grad=fv[1] if fv is not None else None)
        self.global_step += 1
        return loss.detach()

    # -- data parallel: the flat gradient is reduced in two pieces, the big one overlapped with the embedding backward
    @staticmethod
    def _layers_lo(fp) -> int:
        """Offset in the flat parameter order where the encoder layers start (everything before it is the embedding
        block, whose gradients are produced LAST by the backward pass)."""
        for n in fp.names:
            if ".encoder.layer." in n or n.startswith("nfr_loss."):
                return fp.offsets[n]
        return fp.total

    def _reduce_layers_early(self, arena) -> None:
        """Called from inside the encoder backward (ops.host_hook) when all gradients except the embedding block's are
        final.  Only for the persistent step arena, whose buffer is what the optimizer steps with (zero-copy)."""
        if not getattr(arena, "persistent", False):
            return
        buf = arena.get()
        lo = self._layers_lo(arena.fp)
        if lo >= buf.numel():
            return
        self._work_buf = buf
        self._work = dist.all_reduce(buf[lo:], async_op=True)

    def last_loss(self) -> float:
        """Host value of the most recent ``train_on_indices`` loss (device -> pinned-host copy issued right after the
        forward pass; this call waits for that copy only).  ``float(loss)`` on the returned tensor gives the same number
        but drains the whole stream first."""
        if self._loss_event is None:
            raise RuntimeError("last_loss() before the first train_on_indices()")
        self._loss_event.synchronize()
        return float(self._loss_pin)

    @torch.no_grad()
    def evaluate(self, dataset: PMGTDataset, batch_size: int) -> Dict[str, float]:
        """validation/test epoch (trainer.py:162-206): mean loss + ROC-AUC of sigmoid(logits)."""
        from sklearn.metrics import roc_auc_score

        self.net.eval()
        rank, ws = world()
        preds, labels, losses = [], [], []
        idx_all = np.arange(len(dataset))[rank::ws]
        for lo in range(0, len(idx_all), batch_size):
            loss, p, l = self._validation_and_test_step(dataset.sample_batch(idx_all[lo: lo + batch_size], epoch=0))
            preds.append(p)
            labels.append(l)
            losses.append(float(loss))
        preds = np.concatenate(preds) if preds else np.zeros(0, dtype=np.float32)   # a rank's shard may be empty
        labels = np.concatenate(labels) if labels else np.zeros(0, dtype=np.float32)
        if ws > 1:
            gathered = [None] * ws
            dist.all_gather_object(gathered, (preds, labels, losses))
            preds = np.concatenate([g[0] for g in gathered])
            labels = np.concatenate([g[1] for g in gathered])
            losses = sum((g[2] for g in gathered), [])
        return {"loss": float(np.mean(losses)), "auc": float(roc_auc_score(labels, preds))}

    def state_dict(self):
        return {"state_dict": {"net." + k: v for k, v in self.net.state_dict().items()},  # Lightning's "net." prefix
                "optimizer": self.optimizer.state_dict(), "global_step": self.global_step, "epoch": self.epoch,
                "early_stopping": {"best": self.best, "bad_epochs": self.bad_epochs, "best_path": self.best_path}}

    def load_state_dict(self, ckpt, weights_only: bool = False):
        """Restore a checkpoint.  Like Lightning's ``fit(ckpt_path=...)`` (base_trainer.py:324-332) this brings back the
        weights, the optimizer state (AdamW moments and step count), the epoch counter and the early-stopping
        bookkeeping; ``weights_only`` restores just the weights (evaluation / inference of a best checkpoint)."""
        self.net.load_state_dict({k[len("net."):]: v for k, v in ckpt["state_dict"].items()})
        self.net._tables_bf16 = None
        if weights_only:
            return
        self.global_step = ckpt.get("global_step", 0)
        self.epoch = ckpt.get("epoch", 0)
        es = ckpt.get("early_stopping") or {}
        self.best, self.bad_epochs, self.best_path = es.get("best"), es.get("bad_epochs", 0), es.get("best_path")
        if ckpt.get("optimizer") is not None:
            self.optimizer.load_state_dict(ckpt["optimizer"])


def _ckpt_dir(args: AttrDict) -> str:
    d = os.path.join(args.log_dir, args.run_id or "pmgt_b200_run", "checkpoints")
    os.makedirs(d, exist_ok=True)
    return d


def _barrier():
    if dist.is_available() and dist.is_initialized():
        dist.barrier()


def epoch_batches(n: int, batch: int, rank: int, ws: int, perm: np.ndarray) -> List[np.ndarray]:
    """Index batches of ``rank`` for one epoch: every full global batch of ``batch * ws`` targets, then the tail
    (the reference's DataLoader keeps the partial last batch: shuffle=True, drop_last=False, trainer.py:90-103), split
    evenly over the ranks; ranks whose tail share would be empty re-use the first tail targets so that every rank runs
    the same number of steps (the allreduce is collective)."""
    per = batch * ws
    full = n // per
    out = [shard_indices(perm, step, batch, rank, ws) for step in range(full)]
    tail = perm[full * per:]
    if len(tail):
        share = -(-len(tail) // ws)
        mine = tail[rank * share: (rank + 1) * share]
        if len(mine) == 0:
            mine = tail[:1]
        out.append(mine)
    return out


def train(args: AttrDict, is_hptuning: bool = False, trial=None, enable_trial_pruning: bool = False):
    """base_trainer.py:266-341: fit with early stopping + last/best checkpoints.  Returns (best_score, trainer)."""
    tm = PMGTTrainerModel(args)
    rank, ws = world()
    ds: PMGTDataset = args.train_dataset
    B = args.train_batch_size
    monitor = "loss" if args.early_criterion == "loss" else "auc"
    ckpt_dir = _ckpt_dir(args)
    last_path = os.path.join(ckpt_dir, "last.ckpt")
    if args.run_id is not None and os.path.exists(last_path):  # resume (base_trainer.py:324-332)
        tm.load_state_dict(torch.load(last_path, map_location=args.device, weights_only=False))
    args.history = []
    for epoch in range(tm.epoch, args.num_epochs):
        if args.early and tm.bad_epochs >= args.early:
            break
        perm = epoch_permutation(len(ds), args.seed, epoch)
        t0 = time.time()
        running = []
        shards = epoch_batches(len(ds), B, rank, ws, perm)
        for step in range(len(shards)):
            loss = tm.train_on_indices(ds, shards[step], epoch)
            if step + 1 < len(shards):
                tm.prefetch(ds, shards[step + 1], epoch)  # sampling + corruption of the next batch overlap this step
            running.append(loss)
        train_loss = float(torch.stack(running).mean())
        val = tm.evaluate(args.valid_dataset, args.test_batch_size)
        args.history.append({"epoch": epoch, "loss/train": train_loss, "loss/val": val["loss"], "val/auc": val["auc"],
                             "sec": time.time() - t0})
        score = val[monitor]
        improved = tm.best is None or (score < tm.best if monitor == "loss" else score > tm.best)
        tm.epoch = epoch + 1
        if improved:
            tm.best, tm.bad_epochs = score, 0
            tm.best_path = os.path.join(ckpt_dir, f"epoch={epoch}.ckpt")
            if rank == 0:
                torch.save(tm.state_dict(), tm.best_path)
        else:
            tm.bad_epochs += 1
        if rank == 0:
            torch.save(tm.state_dict(), last_path)
        _barrier()  # no rank reads a checkpoint that rank 0 is still writing
    args.best_model_path = tm.best_path
    return tm.best, tm


def _load_best(tm: "PMGTTrainerModel", args: AttrDict) -> None:
    """Weights of the best checkpoint (base_trainer.py get_ckpt_path): loud when the path is set but the file is not there."""
    if not args.best_model_path:
        return
    _barrier()
    if not os.path.exists(args.best_model_path):
        raise FileNotFoundError(f"best_model_path is set but missing: {args.best_model_path}")
    tm.load_state_dict(torch.load(args.best_model_path, map_location=args.device, weights_only=False), weights_only=True)


def test(args: AttrDict, trainer: Optional[PMGTTrainerModel] = None, is_hptuning: bool = False) -> Dict[str, float]:
    """base_trainer.py test(): AUC on the test split with the best checkpoint."""
    tm = trainer or PMGTTrainerModel(args)
    _load_best(tm, args)
    res = tm.evaluate(args.test_dataset, args.test_batch_size)
    return {"test/auc": res["auc"]}


@torch.no_grad()
def inference(args: AttrDict) -> np.ndarray:
    """trainer.py:259-275 + base_trainer.py:382-409: (N, H) float32 embeddings, row i <-> node id i+2,
    node range sharded contiguously across ranks; rank 0 saves ``inference_result_path`` (.npy)."""
    tm = PMGTTrainerModel(args)
    _load_best(tm, args)
    tm.net.eval()
    ds = PMGTDataset(args.graph, max_ctx_neigh=args.max_ctx_neigh, hop_sampling_sizes=args.hop_sampling_sizes,
                     is_training=False, is_inference=True, seed=args.seed)
    rank, ws = world()
    n = len(ds)
    lo, hi = n * rank // ws, n * (rank + 1) // ws
    # position-0 states only (the last layer is pruned to them), written batch by batch into PINNED host memory with
    # asynchronous copies that overlap the next batch's sampling and encoding; one synchronisation at the end
    out = torch.empty((hi - lo, args.hidden_size), dtype=torch.float32).pin_memory()
    bs = args.test_batch_size
    order = torch.arange(lo, hi, device=args.device)
    tm.net.bert.use_launch_plans = True   # fixed-shape forward passes: record the launch list once, replay it
    for s in range(lo, hi, bs):
        e = min(s + bs, hi)
        emb = tm.net.item_embeddings(ds.sample_batch(order[s - lo: e - lo]))
        # (a planned pass's output aliases a plan-owned buffer that the next pass overwrites: the copy is enqueued on
        # the same stream before that pass, so it reads the right data)
        out[s - lo: e - lo].copy_(emb, non_blocking=True)
    torch.cuda.synchronize(args.device)
    res = out.numpy()
    if ws > 1:
        parts = [None] * ws
        dist.all_gather_object(parts, res)
        res = np.concatenate(parts)
    if args.inference_result_path and rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(args.inference_result_path)), exist_ok=True)
        np.save(args.inference_result_path, res)
    return res


def train_model(**over):
    """train.py:298-344 dispatcher for ``train-pmgt``."""
    args = make_args(**over)
    check_args(args)
    init_run(args)
    init_dataloader(args)
    init_model(args)
    if args.mode == "inference":
        return inference(args)
    best, tm = train(args)
    res = test(args, tm)
    return best, res
