"""TEST INFRASTRUCTURE ONLY -- import shim for the *unmodified* reference.

Makes a checkout of the upstream reference (uoo723/PMGT, pinned to
transformers 4.11.2) importable under transformers 5.x, without editing the
reference tree.  The checkout is not part of this repository: it is used when
``PMGT_REFERENCE_ROOT`` names it or its ``pmgt`` package is importable, by ``tests/golden/make_golden.py`` to
generate the committed golden vectors and by CPU-side tests that cross-check
``oracle/model_ref.py`` / ``oracle/sampler_ref.py`` against the real thing.

Nothing under ``pmgt_b200/`` may import this module.
"""
import os
import sys

def _find_root() -> str:
    """``PMGT_REFERENCE_ROOT``, else the checkout whose upstream ``pmgt`` package is importable (installed, or its root
    on ``sys.path``); "" when there is neither."""
    root = os.environ.get("PMGT_REFERENCE_ROOT")
    if root:
        return root
    import importlib.util

    try:
        spec = importlib.util.find_spec("pmgt")
    except (ImportError, ValueError):
        return ""
    for loc in (spec.submodule_search_locations or []) if spec else []:
        if os.path.isdir(os.path.join(loc, "pmgt")):
            return os.path.dirname(os.path.abspath(loc))
    return ""


REFERENCE_ROOT = _find_root()
STAGED_ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")   # oracle/build.py::build_ref()


def available() -> bool:
    """The reference tree itself (``_find_root``): what the parity tests and the golden generator need."""
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, "pmgt", "pmgt"))


def staged_available() -> bool:
    """The unmodified hot-path modules staged under oracle/_ref/ (bench CPU arm only)."""
    return os.path.isdir(os.path.join(STAGED_ROOT, "pmgt", "pmgt"))


def load_any():
    """The reference tree when present, else the staged copy."""
    global REFERENCE_ROOT
    if not available() and staged_available():
        REFERENCE_ROOT = STAGED_ROOT
        return load(_root_ok=True)
    return load()


_loaded = None


def load(_root_ok: bool = False):
    """Return a namespace with the reference's hot-path symbols."""
    global _loaded
    if _loaded is not None:
        return _loaded
    if not _root_ok and not available():
        raise RuntimeError(f"no reference tree at {REFERENCE_ROOT!r}: set PMGT_REFERENCE_ROOT to a checkout of "
                           "uoo723/PMGT")
    sys.dont_write_bytecode = True  # the reference tree is read-only
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)

    import transformers.modeling_utils as mu
    import transformers.pytorch_utils as pu

    # names the reference imports from transformers.modeling_utils (modeling_pmgt.py:18-23)
    mu.apply_chunking_to_forward = pu.apply_chunking_to_forward
    mu.prune_linear_layer = pu.prune_linear_layer

    def _no_prune(*a, **k):  # only reachable through prune_heads(), never called
        raise NotImplementedError

    mu.find_pruneable_heads_and_indices = _no_prune

    import pmgt.pmgt.modeling_pmgt as mp

    # transformers 4.11.2 semantics of the three PreTrainedModel helpers the
    # reference calls (modeling_pmgt.py:74,118-120,127)
    def _ext_mask(self, attention_mask, input_shape, device=None):
        assert attention_mask.dim() == 2
        return (1.0 - attention_mask[:, None, None, :].to(dtype=self.dtype)) * -10000.0

    def _head_mask(self, head_mask, num_hidden_layers, is_attention_chunked=False):
        assert head_mask is None
        return [None] * num_hidden_layers

    def _init_weights_4x(self):
        self.apply(self._init_weights)

    mp.PMGTPretrainedModel.get_extended_attention_mask = _ext_mask
    mp.PMGTPretrainedModel.get_head_mask = _head_mask
    mp.PMGTPretrainedModel.init_weights = _init_weights_4x

    from types import SimpleNamespace

    import pmgt.pmgt.datasets as ds
    from pmgt.optimizers import DenseSparseAdamW
    from pmgt.pmgt.configuration_pmgt import PMGTConfig
    from pmgt.pmgt.models import PMGT

    _loaded = SimpleNamespace(
        modeling=mp,
        datasets=ds,
        PMGT=PMGT,
        PMGTConfig=PMGTConfig,
        PMGTModel=mp.PMGTModel,
        PMGTDataset=ds.PMGTDataset,
        pmgt_collate_fn=ds.pmgt_collate_fn,
        get_input_tensor=ds.get_input_tensor,
        sample_context_neigh=ds._sample_context_neigh,
        DenseSparseAdamW=DenseSparseAdamW,
    )
    return _loaded
