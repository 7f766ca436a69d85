"""``PMGTConfig`` with the reference's fields and defaults
(``pmgt/pmgt/configuration_pmgt.py:13-41``).  It does not derive from
transformers' ``PretrainedConfig`` (nothing on the hot path needs it), but it
keeps the attributes the reference's model code reads from that base class:
``output_attentions``, ``output_hidden_states``, ``use_return_dict``,
``chunk_size_feed_forward``.
"""
import copy
import json

# PMGT_MAX_MODALITIES of include/pmgt_b200.h: the embedding fusion kernels take one to four feature modalities
MAX_MODALITIES = 4


class PMGTConfig:
    model_type = "pmgt"

    def __init__(
        self,
        hidden_size=128,
        feat_hidden_sizes=(1536, 768),
        num_hidden_layers=5,
        num_attention_heads=1,
        intermediate_size=128,
        hidden_act="gelu",
        hidden_dropout_prob=0.1,
        attention_probs_dropout_prob=0.1,
        max_position_embeddings=100,
        initializer_range=0.02,
        layer_norm_eps=1e-12,
        beta=0.5,  # diversity promoting attention weight
        **kwargs,
    ):
        self.hidden_size = hidden_size
        self.feat_hidden_sizes = list(feat_hidden_sizes)
        self.num_hidden_layers = num_hidden_layers
        self.num_attention_heads = num_attention_heads
        self.hidden_act = hidden_act
        self.intermediate_size = intermediate_size
        self.hidden_dropout_prob = hidden_dropout_prob
        self.attention_probs_dropout_prob = attention_probs_dropout_prob
        self.max_position_embeddings = max_position_embeddings
        self.initializer_range = initializer_range
        self.layer_norm_eps = layer_norm_eps
        self.beta = beta
        self.output_attentions = kwargs.pop("output_attentions", False)
        self.output_hidden_states = kwargs.pop("output_hidden_states", False)
        self.return_dict = kwargs.pop("return_dict", True)
        self.chunk_size_feed_forward = kwargs.pop("chunk_size_feed_forward", 0)
        for k, v in kwargs.items():
            setattr(self, k, v)
        self._validate()

    def _validate(self):
        if self.hidden_size % self.num_attention_heads != 0:
            # same message as PMGTSelfAttention.__init__ (modeling_pmgt.py:381-387)
            raise ValueError(
                f"The hidden size ({self.hidden_size}) is not a multiple of the number of attention "
                f"heads ({self.num_attention_heads})")
        if self.hidden_act != "gelu":
            raise ValueError("pmgt_b200 implements the reference's only activation, erf-GELU (hidden_act='gelu')")
        if getattr(self, "position_embedding_type", "absolute") != "absolute":
            raise ValueError("only absolute position embeddings are supported (the reference never enables the others)")
        if not 1 <= len(self.feat_hidden_sizes) <= MAX_MODALITIES:
            raise ValueError(f"pmgt_b200 supports 1 to {MAX_MODALITIES} feature modalities; feat_hidden_sizes has "
                             f"{len(self.feat_hidden_sizes)} entries")

    @property
    def use_return_dict(self):
        return self.return_dict

    def to_dict(self):
        return {k: copy.deepcopy(v) for k, v in self.__dict__.items()}

    def to_json_string(self):
        return json.dumps(self.to_dict(), indent=2, sort_keys=True)

    def __repr__(self):
        return f"PMGTConfig {self.to_json_string()}"
