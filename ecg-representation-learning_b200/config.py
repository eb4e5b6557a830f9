"""
`EcgVitConfig` -- same field names, defaults and named sizes as the reference
(/root/reference/ecg_transformer/models/ecg_vit.py:26-92), plus B200-specific knobs that default to the
reference behaviour.
"""
import re

from transformers import PretrainedConfig

# ecg_vit.py:64-91: size -> (hidden_size, num_hidden_layers, num_attention_heads, intermediate_size)
_DEFINED_SIZES = {
    'debug': (64, 4, 4, 256),
    'tiny': (256, 4, 4, 1024),
    'small': (512, 8, 8, 2048),
    'base': (768, 12, 12, 3072),
    'large': (1024, 24, 16, 4096),
}


class EcgVitConfig(PretrainedConfig):
    pattern_model_name = re.compile(r'^(?P<name>\S+)-(?P<size>\S+)$')

    def __init__(self, max_signal_length: int = 2560, patch_size: int = 64, num_channels: int = 12,
                 hidden_size: int = 512, num_hidden_layers: int = 8, num_attention_heads: int = 8,
                 intermediate_size: int = 2048, hidden_dropout_prob: float = 0.1,
                 attention_probs_dropout_prob: float = 0.1, num_class: int = 71,
                 compute_dtype: str = 'bf16', per_lead_tokens: bool = False, residual_dtype: str = 'auto',
                 activation_checkpointing: bool = False, pool: str = 'cls', **kwargs):
        self.max_signal_length = max_signal_length
        self.patch_size = patch_size
        self.num_channels = num_channels
        self.hidden_size = hidden_size
        self.num_hidden_layers = num_hidden_layers
        self.num_attention_heads = num_attention_heads
        self.intermediate_size = intermediate_size
        self.hidden_dropout_prob = hidden_dropout_prob
        self.attention_probs_dropout_prob = attention_probs_dropout_prob
        self.num_class = num_class
        # B200 knob: 'bf16' = tcgen05 contractions with fp32 accumulation/statistics (performance mode);
        #            'fp32' = FFMA contractions (parity mode, <= 1e-5 relative to the reference CPU model)
        self.compute_dtype = compute_dtype
        # False = the reference wrapper (one token per time window, all leads inside it: ecg_vit.py:102-104).
        # True  = BASELINE.json configs[3]: every lead is tokenised on its own (vit_pytorch ViT(image_size=(C, L),
        #         patch_size=(1, P), channels=1)), N = C * L / P + 1 -- not constructible through the reference wrapper
        self.per_lead_tokens = per_lead_tokens
        # storage type of the residual stream (the running sum through the blocks) in bf16 mode: 'bf16', 'fp32', or 'auto'
        # = fp32 for models deeper than 12 layers.  bf16 rounding of the stream random-walks with depth: the 24-layer
        # 'large' model needs fp32 here to stay within 1e-2 of the fp32 reference; up to 12 layers bf16 is inside the bar
        self.residual_dtype = residual_dtype
        # True: keep only every block's input and recompute the block's activations in backward (BASELINE.json configs[4]).
        # Costs one extra block forward per layer (minus the last Linear); 'large' at 512 records per GPU fits 180 GB
        # without it (33.5 GB), so it is off by default
        self.activation_checkpointing = activation_checkpointing
        # classification pooling, vit_pytorch's `pool`: 'cls' = the CLS token's output (the reference's), 'mean' = the
        # mean over all tokens, CLS included (the usual head for fine-tuning MAE-style encoders).  The pre-training
        # models ignore it: their heads read every patch token
        if pool not in ('cls', 'mean'):
            raise ValueError(f"pool must be 'cls' or 'mean', got {pool!r}")
        self.pool = pool
        super().__init__(**kwargs)
        self.size = None

    @classmethod
    def from_defined(cls, model_name):
        """`'ecg-vit-<size>'` with size in debug | tiny | small | base | large (ecg_vit.py:56-92)."""
        m = cls.pattern_model_name.match(model_name)
        if m is None or m.group('name') != 'ecg-vit' or m.group('size') not in _DEFINED_SIZES:
            # the reference validates through its `ca(model_name=...)` arg checker (util/check_args.py:39-41)
            raise ValueError(f'Unexpected model_name: expect one of '
                             f'{["ecg-vit-" + s for s in _DEFINED_SIZES]}, got {model_name!r}')
        conf = cls()
        conf.size = m.group('size')
        (conf.hidden_size, conf.num_hidden_layers, conf.num_attention_heads,
         conf.intermediate_size) = _DEFINED_SIZES[conf.size]
        return conf
