"""
`EcgVit` -- drop-in for the reference nn.Module (/root/reference/ecg_transformer/models/ecg_vit.py:95-149):
same constructor, `forward(sample_values[B,12,L], labels=None) -> ModelOutput(loss, logits)`, attributes
(`vit`, `config`, `meta`, `meta_str`, `loss_reduction`, `loss_weight`, `to_str()`) and `state_dict()` keys of the
reference over `vit-pytorch==0.33.2`, but every arithmetic op runs in hand-written sm_100a kernels.

The module tree below only HOLDS parameters (it mirrors vit_pytorch's Sequential/ModuleList indices so the keys
match); it has no eager PyTorch forward.  All parameters are views into one flat fp32 buffer so that gradient
clipping, AdamW and the DDP all-reduce are single passes over contiguous memory.
"""
from collections import namedtuple, OrderedDict

import weakref

import torch
from torch import nn

from . import _lib
from .config import EcgVitConfig, check_drop_path_rate
from .engine import StepEngine, MaskedPatchEngine, MaskedAutoencoderEngine

ModelOutput = namedtuple('ModelOutput', ['loss', 'logits'])  # reference: util/models.py:3
MaskedPatchOutput = namedtuple('MaskedPatchOutput', ['loss', 'reconstruction', 'bool_masked_pos'])

_ALIGN = 64  # elements: every tensor starts on a 256-byte boundary of the flat buffers

# The trainable part of a model, derived from the `requires_grad` flags (`EcgVit.trainable_span`):
#   lowest        lowest forward position holding a trainable parameter: -1 = patch embedding / pos / cls / mask token,
#                 0 .. depth - 1 = encoder block, depth = everything above the encoder; None when nothing is trainable
#   lo            flat offset of the first trainable tensor (the flat length when nothing is trainable)
#   frozen_inside whether a frozen tensor lies in [lo, flat length)
#   frozen        flat-buffer keys of the frozen tensors
#   key           the flags themselves, in `named_parameters()` order (cache and graph key)
TrainableSpan = namedtuple('TrainableSpan', ['lowest', 'lo', 'frozen_inside', 'frozen', 'key'])


def _forward_position(key, depth):
    """forward position of the flat-buffer key `key` (see TrainableSpan.lowest)"""
    if key in ('pos', 'cls', 'mask') or key.startswith('embed.'):
        return -1
    if key[0] == 'l' and key[1].isdigit():
        return int(key[1:key.index('.')])
    return depth


class _Slot(nn.Module):
    """parameter-free placeholder keeping vit_pytorch's child indices (Rearrange, GELU, Dropout...)"""

    def __init__(self, what):
        super().__init__()
        self.what = what

    def extra_repr(self):
        return self.what


def _no_eager(self, *a, **k):
    raise RuntimeError('ecg_b200 modules hold parameters only; call EcgVit.forward (sm_100a kernels, no eager path)')


class PreNorm(nn.Module):
    def __init__(self, dim, fn):
        super().__init__()
        self.norm = nn.LayerNorm(dim)
        self.fn = fn
    forward = _no_eager


class Attention(nn.Module):
    def __init__(self, dim, heads, dim_head, dropout):
        super().__init__()
        inner = heads * dim_head
        self.heads, self.scale = heads, dim_head ** -0.5
        self.attend = _Slot('Softmax(dim=-1) [fused]')
        self.dropout = _Slot(f'Dropout(p={dropout})')
        self.to_qkv = nn.Linear(dim, inner * 3, bias=False)
        self.to_out = nn.Sequential(nn.Linear(inner, dim), _Slot(f'Dropout(p={dropout})'))
    forward = _no_eager


class FeedForward(nn.Module):
    def __init__(self, dim, hidden_dim, dropout):
        super().__init__()
        self.net = nn.Sequential(nn.Linear(dim, hidden_dim), _Slot('GELU(erf) [fused]'), _Slot(f'Dropout(p={dropout})'),
                                 nn.Linear(hidden_dim, dim), _Slot(f'Dropout(p={dropout})'))
    forward = _no_eager


class Transformer(nn.Module):
    def __init__(self, dim, depth, heads, dim_head, mlp_dim, dropout):
        super().__init__()
        self.layers = nn.ModuleList([
            nn.ModuleList([PreNorm(dim, Attention(dim, heads, dim_head, dropout)),
                           PreNorm(dim, FeedForward(dim, mlp_dim, dropout))])
            for _ in range(depth)])
    forward = _no_eager


class ViT(nn.Module):
    """parameter container with vit_pytorch.ViT's attribute names / init distributions.
    head=False leaves out `mlp_head`; mask_token=True adds the zero-initialised `mask_token` [1, 1, dim] of masked-patch
    pre-training, registered right after `cls_token`: the flat buffers follow registration order, so its gradient
    (produced last, by the embedding backward) sits with the other pre-block parameters in the last gradient bucket."""

    def __init__(self, *, signal_length, patch_size, num_classes, dim, depth, heads, mlp_dim, channels, dim_head,
                 dropout, emb_dropout, per_lead=False, head=True, mask_token=False, pool='cls'):
        super().__init__()
        assert signal_length % patch_size == 0, 'Image dimensions must be divisible by the patch size.'
        n_patch = signal_length // patch_size * (channels if per_lead else 1)
        patch_dim = patch_size if per_lead else channels * patch_size
        self.to_patch_embedding = nn.Sequential(_Slot('Rearrange b c (w p) -> b w (p c) [fused]'),
                                                nn.Linear(patch_dim, dim))
        self.pos_embedding = nn.Parameter(torch.randn(1, n_patch + 1, dim))
        self.cls_token = nn.Parameter(torch.randn(1, 1, dim))
        if mask_token:
            self.mask_token = nn.Parameter(torch.zeros(1, 1, dim))
        self.dropout = _Slot(f'Dropout(p={emb_dropout})')
        self.transformer = Transformer(dim, depth, heads, dim_head, mlp_dim, dropout)
        self.pool = pool
        self.to_latent = nn.Identity()
        if head:
            self.mlp_head = nn.Sequential(nn.LayerNorm(dim), nn.Linear(dim, num_classes))
    forward = _no_eager


class _EcgVitFunction(torch.autograd.Function):
    """autograd bridge for the reference-style loop (`loss.backward()`, train.py:280)"""

    @staticmethod
    def forward(ctx, model, sample_values, labels, *params):
        loss, logits = model._engine.forward(sample_values, labels, model.loss_reduction)
        ctx.model = model
        ctx.ws = model._engine._cur
        ctx.fwd_id = ctx.ws.fwd_id           # workspaces are cached per shape: the object alone does not identify a pass
        ctx.seed = model._engine.last_seed   # dropout seed of THIS forward: backward regenerates its masks from it
        # hand out copies: the workspace buffers are overwritten by the next forward
        loss, logits = loss.clone(), logits.clone()
        ctx.mark_non_differentiable(logits)
        return loss, logits

    @staticmethod
    def backward(ctx, grad_loss, *_grad_outputs):
        model = ctx.model
        eng = model._engine
        if ctx.ws.fwd_id != ctx.fwd_id:
            raise RuntimeError(
                'ecg_b200.EcgVit: another forward of the same input shape ran between this forward and its backward; '
                'the activation workspace (cached per shape) holds the later pass.  Call backward() before the next '
                'forward of that shape, or run the extra forward under torch.no_grad() on a different batch size.')
        eng._cur = ctx.ws   # a forward of ANOTHER shape may have run in between: its workspace is not ours
        if ctx.seed is not None and eng.last_seed != ctx.seed:
            eng.upload_seed(*ctx.seed)   # ... and it drew a new dropout seed
        # the upstream gradient stays on the device (float(grad_loss) would stall the host on the whole queue)
        g_dev = grad_loss.detach().to(torch.float32).reshape(1).contiguous()
        # Gradients are produced straight into the flat fp32 buffer and `.grad` is pointed at its views, so the
        # clip / AdamW kernels later see one contiguous array (no per-tensor copies through AccumulateGrad).
        params, views = model._param_list(), model._grad_views()
        # frozen parameters (requires_grad=False) never get a .grad, as with autograd; backward skips what only they need
        # (trainable_span), and whatever a fused kernel still writes into their slot the optimizer front end ignores
        live = [(p, v) for p, v in zip(params, views) if p.requires_grad]
        ours = [p.grad is not None and p.grad.data_ptr() == v.data_ptr() for p, v in live]
        if all(ours):
            eng.backward(grad_scale=1.0, zero_grads=False, grad_scale_dev=g_dev)  # accumulate, like autograd
        else:
            earlier = [(v, p.grad.clone()) for p, v in live if p.grad is not None]
            eng.backward(grad_scale=1.0, zero_grads=True, grad_scale_dev=g_dev)
            with torch.no_grad():
                for v, g in earlier:  # gradients accumulated before this backward (mixed ownership: rare)
                    v.add_(g)
                for p, v in live:
                    p.grad = v
        return (None, None, None) + (None,) * len(params)


def _draws_masks(config):
    """whether a training forward of this config draws dropout masks or drop-path keeps"""
    return (config.hidden_dropout_prob > 0 or config.attention_probs_dropout_prob > 0 or
            float(getattr(config, 'drop_path_rate', 0.0)) > 0)


class EcgVit(nn.Module):
    _classification_head = True   # ViT container with `mlp_head`
    _encoder_mask_token = False   # ... and without `mask_token`
    _engine_class = StepEngine

    def __init__(self, num_class: int = 71, config: EcgVitConfig = None, loss_reduction: str = 'mean'):
        super().__init__()
        config = config if config is not None else EcgVitConfig()
        hd_sz, n_head = config.hidden_size, config.num_attention_heads
        assert hd_sz % n_head == 0  # ecg_vit.py:99
        pool = getattr(config, 'pool', 'cls')
        if pool not in ('cls', 'mean'):
            raise ValueError(f"pool must be 'cls' or 'mean', got {pool!r}")
        # only the classification head pools; the pre-training heads read every patch token and ignore `pool`
        self._mean_pool = pool == 'mean' and self._classification_head
        check_drop_path_rate(getattr(config, 'drop_path_rate', 0.0))
        self.config = config
        self.num_class = num_class  # the reference builds the head from the ctor arg, not config.num_class (:105)
        self.vit = ViT(signal_length=config.max_signal_length, patch_size=config.patch_size, num_classes=num_class,
                       dim=hd_sz, depth=config.num_hidden_layers, heads=n_head, mlp_dim=config.intermediate_size,
                       channels=config.num_channels, dim_head=hd_sz // n_head,
                       dropout=config.hidden_dropout_prob,              # attention + feed-forward (ecg_vit.py:113)
                       emb_dropout=config.attention_probs_dropout_prob,  # embedding (ecg_vit.py:114)
                       per_lead=bool(getattr(config, 'per_lead_tokens', False)),
                       head=self._classification_head, mask_token=self._encoder_mask_token,
                       pool='mean' if self._mean_pool else 'cls')
        self.vit._owner = weakref.ref(self)  # lets `Recorder(model.vit)` reach the kernels (not a module: no cycle)
        self._loss_reduction = loss_reduction
        self.loss_weight = None
        # optional `transform.InputPipeline`: forward then takes RAW records and the per-record transforms of the
        # reference's dataset (Normalize / TimeEndPad / TimeOut) run inside the patch gather
        self.input_pipeline = None

        C, L = config.num_channels, config.max_signal_length
        cls_nm = self.__class__.__qualname__
        n_pch, n_l = L // config.patch_size, config.num_hidden_layers
        self.meta = {'name': cls_nm, 'input shape': f'{C} x {L}', '#patch': n_pch, '#layer': n_l, '#head': n_head}
        self.meta_str = '{' + ', '.join(f'{k}={v}' for k, v in
                                        {'nm': cls_nm, 'in-sp': f'{C}x{L}', '#p': n_pch, '#l': n_l, '#h': n_head}.items()) + '}'

        dt = getattr(config, 'compute_dtype', 'bf16')
        if dt not in ('bf16', 'fp32'):
            raise ValueError(f"compute_dtype must be 'bf16' or 'fp32', got {dt!r}")
        self._dtype_code = _lib.BF16 if dt == 'bf16' else _lib.F32
        self._act_dtype = torch.bfloat16 if dt == 'bf16' else torch.float32
        rd = getattr(config, 'residual_dtype', 'auto')
        if rd not in ('auto', 'bf16', 'fp32'):
            raise ValueError(f"residual_dtype must be 'auto', 'bf16' or 'fp32', got {rd!r}")
        # fp32 residual stream in bf16 mode (config.py): the kernels that touch the stream get dtype code BF16_RES32
        self._res_f32 = dt == 'bf16' and (rd == 'fp32' or (rd == 'auto' and config.num_hidden_layers > 12))
        self._res_code = _lib.BF16_RES32 if self._res_f32 else self._dtype_code
        self._res_dtype = torch.float32 if self._res_f32 else self._act_dtype
        self._flat_p = self._flat_g = self._shadow = None
        self._layout = None
        self._engine = None
        self._shadow_versions = None
        self._after_layer_backward = None  # hook used by the data-parallel gradient bucketing
        self._before_layer_forward = None  # hook used by the deferred optimizer (a layer waits for ITS weights only)
        self._flush_pending = None         # set by a trainer whose last update is still pending (deferred optimizer)

    # ---- reference API -----------------------------------------------------------------------------
    def to_str(self):
        return f'{self.__class__.__qualname__}, {self.config.size}'

    @property
    def loss_reduction(self):
        return self._loss_reduction

    @loss_reduction.setter
    def loss_reduction(self, r):
        self._loss_reduction = r

    def state_dict(self, *args, **kwargs):
        if self._flush_pending is not None:
            self._flush_pending()   # a deferred optimizer update is applied before anyone reads the weights
        return super().state_dict(*args, **kwargs)

    def forward(self, sample_values: torch.FloatTensor, labels: torch.LongTensor = None, time_out_spans=None):
        """`time_out_spans` (only with an `input_pipeline` that has TimeOut, training mode): int [B, 2] (start, length)
        per record; drawn on the host like the reference's TimeOut when omitted."""
        if self._flush_pending is not None:
            self._flush_pending()
        self._prepare(sample_values.device)
        pipe = self.input_pipeline
        if pipe is not None and pipe.timeout is not None and self.training:
            if time_out_spans is None:
                time_out_spans = pipe.draw_spans(sample_values.shape[0], pipe.padded_length(sample_values.shape[2]))
            self._engine.set_spans(time_out_spans)
        need_grad = torch.is_grad_enabled() and labels is not None and any(p.requires_grad for p in self.parameters())
        if self._draws_step_seed():
            self._engine.new_dropout_seed()  # masks of this forward; its backward regenerates them from the same seed
        if need_grad:
            loss, logits = _EcgVitFunction.apply(self, sample_values, labels, *self._param_list())
        else:
            loss, logits = self._engine.forward(sample_values, labels, self._loss_reduction)
            loss = None if loss is None else loss.clone()
            logits = logits.clone()
        return ModelOutput(loss=loss, logits=logits)

    def _draws_step_seed(self):
        """whether a training forward needs a fresh device seed (dropout masks, drop-path keeps)"""
        return self.training and _draws_masks(self.config)

    # ---- flat storage ------------------------------------------------------------------------------
    def _param_list(self):
        return [p for _, p in self.named_parameters()]

    def _short_names(self):
        """flat-buffer key for every parameter, in `named_parameters()` order"""
        out = OrderedDict()
        for name, _ in self.named_parameters():
            parts = name.split('.')
            wb = 'w' if parts[-1] == 'weight' else 'b'
            if parts[0] == 'recon_head':
                k = ('recon.ln.' if parts[1] == '0' else 'recon.') + wb
            elif parts[0] == 'decoder' and parts[1] != 'transformer':
                k = {'norm': 'dec.ln.' + wb, 'embed': 'dec.embed.' + wb, 'mask_token': 'dec.mask',
                     'pos_embedding': 'dec.pos'}[parts[1]]
            elif name == 'vit.pos_embedding':
                k = 'pos'
            elif name == 'vit.cls_token':
                k = 'cls'
            elif name == 'vit.mask_token':
                k = 'mask'
            elif parts[1] == 'to_patch_embedding':
                k = 'embed.' + ('w' if parts[-1] == 'weight' else 'b')
            elif parts[1] == 'mlp_head':
                k = ('head.ln.' if parts[2] == '0' else 'head.') + ('w' if parts[-1] == 'weight' else 'b')
            else:  # (vit|decoder).transformer.layers.{i}.{0|1}.(norm|fn)...
                i, branch = int(parts[3]), int(parts[4])
                wb = 'w' if parts[-1] == 'weight' else 'b'
                L = 'dec' if parts[0] == 'decoder' else 'l'
                if parts[5] == 'norm':
                    k = f'{L}{i}.ln{branch + 1}.{wb}'
                elif branch == 0:
                    k = f'{L}{i}.qkv.{wb}' if parts[6] == 'to_qkv' else f'{L}{i}.out.{wb}'
                else:
                    k = f'{L}{i}.ff1.{wb}' if parts[7] == '0' else f'{L}{i}.ff2.{wb}'
            out[name] = k
        return out

    def _flat_layout(self):
        """(layout, total): flat-buffer key -> (offset, numel, shape, parameter name), every offset a multiple of
        _ALIGN elements, in `named_parameters()` order"""
        params = dict(self.named_parameters())
        layout, off = OrderedDict(), 0
        for name, key in self._short_names().items():
            n = params[name].numel()
            layout[key] = (off, n, tuple(params[name].shape), name)
            off += (n + _ALIGN - 1) // _ALIGN * _ALIGN
        return layout, off

    def _flatten(self, device):
        params = dict(self.named_parameters())
        layout, total = self._flat_layout()
        flat = torch.zeros(total, device=device, dtype=torch.float32)
        for key, (o, n, shape, name) in layout.items():
            flat[o:o + n].copy_(params[name].detach().reshape(-1))
            params[name].data = flat[o:o + n].view(shape)
            params[name].grad = None
        self._layout, self._flat_p = layout, flat
        self._flat_g = torch.zeros(total, device=device, dtype=torch.float32)
        self._shadow = torch.empty(total, device=device, dtype=torch.bfloat16) if self._dtype_code == _lib.BF16 else None
        self._views_p = {k: self._flat_p[o:o + n].view(shape) for k, (o, n, shape, _) in layout.items()}
        self._views_g = {k: self._flat_g[o:o + n].view(shape) for k, (o, n, shape, _) in layout.items()}
        self._views_w = self._views_p if self._shadow is None else \
            {k: self._shadow[o:o + n].view(shape) for k, (o, n, shape, _) in layout.items()}
        self._shadow_versions = None
        self._engine = self._engine_class(self)

    def _is_flat(self, device):
        if self._flat_p is None or self._flat_p.device != device:
            return False
        params = dict(self.named_parameters())
        base = self._flat_p.data_ptr()
        return all(params[name].data_ptr() == base + 4 * o for _, (o, n, shape, name) in self._layout.items())

    def _prepare(self, device):
        """make sure parameters live in the flat buffer on `device` and the bf16 shadow is current"""
        if device.type != 'cuda':
            raise RuntimeError('ecg_b200.EcgVit runs on CUDA (sm_100a) only: there is no CPU path. '
                               'Move the model and inputs to a B200 with .cuda().')
        _lib.load()
        p0 = next(self.parameters())
        if p0.device != device:
            raise RuntimeError(f'model parameters are on {p0.device} but inputs are on {device}')
        if not self._is_flat(device):
            self._flatten(device)
        self.sync_shadow()

    def sync_shadow(self, force=False):
        """re-cast the bf16 weight shadow if any parameter was modified outside the fused optimizer"""
        if self._shadow is None:
            return
        versions = sum(p._version for p in self.parameters())
        if force or versions != self._shadow_versions:
            _lib.check(_lib.load().ecgvit_cast_f32_to_bf16(self._flat_p.data_ptr(), self._shadow.data_ptr(),
                                                           self._flat_p.numel(),
                                                           torch.cuda.current_stream().cuda_stream), 'cast')
            self._shadow_versions = versions

    def _weights(self):
        return self._views_w

    def _params_f32(self):
        return self._views_p

    def _grads_f32(self):
        return self._views_g

    def _grad_views(self):
        names = self._short_names()
        return [self._views_g[k] for k in names.values()]

    def trainable_span(self):
        """`TrainableSpan` of the current `requires_grad` flags: what backward, the optimizers and the gradient exchange
        have to cover.  The encoder is the bottom of every model, and the flat buffers follow forward order, so every
        trainable tensor lies in [lo, flat length) and backward can stop at the lowest trainable encoder position."""
        flags = tuple(p.requires_grad for p in self.parameters())
        span = getattr(self, '_span_cache', None)
        if span is not None and span.key == flags:
            return span
        layout, total = (self._layout, self._flat_p.numel()) if self._layout is not None else self._flat_layout()
        keys = list(layout)
        first = next((i for i, trains in enumerate(flags) if trains), None)
        if first is None:
            lowest, lo = None, total
        else:
            lo = layout[keys[first]][0]
            lowest = _forward_position(keys[first], self.config.num_hidden_layers)
        span = TrainableSpan(lowest=lowest, lo=lo,
                             frozen_inside=first is not None and not all(flags[first:]),
                             frozen=frozenset(k for k, trains in zip(keys, flags) if not trains), key=flags)
        self._span_cache = span
        return span


def _recon_patch_dim(c):
    """features of one patch, the reconstruction target's width; rejects the widths the reconstruction kernels cannot
    read"""
    per_lead = bool(getattr(c, 'per_lead_tokens', False))
    patch_dim = c.patch_size if per_lead else c.patch_size * c.num_channels
    if not per_lead and patch_dim % 8 != 0:
        # the residual / its gradient share the patch matrix's row length, and their column kernels read 8 elements
        # at a time (per-lead rows are padded to a multiple of 8 instead)
        raise ValueError(f'masked-patch pre-training needs patch_size * num_channels = {patch_dim} to be a multiple '
                         f'of 8')
    return patch_dim


class _MaskedPatchFunction(_EcgVitFunction):
    """autograd bridge of `EcgVitForMaskedPatchModeling` (`loss.backward()` then e.g. `FusedAdamW`); backward, with its
    workspace / seed guards, is `_EcgVitFunction`'s"""

    @staticmethod
    def forward(ctx, model, sample_values, bool_masked_pos, *params):
        eng = model._engine
        loss, _ = eng.forward(sample_values, bool_masked_pos=bool_masked_pos)
        ctx.model = model
        ctx.ws = eng._cur
        ctx.fwd_id = ctx.ws.fwd_id
        ctx.seed = eng.last_seed
        recon, mask = eng.reconstruction(), eng.mask()
        ctx.mark_non_differentiable(recon, mask)
        return loss.clone(), recon, mask


class EcgVitForMaskedPatchModeling(EcgVit):
    """SimMIM-style masked-patch pre-training of the `EcgVit` encoder on unlabelled records.

    Masked patches keep their place in the sequence (the encoder's shapes do not change) and enter it as the learned
    `vit.mask_token`; `recon_head` = LayerNorm + Linear(d, patch_dim) predicts every patch from its encoder output, and
    the loss is the mean squared error over the masked patches:

        loss = sum_{masked (b, w), k < K} (pred - a)^2 / (n_masked * K),   a = the patch matrix (the embedding's input)

    `forward(sample_values, bool_masked_pos=None)` -> `MaskedPatchOutput(loss, reconstruction, bool_masked_pos)`:
    `reconstruction` is fp32 [B, n, patch_dim] in the patch matrix's feature order (`t*C + c`, or `t` with per-lead
    tokens; `unpatchify` maps it back to [B, C, L]).  It is rebuilt as r + a from the residual r = pred - a that the
    loss GEMM stores, so in bf16 mode it carries r's bf16 rounding (relative error up to ~1e-2): an output to look
    at, not the loss's own prediction; `bool_masked_pos` [B, n] is the mask used.  Without one, exactly
    round(mask_ratio * n) patches per record are masked: in training mode drawn afresh every forward from the step's
    device seed (a captured training step draws new masks on every replay), in eval mode from a fixed seed (the same
    batch always gets the same mask).

    `encoder_state_dict()` hands the encoder over to fine-tuning:
    `EcgVit(config=...).load_state_dict(pre.encoder_state_dict(), strict=False)` misses only `vit.mlp_head.*`.
    `config.pool` is ignored here (the head reads every patch token); it applies to the `EcgVit` that is fine-tuned."""
    _classification_head = False
    _encoder_mask_token = True
    _engine_class = MaskedPatchEngine

    def __init__(self, config: EcgVitConfig = None, mask_ratio: float = 0.5):
        if not 0.0 <= float(mask_ratio) <= 1.0:
            raise ValueError(f'mask_ratio must lie in [0, 1], got {mask_ratio}')
        super().__init__(num_class=0, config=config)
        c = self.config
        self.recon_head = nn.Sequential(nn.LayerNorm(c.hidden_size), nn.Linear(c.hidden_size, _recon_patch_dim(c)))
        self.mask_ratio = float(mask_ratio)

    def _draws_step_seed(self):
        return self.training   # the mask is drawn afresh every training forward

    def encoder_state_dict(self):
        """the `vit.*` entries an `EcgVit` loads (everything but the mask token)"""
        return OrderedDict((k, v) for k, v in self.state_dict().items()
                           if k.startswith('vit.') and k != 'vit.mask_token')

    def unpatchify(self, reconstruction):
        """[B, n, patch_dim] in patch-matrix feature order -> [B, C, L] (the inverse of the patch gather)"""
        c = self.config
        B, n, K = reconstruction.shape
        P, C = c.patch_size, c.num_channels
        if bool(getattr(c, 'per_lead_tokens', False)):
            return reconstruction.reshape(B, C, (n // C) * P)
        return reconstruction.reshape(B, n, P, C).permute(0, 3, 1, 2).reshape(B, C, n * P)

    def forward(self, sample_values: torch.FloatTensor, bool_masked_pos: torch.BoolTensor = None, time_out_spans=None):
        if self._flush_pending is not None:
            self._flush_pending()
        self._prepare(sample_values.device)
        pipe = self.input_pipeline
        if pipe is not None and pipe.timeout is not None and self.training:
            if time_out_spans is None:
                time_out_spans = pipe.draw_spans(sample_values.shape[0], pipe.padded_length(sample_values.shape[2]))
            self._engine.set_spans(time_out_spans)
        if bool_masked_pos is not None:
            bool_masked_pos = bool_masked_pos.to(device=sample_values.device, dtype=torch.bool)
        if self._draws_step_seed():
            self._engine.new_dropout_seed()   # mask and dropout of this forward; backward reuses both
        need_grad = torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())
        if need_grad:
            loss, recon, mask = _MaskedPatchFunction.apply(self, sample_values, bool_masked_pos, *self._param_list())
        else:
            eng = self._engine
            loss, _ = eng.forward(sample_values, bool_masked_pos=bool_masked_pos)
            loss, recon, mask = loss.clone(), eng.reconstruction(), eng.mask()
        return MaskedPatchOutput(loss=loss, reconstruction=recon, bool_masked_pos=mask)


class _Decoder(nn.Module):
    """MAE decoder parameters: `norm` (the LayerNorm MAE puts at the end of its encoder; here, so that the encoder keys
    stay those of `EcgVit`), `embed` Linear(d -> d_dec), `mask_token` [1, 1, d_dec], the learned `pos_embedding`
    [1, n + 1, d_dec] and `transformer`, blocks with the encoder's structure and no dropout"""

    def __init__(self, dim, n_patch, dec_dim, depth, heads, mlp_dim):
        super().__init__()
        self.norm = nn.LayerNorm(dim)
        self.embed = nn.Linear(dim, dec_dim)
        self.mask_token = nn.Parameter(torch.zeros(1, 1, dec_dim))
        self.pos_embedding = nn.Parameter(torch.randn(1, n_patch + 1, dec_dim))
        self.transformer = Transformer(dec_dim, depth, heads, dec_dim // heads, mlp_dim, 0.0)
    forward = _no_eager


class EcgVitForMaskedAutoencoding(EcgVitForMaskedPatchModeling):
    """MAE-style pre-training of the `EcgVit` encoder on unlabelled records.

    The encoder runs over the CLS token and the visible patches only (their embeddings plus the positional embedding of
    their own positions).  `decoder` normalises and embeds its output at the decoder width, puts `decoder.mask_token` on
    every masked position, adds `decoder.pos_embedding` and runs its own, narrower blocks over all n + 1 positions;
    `recon_head` = LayerNorm + Linear(d_dec, patch_dim) predicts every patch.  The loss is the mean squared error over
    the masked patches, as in `EcgVitForMaskedPatchModeling`, whose interface this model shares: `forward` returns
    `MaskedPatchOutput(loss, reconstruction [B, n, patch_dim], bool_masked_pos)`, and `encoder_state_dict()` /
    `unpatchify()` behave the same.

    Exactly k = round(mask_ratio * n) patches of every record are masked (training: a fresh mask every forward, eval: a
    fixed one).  A caller's `bool_masked_pos` must mask the same number of patches, between 1 and n - 1, in every
    record (the encoder's token count depends on it); it is checked on the host.  The decoder has no dropout and never
    checkpoints; the encoder follows the config."""
    _encoder_mask_token = False
    _engine_class = MaskedAutoencoderEngine

    def __init__(self, config: EcgVitConfig = None, mask_ratio: float = 0.75, decoder_hidden_size: int = 256,
                 decoder_num_hidden_layers: int = 4, decoder_num_attention_heads: int = 4,
                 decoder_intermediate_size: int = 1024):
        EcgVit.__init__(self, num_class=0, config=config)
        c = self.config
        n = c.max_signal_length // c.patch_size * (c.num_channels if getattr(c, 'per_lead_tokens', False) else 1)
        k = int(round(float(mask_ratio) * n))
        if not 1 <= k <= n - 1:
            raise ValueError(f'mask_ratio {mask_ratio} masks {k} of {n} patches: MAE needs at least one masked and one '
                             f'visible patch')
        dd, dh = int(decoder_hidden_size), int(decoder_num_attention_heads)
        if dh < 1 or dd % dh != 0:
            raise ValueError(f'decoder_hidden_size {dd} is not a multiple of decoder_num_attention_heads {dh}')
        if (dd // dh) % 8 != 0:
            raise ValueError(f'decoder head dim {dd // dh} must be a multiple of 8')
        if int(decoder_intermediate_size) < 8 or int(decoder_intermediate_size) % 8 != 0:
            # the decoder's MLP width is a GEMM row length: 16-byte aligned rows
            raise ValueError(f'decoder_intermediate_size {decoder_intermediate_size} must be a positive multiple of 8')
        if int(decoder_num_hidden_layers) < 1:
            raise ValueError('the decoder needs at least one block')
        patch_dim = _recon_patch_dim(c)
        self.decoder = _Decoder(c.hidden_size, n, dd, int(decoder_num_hidden_layers), dh, int(decoder_intermediate_size))
        self.recon_head = nn.Sequential(nn.LayerNorm(dd), nn.Linear(dd, patch_dim))
        self.mask_ratio = float(mask_ratio)
        self.decoder_hidden_size, self.decoder_num_hidden_layers = dd, int(decoder_num_hidden_layers)
        self.decoder_num_attention_heads, self.decoder_intermediate_size = dh, int(decoder_intermediate_size)

    def forward(self, sample_values: torch.FloatTensor, bool_masked_pos: torch.BoolTensor = None, time_out_spans=None):
        if bool_masked_pos is not None:
            counts = bool_masked_pos.reshape(bool_masked_pos.shape[0], -1).sum(1).cpu()
            n = self.vit.pos_embedding.shape[1] - 1
            if not (counts == counts[0]).all() or not 1 <= int(counts[0]) <= n - 1:
                raise ValueError(f'bool_masked_pos must mask the same number of patches, between 1 and {n - 1}, in every '
                                 f'record; got counts {counts.tolist()}')
        return super().forward(sample_values, bool_masked_pos, time_out_spans)


class Recorder(nn.Module):
    """`vit_pytorch.recorder.Recorder` for the fused model: `Recorder(model.vit)(img)` returns
    `(logits, attns[b, layers, heads, n, n])`, the per-layer softmax probabilities the reference's `EcgVitVisualizer`
    reads (`ecg_vit.py:176-193`; `img` is `[B, C, 1, L]`, the dummy height axis the reference adds).  vit_pytorch
    collects them with forward hooks on `Attention.attend`; here a slow-path kernel writes them next to the fused
    attention (which never materialises them).  Dropout is not applied to the recorded probabilities (the hook sits on
    the Softmax), and the pass runs in whatever mode the model is in, as in vit_pytorch."""

    def __init__(self, vit, device=None):
        super().__init__()
        owner = getattr(vit, '_owner', None)
        if owner is None or owner() is None:
            raise RuntimeError('Recorder needs the `.vit` of an ecg_b200.EcgVit')
        self.vit = vit
        self.device = device
        self.ejected = False
        self.recordings = []

    def eject(self):
        self.ejected = True
        self.recordings = []
        return self.vit

    def clear(self):
        self.recordings = []

    def forward(self, img):
        assert not self.ejected, 'recorder has been ejected, cannot be used anymore'
        self.clear()
        model = self.vit._owner()
        assert img.dim() == 4 and img.shape[2] == 1, 'expected [B, C, 1, L] (height axis of 1, ecg_vit.py:141)'
        model._prepare(img.device)
        if model.training and _draws_masks(model.config):
            model._engine.new_dropout_seed()
        with torch.no_grad():
            _, logits = model._engine.forward(img.squeeze(2), None, model.loss_reduction, record_attention=True)
        attns = model._engine.recorded_attention
        target = self.device if self.device is not None else img.device
        self.recordings = [attns[:, l] for l in range(attns.shape[1])]
        return logits.clone(), attns.to(target)
