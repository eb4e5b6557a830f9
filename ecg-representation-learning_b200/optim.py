"""
`torch.optim`-compatible front ends for the fused flat-buffer kernels, so a reference-style loop
(/root/reference/ecg_transformer/models/train.py:242-252,271-283)

    optimizer = FusedAdamW(model, lr=lr, weight_decay=dc); scheduler = get_*_schedule_with_warmup(optimizer, ...)
    optimizer.zero_grad(); loss = model(**inputs).loss; loss.backward()
    clip_grad_norm_(model, max_norm=1.0, error_if_nonfinite=True); optimizer.step(); scheduler.step()

keeps working unchanged while each of clip / step is one or two kernel launches instead of ~1.4 k.
"""
import contextlib
import math
from collections import OrderedDict

import torch

from . import _lib



UNGROUPED = 255   # group id of the parameters in no group: the grouped AdamW leaves them untouched
MAX_GROUPS = 255
NO_WEIGHT_DECAY = ('vit.pos_embedding', 'vit.cls_token', 'vit.mask_token', 'decoder.mask_token')


def _layer_id(name, depth):
    """MAE's `get_layer_id_for_vit` over this model's names: 0 = embedding, CLS, positions and mask token, i + 1 = encoder
    block i, depth + 1 = everything else (the classification head, or the pre-training decoder and head)"""
    if name.startswith('vit.to_patch_embedding.') or name in ('vit.pos_embedding', 'vit.cls_token', 'vit.mask_token'):
        return 0
    if name.startswith('vit.transformer.layers.'):
        return int(name.split('.')[3]) + 1
    return depth + 1


def param_groups_lrd(model, weight_decay=0.05, layer_decay=0.75, no_weight_decay=NO_WEIGHT_DECAY):
    """Parameter groups for fine-tuning with layer-wise learning-rate decay (MAE's `param_groups_lrd`): encoder block i
    gets lr * layer_decay^(depth - i), the embedding layer_decay^(depth + 1), the head the full lr; 1-D tensors (biases,
    LayerNorms) and the `no_weight_decay` parameter names get no weight decay.  Returns one
    `{'params', 'lr_scale', 'weight_decay'}` dict per (layer, decay or not), in order of first appearance, for
    `FusedAdamW(..., param_groups=...)`, `FusedTrainer(..., param_groups=...)` or `torch.optim.AdamW`.
    layer_decay=1.0 gives the plain decay / no-decay split."""
    depth = model.config.num_hidden_layers
    no_wd = set(no_weight_decay)
    groups = {}
    for name, p in model.named_parameters():
        if not p.requires_grad:
            continue
        decay = not (p.ndim == 1 or name in no_wd)
        lid = _layer_id(name, depth)
        g = groups.get((lid, decay))
        if g is None:
            g = groups[(lid, decay)] = {'params': [], 'lr_scale': float(layer_decay) ** (depth + 1 - lid),
                                        'weight_decay': float(weight_decay) if decay else 0.0}
        g['params'].append(p)
    return list(groups.values())


def group_names(model, param_groups):
    """the parameter names of every group (`model.named_parameters()` names); raises on a tensor that is not one of the
    model's parameters or that sits in two groups"""
    names = {id(p): n for n, p in model.named_parameters()}
    seen, out = set(), []
    for g in param_groups:
        ps = g['params']
        ps = [ps] if isinstance(ps, torch.Tensor) else list(ps)
        row = []
        for p in ps:
            if id(p) not in names:
                raise ValueError('a parameter group holds a tensor that is not a parameter of the model')
            if id(p) in seen:
                raise ValueError('some parameters appear in more than one parameter group')
            seen.add(id(p))
            row.append(names[id(p)])
        out.append(tuple(row))
    if len(out) > MAX_GROUPS:
        raise ValueError(f'at most {MAX_GROUPS} parameter groups, got {len(out)}')
    return out


def group_map(model, names_per_group):
    """uint8 [flat length / 64] (host): the group id of every 64-element block of the model's flat buffers, UNGROUPED
    for parameters in no group (every tensor starts on a 64-element boundary, so a block never straddles two)"""
    from .model import _ALIGN
    layout, total = (model._layout, model._flat_p.numel()) if model._layout is not None else model._flat_layout()
    where = {name: (o, n) for o, n, _, name in layout.values()}
    gm = torch.full((total // _ALIGN,), UNGROUPED, dtype=torch.uint8)
    for gid, names in enumerate(names_per_group):
        for name in names:
            o, n = where[name]
            gm[o // _ALIGN:(o + n + _ALIGN - 1) // _ALIGN] = gid
    return gm


def group_table(lrs, weight_decays, beta1, step):
    """the grouped AdamW's per-group scalars [1 - lr * wd, lr / (1 - beta1^t)] in double precision, as
    `adamw_hyper` derives hyper's own"""
    bc1 = 1.0 - beta1 ** step
    out = []
    for lr, wd in zip(lrs, weight_decays):
        out += [1.0 - lr * wd, lr / bc1]
    return out


class WeightEma:
    """The exponential moving average of a model's weights that `FusedTrainer` and `FusedAdamW` update inside their AdamW
    kernel (`ecgvit_adamw_step_ema`): a flat fp32 buffer shaped like `model._flat_p`.  After the AdamW update of
    optimizer step t (1-based, the step of AdamW's bias correction) has written p_t,

        ema <- ema + (1 - d_t) * (p_t - ema),    d_t = decay,  or with warmup  d_t = min(decay, (1 + t) / (10 + t))

    (the `num_updates` form of TensorFlow's `ExponentialMovingAverage`).  The buffer starts as a copy of the weights
    when the optimizer state is created (the first step).  Exactly the elements the step updates are averaged: frozen
    tensors and skipped updates leave it untouched."""

    def __init__(self, decay, warmup=False):
        if warmup and decay is None:
            raise ValueError('ema_warmup=True needs ema_decay')
        if not 0.0 < float(decay) < 1.0:
            raise ValueError(f'ema_decay must lie in (0, 1), got {decay!r}')
        self.decay, self.warmup = float(decay), bool(warmup)
        self.buf = None
        self.active = False    # inside `weights()`
        self.swapped = False   # ... and the model holds the average, `buf` the trained weights

    @classmethod
    def create(cls, decay, warmup):
        """None without EMA (`ema_decay=None`); raises on a decay outside (0, 1) or a warm-up without a decay"""
        if decay is None and not warmup:
            return None
        return cls(decay, warmup)

    def decay_at(self, t):
        return min(self.decay, (1.0 + t) / (10.0 + t)) if self.warmup else self.decay

    def rate(self, t):
        """hyper[15] of optimizer step t: 1 - d_t in double precision"""
        return 1.0 - self.decay_at(t)

    def ensure(self, flat_p):
        """create the buffer from the weights (first step), or move it to the weights' device; keeps a buffer of the same
        length (loaded before the first step, or the model re-flattened its parameters)"""
        if self.buf is not None and self.buf.numel() == flat_p.numel() and self.buf.device == flat_p.device:
            return
        old = self.buf
        self.buf = flat_p.detach().clone()
        if old is not None and old.numel() == flat_p.numel():
            self.buf.copy_(old)

    def check_inactive(self, what):
        if self.active:
            raise RuntimeError(f'{what} inside ema_weights(): leave the context first')

    def average(self, model):
        """the flat tensor that holds the average right now (None before the first step)"""
        return model._flat_p if self.swapped else self.buf

    @contextlib.contextmanager
    def weights(self, model):
        """the model's weights (fp32 master and bf16 shadow) are the average inside the context, and bit-identical to
        before on exit; `ecgvit_swap_f32_cast` exchanges the two buffers in place and re-casts the shadow in one pass.
        Before the first step the average is the weights themselves and nothing is swapped."""
        if self.active:
            raise RuntimeError('ema_weights() is already active: it does not nest')
        swap = self.buf is not None
        if swap:
            self._swap(model)
        self.active, self.swapped = True, swap
        try:
            yield
        finally:
            if swap:
                self._swap(model)
            self.active = self.swapped = False

    def _swap(self, model):
        _lib.check(_lib.load().ecgvit_swap_f32_cast(model._flat_p.data_ptr(), self.buf.data_ptr(), _lib.ptr(model._shadow),
                                                    self.buf.numel(), torch.cuda.current_stream().cuda_stream),
                   'swap_f32_cast')

    def state_dict(self, model):
        """the average in the model's own `state_dict()` keys (loads with strict=True into the same model class)"""
        sd = model.state_dict()
        avg = self.average(model)
        if avg is None or self.swapped:
            return OrderedDict((k, v.detach().clone()) for k, v in sd.items())
        for o, n, shape, name in model._layout.values():
            sd[name] = avg[o:o + n].view(shape).clone()
        return sd

    def load(self, model, flat):
        """the buffer from a checkpoint's flat tensor, or from the current weights when the checkpoint has none"""
        self.check_inactive('loading a checkpoint')
        self.ensure(model._flat_p)
        self.buf.copy_(model._flat_p if flat is None else flat)


def _flat_grads(model):
    """make `model._flat_g` hold the current `.grad` of every parameter and return it"""
    views = model._grad_views()
    params = model._param_list()
    src, dst = [], []
    for p, v in zip(params, views):
        if p.grad is None:
            v.zero_()
        elif p.grad.data_ptr() != v.data_ptr():
            src.append(p.grad)
            dst.append(v)
    if dst:
        torch._foreach_copy_(dst, src)
        for p, v in zip(params, views):
            if p.grad is not None:
                p.grad = v
    return model._flat_g


def _scratch(model):
    if getattr(model, '_opt_scratch', None) is None or model._opt_scratch[0].device != model._flat_p.device:
        dev = model._flat_p.device
        model._opt_scratch = (torch.zeros(16, device=dev), torch.zeros(_lib.STATS_FLOATS, device=dev))
    return model._opt_scratch


def _upload(model, hyper, values):
    """asynchronous upload of the 64-byte hyper-parameter block through a ring of pinned slots (a copy from pageable
    memory would make the host wait for everything queued on the stream, i.e. for the previous step)"""
    ring = getattr(model, '_opt_ring', None)
    if ring is None:
        ring = model._opt_ring = _lib.PinnedRing(len(values), torch.float32)
    ring.upload(hyper, values)


def clip_grad_norm_(model, max_norm, norm_type=2.0, error_if_nonfinite=False):
    """`nn.utils.clip_grad_norm_` over all parameters of an `EcgVit` (train.py:281); returns the total norm."""
    if float(norm_type) != 2.0:
        raise NotImplementedError('only the 2-norm is implemented')
    lib = _lib.load()
    g = _flat_grads(model)
    hyper, stats = _scratch(model)
    _upload(model, hyper, _lib.adamw_hyper(0.0, 0.9, 0.999, 1e-8, 0.0, 1, float(max_norm), 1.0))
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.ecgvit_grad_sumsq(g.data_ptr(), _lib.F32, g.numel(), hyper.data_ptr(), stats.data_ptr(), st), 'grad_sumsq')
    _lib.check(lib.ecgvit_grad_scale_by_clip(g.data_ptr(), g.numel(), hyper.data_ptr(), stats.data_ptr(), st),
               'grad_scale_by_clip')
    total_norm = stats[2].clone()   # a device scalar, like torch's; only error_if_nonfinite reads it on the host
    if error_if_nonfinite and not math.isfinite(float(total_norm)):
        raise RuntimeError(
            f'The total norm of order {float(norm_type)} for gradients from `parameters` is non-finite, so it cannot '
            f'be clipped. To disable this error and scale the gradients by the non-finite norm anyway, set '
            f'`error_if_nonfinite=False`')
    return total_norm


class FusedAdamW(torch.optim.Optimizer):
    """AdamW over the model's flat parameter buffer; by default one group, decay on everything (train.py:242-244).

    `param_groups` (e.g. from `param_groups_lrd`): a list of `{'params', 'lr_scale', 'weight_decay', ...}` dicts.  A
    group's `lr` defaults to `lr * lr_scale`, so `LambdaLR` and transformers' schedulers scale every group as they do
    for `torch.optim.AdamW`; `step()` reads every group's current `lr` and `weight_decay`.  Parameters in no group are
    not updated.  All groups share the constructor's betas and eps (a group with others raises `ValueError`).

    `state_dict()` / `load_state_dict()` carry the moments and the step count (as flat tensors under `state['flat']`),
    so the usual `torch.save(optimizer.state_dict())` checkpoint resumes exactly.  Parameters whose `.grad` is None
    (frozen ones: requires_grad=False) are left untouched (value and moments), as torch.optim.AdamW leaves them: the
    grouped kernel's map gives them id 255.

    `ema_decay` (in (0, 1); None = no average) keeps an exponential moving average of the weights, updated by the AdamW
    kernel itself (`WeightEma`: ema <- ema + (1 - d_t) * (p_t - ema), d_t = ema_decay, or with `ema_warmup=True`
    min(ema_decay, (1 + t) / (10 + t))).  `ema_weights()` puts it into the model for evaluation or saving,
    `ema_state_dict()` returns it in the model's keys, and `state_dict()['flat']['ema']` carries it."""

    def __init__(self, model, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, param_groups=None,
                 ema_decay=None, ema_warmup=False):
        self.ema = WeightEma.create(ema_decay, ema_warmup)
        self.model = model
        self._grouped = param_groups is not None
        params = model.parameters()
        if self._grouped:
            params = []
            for g in param_groups:
                g = dict(g)
                g.setdefault('lr', lr * float(g.get('lr_scale', 1.0)))
                params.append(g)
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        if self._grouped:
            self._check_groups()
        self._step = 0
        self._m = self._v = None
        self._gmap = self._gmap_key = None
        self._ghyper = self._gring = None

    def _check_groups(self):
        b, e = tuple(self.defaults['betas']), self.defaults['eps']
        for g in self.param_groups:
            if tuple(g['betas']) != b or g['eps'] != e:
                raise ValueError(f'FusedAdamW: every parameter group shares betas {b} and eps {e}; a group has '
                                 f'betas {tuple(g["betas"])}, eps {g["eps"]}')

    def _ensure_moments(self, g):
        n = g.numel()
        if self._m is None or self._m.numel() != n or self._m.device != g.device:
            old = (self._m, self._v)
            self._m, self._v = torch.zeros_like(g), torch.zeros_like(g)
            if old[0] is not None and old[0].numel() == n:   # moved device / loaded on the CPU before the first step
                self._m.copy_(old[0])
                self._v.copy_(old[1])

    @torch.no_grad()
    def step(self, closure=None):
        if self.ema is not None:
            self.ema.check_inactive('step()')
        loss = closure() if closure is not None else None
        model = self.model
        model._prepare(next(model.parameters()).device)
        # parameters without a gradient (frozen tensors) keep their value and moments, as torch skips them: the grouped
        # kernel leaves them out through its map (one group when no groups were given)
        no_grad = frozenset(name for name, p in model.named_parameters() if p.grad is None)
        g = _flat_grads(model)
        n = g.numel()
        self._ensure_moments(g)
        if self.ema is not None:
            self.ema.ensure(model._flat_p)
        grp = self.param_groups[0]
        self._step += 1
        hyper, stats = _scratch(model)
        b1, b2 = grp['betas']
        st = torch.cuda.current_stream().cuda_stream
        if self._grouped or no_grad:
            self._grouped_step(g, stats, st, no_grad)
        else:
            # max_norm 0: clipping is a separate call in the reference loop
            _upload(model, hyper, _lib.adamw_hyper(grp['lr'], b1, b2, grp['eps'], grp['weight_decay'], self._step, 0.0,
                                                   1.0, ema_rate=self._ema_rate()))
            stats.zero_()
            args = (model._flat_p.data_ptr(), self._m.data_ptr(), self._v.data_ptr(), g.data_ptr(), _lib.F32,
                    _lib.ptr(model._shadow))
            if self.ema is None:
                _lib.check(_lib.load().ecgvit_adamw_step(*args, n, hyper.data_ptr(), stats.data_ptr(), 0, st),
                           'adamw_step')
            else:
                _lib.check(_lib.load().ecgvit_adamw_step_ema(*args, self.ema.buf.data_ptr(), n, None, None,
                                                             hyper.data_ptr(), stats.data_ptr(), 0, st), 'adamw_step_ema')
        return loss

    def _ema_rate(self):
        return 0.0 if self.ema is None else self.ema.rate(self._step)

    def _grouped_step(self, g, stats, st, no_grad):
        """ecgvit_adamw_step_grouped with every group's current lr / weight decay and the parameters named in `no_grad`
        at id 255; the group map is rebuilt when the membership, the parameters without a gradient or the flat layout
        change"""
        model = self.model
        self._check_groups()
        names = group_names(model, self.param_groups) if self._grouped else [tuple(n for n, _ in model.named_parameters())]
        names = [tuple(n for n in row if n not in no_grad) for row in names]
        key = (tuple(names), model._flat_p.data_ptr())
        if self._gmap_key != key:
            self._gmap = group_map(model, names).to(model._flat_p.device)
            self._gmap_key = key
        b1, b2 = self.defaults['betas']
        vals = _lib.adamw_hyper(0.0, b1, b2, self.defaults['eps'], 0.0, self._step, 0.0, 1.0, ema_rate=self._ema_rate())
        vals += group_table([grp['lr'] for grp in self.param_groups], [grp['weight_decay'] for grp in self.param_groups],
                            b1, self._step)
        if self._ghyper is None or self._ghyper.numel() != len(vals) or self._ghyper.device != g.device:
            self._ghyper = torch.zeros(len(vals), device=g.device)
            self._gring = _lib.PinnedRing(len(vals), torch.float32)
        self._gring.upload(self._ghyper, vals)   # hyper block, then the group table right behind it
        stats.zero_()
        args = (model._flat_p.data_ptr(), self._m.data_ptr(), self._v.data_ptr(), g.data_ptr(), _lib.F32,
                _lib.ptr(model._shadow))
        tail = (g.numel(), self._gmap.data_ptr(), self._ghyper.data_ptr() + 64, self._ghyper.data_ptr(),
                stats.data_ptr(), 0, st)
        if self.ema is None:
            _lib.check(_lib.load().ecgvit_adamw_step_grouped(*args, *tail), 'adamw_step_grouped')
        else:
            _lib.check(_lib.load().ecgvit_adamw_step_ema(*args, self.ema.buf.data_ptr(), *tail), 'adamw_step_ema')

    # ---- the weight moving average ----
    def ema_weights(self):
        """context manager: inside it the model's weights are the moving average (`WeightEma.weights`); `step()`
        inside it and nesting it raise `RuntimeError`"""
        return _require_ema(self.ema).weights(self.model)

    def ema_state_dict(self):
        """the moving average in the model's `state_dict()` keys"""
        return _require_ema(self.ema).state_dict(self.model)

    # ---- checkpointing: torch.optim.Optimizer.state is empty here (the moments are flat), so carry them explicitly ----
    def state_dict(self):
        sd = super().state_dict()
        sd['flat'] = {'step': self._step,
                      'exp_avg': None if self._m is None else self._m.detach().clone(),
                      'exp_avg_sq': None if self._v is None else self._v.detach().clone()}
        if self.ema is not None:
            avg = self.ema.average(self.model)
            sd['flat']['ema'] = None if avg is None else avg.detach().clone()
        return sd

    def load_state_dict(self, state_dict):
        state_dict = dict(state_dict)
        flat = state_dict.pop('flat', None)
        super().load_state_dict(state_dict)
        if flat is not None:
            self._step = int(flat['step'])
            if flat['exp_avg'] is not None:
                dev = next(self.model.parameters()).device
                self._m = flat['exp_avg'].detach().to(device=dev, dtype=torch.float32).clone()
                self._v = flat['exp_avg_sq'].detach().to(device=dev, dtype=torch.float32).clone()
            else:
                self._m = self._v = None
            if self.ema is not None:
                self.ema.check_inactive('load_state_dict()')
                ema = flat.get('ema')
                if ema is not None:
                    self.ema.buf = ema.detach().to(device=next(self.model.parameters()).device,
                                                   dtype=torch.float32).clone()
                elif self.ema.buf is not None:   # no average in the checkpoint: start it from the loaded weights
                    self.ema.load(self.model, None)


def _require_ema(ema):
    if ema is None:
        raise ValueError('the optimizer keeps no weight moving average: pass ema_decay=...')
    return ema
