"""
Fused training step with the semantics of `MyTrainer.train`'s inner loop
(/root/reference/ecg_transformer/models/train.py:268-283):

    zero_grad -> model(**inputs) -> loss.backward() -> clip_grad_norm_(1.0, error_if_nonfinite=True)
              -> AdamW.step() -> scheduler.step()

but with no autograd graph, no per-tensor optimizer launches and no host synchronisation: the loss stays on the
device (the reference syncs twice per step for logging, train.py:278,289), the LR schedule runs on the host and
reaches the kernels through a 64-byte device block, and the non-finite check of `clip_grad_norm_` is a device
flag polled on request.  With `world_size > 1` gradients are summed over NCCL in per-layer buckets on a side
stream while backward is still running (`parallel.py`).
"""
import collections
import contextlib
import math
import os

import torch

from . import _lib
from .optim import WeightEma



def lr_multiplier(schedule, step, n_warmup, n_total):
    """transformers' `get_constant_schedule_with_warmup` / `get_cosine_schedule_with_warmup` (train.py:245-252)."""
    if step < n_warmup:
        return float(step) / float(max(1, n_warmup))
    if schedule == 'constant':
        return 1.0
    progress = float(step - n_warmup) / float(max(1, n_total - n_warmup))
    return max(0.0, 0.5 * (1.0 + math.cos(math.pi * progress)))


def get_train_args(args=None, n_train=None):
    """defaults of the reference trainer (train.py:407-436) that matter to the step"""
    out = dict(num_train_epoch=3, train_batch_size=64, optimizer='AdamW', learning_rate=3e-4, weight_decay=1e-2,
               warmup_ratio=0.05, schedule='cosine', max_grad_norm=1.0)
    out.update(args or {})
    if out['optimizer'] not in ('AdamW',):
        raise ValueError("only optimizer='AdamW' is implemented in the fused step")
    if out['schedule'] not in ('constant', 'cosine'):
        raise ValueError(f"Unexpected schedule: expect one of ['constant', 'cosine'], got {out['schedule']!r}")
    if n_train is not None:
        out['steps_per_epoch'] = n_train // out['train_batch_size']
        out['n_step'] = out['steps_per_epoch'] * out['num_train_epoch']
    return out


class FusedTrainer:
    """`ema_decay` (in (0, 1); None = no average) keeps an exponential moving average of the weights, updated inside
    the AdamW kernel after every update (`optim.WeightEma`): ema <- ema + (1 - d_t) * (p_t - ema) with d_t = ema_decay,
    or with `ema_warmup=True` d_t = min(ema_decay, (1 + t) / (10 + t)), t the 1-based optimizer step.  `ema_weights()`
    evaluates or saves it, `fit` evaluates it next to the weights (`eval_ema/*`) and `save()` writes
    `model_ema - <tag>.pt`."""

    def __init__(self, model, learning_rate=3e-4, weight_decay=1e-2, betas=(0.9, 0.999), eps=1e-8,
                 schedule='constant', n_warmup=0, n_step=1 << 30, max_grad_norm=1.0, process_group=None,
                 bucket_layers=1, use_cuda_graph=False, data_parallel=True, grad_reduce_dtype='auto',
                 defer_optimizer=False, param_groups=None, ema_decay=None, ema_warmup=False):
        self.ema = WeightEma.create(ema_decay, ema_warmup)
        self.model = model
        self._flat_ptr = None
        self.lr, self.wd, self.betas, self.eps = learning_rate, weight_decay, betas, eps
        self.schedule, self.n_warmup, self.n_step = schedule, n_warmup, n_step
        self.max_grad_norm = max_grad_norm
        self.step_count = 0
        self.lib = _lib.load()
        self.group = process_group
        self.world = 1
        if data_parallel and (process_group is not None or
                              (torch.distributed.is_available() and torch.distributed.is_initialized())):
            self.world = torch.distributed.get_world_size(process_group)
        self.bucket_layers = bucket_layers
        # defer_optimizer=True: step k ends after the gradient norm; its clip + AdamW run at the BEGINNING of step k + 1,
        # layer by layer on the side stream, each forward layer waiting only for its own slice: the memory-bound optimizer
        # pass (0.4 ms of a 9 ms step at cfg2) moves off the critical chain.  The training trajectory is unchanged; the last
        # update becomes visible at `flush()` (called by state_dict / save / evaluate / the model's own forward and
        # state_dict).  Off by default: measured on B200 at cfg2 it is neutral (9.17 vs 9.07 ms device-resident, 9.29 vs
        # 9.36 ms end to end) -- the optimizer's CTAs take register space on the SMs and the persistent forward GEMMs
        # (one CTA per SM) then place their last CTAs late.
        self.defer_optimizer = defer_optimizer
        self._pending_step = None   # 1-based optimizer step whose update has not been applied yet
        # dtype of the gradient all-reduce: 'fp32', 'bf16', or 'auto' = bf16 in bf16 compute mode (half the NVLink bytes,
        # half the time NCCL's kernels share the SMs with backward), fp32 in fp32 parity mode
        assert grad_reduce_dtype in ('auto', 'fp32', 'bf16')
        self.grad_reduce_dtype = grad_reduce_dtype
        self.use_cuda_graph = use_cuda_graph
        self._state_ready = False
        self._graph = None
        self._hyper_ring = None
        self._reducer = None
        self.launches_per_step = None
        self._step_done = collections.deque(maxlen=2)
        # the trainable span of the current step (`EcgVit.trainable_span`), and whether it runs the grouped kernels
        self._span = None
        self._grouped = param_groups is not None
        self._gmap = self._gmap_key = None
        # param_groups (e.g. `param_groups_lrd(model)`): per group lr = learning_rate * schedule * lr_scale and its own
        # weight decay (the trainer's when the group has none); parameters in no group are not updated.  Without groups
        # the step issues exactly the ungrouped kernels
        self.param_groups = None
        if param_groups is not None:
            from .optim import group_names
            self._group_names = group_names(model, param_groups)
            self.param_groups = []
            for g in param_groups:
                if tuple(g.get('betas', betas)) != tuple(betas) or g.get('eps', eps) != eps:
                    raise ValueError(f'FusedTrainer: every parameter group shares betas {tuple(betas)} and eps {eps}')
                wd = g.get('weight_decay')
                self.param_groups.append({'lr_scale': float(g.get('lr_scale', 1.0)),
                                          'weight_decay': None if wd is None else float(wd)})

    # ---- lazily created device state ---------------------------------------------------------------
    def _ensure_state(self, device):
        m = self.model
        m._prepare(device)
        if (self._state_ready and self.exp_avg.device == device and self.exp_avg.numel() == m._flat_p.numel()
                and self._flat_ptr == m._flat_p.data_ptr()):
            return
        # (re-)create the flat optimizer state: first use, or the model re-flattened its parameters (.to(), a dtype move,
        # load_state_dict(assign=True)): the reducer, the captured graph and the moments must follow the new buffers
        old = (self.exp_avg, self.exp_avg_sq) if self._state_ready and self.exp_avg.numel() == m._flat_p.numel() else None
        n = m._flat_p.numel()
        self.exp_avg = torch.zeros(n, device=device, dtype=torch.float32)
        self.exp_avg_sq = torch.zeros(n, device=device, dtype=torch.float32)
        if old is not None:
            self.exp_avg.copy_(old[0])
            self.exp_avg_sq.copy_(old[1])
        if self.ema is not None:
            self.ema.ensure(m._flat_p)   # first use: the average starts from the weights
        # with groups (or frozen tensors among the trainable ones: one group), the group table sits right behind the
        # 16-float hyper block: one upload per step feeds both
        n_hyper = 16 + 2 * (len(self.param_groups) if self.param_groups is not None else 1)
        self.hyper = torch.zeros(n_hyper, device=device, dtype=torch.float32)
        self._gmap = self._gmap_key = None   # built per flat layout and requires_grad flags (`_plan`)
        self.stats = torch.zeros(_lib.STATS_FLOATS, device=device, dtype=torch.float32)
        self._flat_ptr = m._flat_p.data_ptr()
        self._graph = None   # a captured graph points at the old flat buffers
        self._norm_slices = None
        if (self.world == 1 and not self.defer_optimizer and m._engine.side_stream is not None
                and os.environ.get('ECGVIT_SLICE_NORM', '0') == '1'):
            # experiment (off by default): reduce the gradient norm slice by slice beside backward (a layer's slice is
            # final -- and still in L2 -- the moment its weight-gradient GEMMs finish) so that only a one-CTA fold sits
            # between backward and AdamW instead of a 342 MB pass.  Measured on B200: 9.18 vs 9.00 ms per step -- the
            # per-layer join of the side stream with the main chain and the extra kernels beside the persistent GEMMs
            # cost more than the 66 us pass they hide.
            from .parallel import bucket_slices
            depth = m.config.num_hidden_layers
            offs = [m._layout[f'l{l}.ln1.w'][0] for l in range(depth)]
            slices = bucket_slices(offs, n, depth, 1)
            per = max(1, min(148, _lib.SUMSQ_MAX_BLOCKS // len(slices)))
            self._norm_slices = {t: (lo, hi, i * per, per) for i, (t, lo, hi) in enumerate(slices)}
            self._norm_blocks = per * len(slices)
            m._after_layer_backward = self._slice_norm
        if self.world > 1:
            from .parallel import BucketedGradReducer
            dist = torch.distributed
            bf16 = self.grad_reduce_dtype == 'bf16' or (self.grad_reduce_dtype == 'auto' and m._dtype_code == _lib.BF16)
            self._reducer = BucketedGradReducer(m, self.group, self.bucket_layers, bf16=bf16)
            m._engine.rank_offset = 7919 * dist.get_rank(self.group)  # independent dropout masks per replica
            # replicas must start from the same weights and optimizer state whatever each rank's RNG or checkpoint did
            # (torch DDP broadcasts at construction too): rank 0 wins
            src = dist.get_global_rank(self.group, 0) if self.group is not None else 0
            for t in (m._flat_p, self.exp_avg, self.exp_avg_sq) + (() if self.ema is None else (self.ema.buf,)):
                dist.broadcast(t, src=src, group=self.group)
            cnt = torch.tensor([self.step_count], device=device, dtype=torch.int64)
            dist.broadcast(cnt, src=src, group=self.group)
            self.step_count = int(cnt)
            m.sync_shadow(force=True)
        self._state_ready = True

    def _plan(self):
        """read the requires_grad flags: the trainable span and, when the grouped kernels run, the group map with the
        frozen tensors at id 255 (no groups: one group at the trainer's lr / weight decay)"""
        m = self.model
        span = m.trainable_span()
        if span.lowest is None:
            raise ValueError('FusedTrainer: every parameter has requires_grad=False, there is nothing to train')
        if span.frozen and self.defer_optimizer:
            raise ValueError('FusedTrainer: defer_optimizer=True does not support frozen parameters '
                             '(requires_grad=False); use the default defer_optimizer=False')
        self._span = span
        self._grouped = self.param_groups is not None or span.frozen_inside
        if self._grouped and self._gmap_key != (span.key, self._flat_ptr):
            from .optim import group_map
            names = self._group_names if self.param_groups is not None else [tuple(v[3] for v in m._layout.values())]
            frozen = {m._layout[k][3] for k in span.frozen}
            self._gmap = group_map(m, [tuple(n for n in g if n not in frozen) for g in names]).to(m._flat_p.device)
            self._gmap_key = (span.key, self._flat_ptr)
        if self._reducer is not None and self._reducer.span_key != span.key:
            from .parallel import BucketedGradReducer
            self._reducer = BucketedGradReducer(m, self.group, self.bucket_layers, bf16=self._reducer.flat_g16 is not None)

    def current_lr(self):
        return self.lr * lr_multiplier(self.schedule, self.step_count, self.n_warmup, self.n_step)

    def _hyper_values(self, t):
        """hyper block of optimizer step t (1-based; lr = schedule(t - 1), the value LambdaLR holds when the reference
        calls optimizer.step() for the t-th time); t None = nothing to apply (skip flag)"""
        b1, b2 = self.betas
        mg = self.max_grad_norm if self.max_grad_norm is not None else 0.0
        groups = self.param_groups if self.param_groups is not None else [{'lr_scale': 1.0, 'weight_decay': None}]
        if t is None:
            vals = _lib.adamw_hyper(0.0, b1, b2, self.eps, self.wd, 1, mg, 1.0 / self.world, skip=True)
            return vals if not self._grouped else vals + [1.0, 0.0] * len(groups)
        lr = self.lr * lr_multiplier(self.schedule, t - 1, self.n_warmup, self.n_step)
        vals = _lib.adamw_hyper(lr, b1, b2, self.eps, self.wd, t, mg, 1.0 / self.world,
                                ema_rate=0.0 if self.ema is None else self.ema.rate(t))
        if not self._grouped:
            return vals
        from .optim import group_table
        return vals + group_table([lr * g['lr_scale'] for g in groups],
                                  [self.wd if g['weight_decay'] is None else g['weight_decay'] for g in groups], b1, t)

    def _adamw(self, p, m, v, g, g_code, shadow, lo, n, flags, stream):
        """AdamW over [lo, lo + n) of the flat buffers (the base pointers are passed; the slice offsets them)"""
        esz = 4 if g_code == _lib.F32 else 2
        args = (p + 4 * lo, m + 4 * lo, v + 4 * lo, g + esz * lo, g_code, None if shadow is None else shadow + 2 * lo, n)
        if self.ema is not None:
            from .model import _ALIGN
            gm, gt = (self._gmap.data_ptr() + lo // _ALIGN, self.hyper.data_ptr() + 64) if self._grouped else (None, None)
            _lib.check(self.lib.ecgvit_adamw_step_ema(*args[:6], self.ema.buf.data_ptr() + 4 * lo, n, gm, gt,
                                                      self.hyper.data_ptr(), self.stats.data_ptr(), flags, stream),
                       'adamw_step_ema')
        elif not self._grouped:
            _lib.check(self.lib.ecgvit_adamw_step(*args, self.hyper.data_ptr(), self.stats.data_ptr(), flags, stream),
                       'adamw_step')
        else:
            from .model import _ALIGN
            _lib.check(self.lib.ecgvit_adamw_step_grouped(*args, self._gmap.data_ptr() + lo // _ALIGN,
                                                          self.hyper.data_ptr() + 64, self.hyper.data_ptr(),
                                                          self.stats.data_ptr(), flags, stream), 'adamw_step_grouped')

    def _upload_hyper(self):
        # immediate mode: this replay applies update step_count + 1; deferred mode: it applies the PENDING update (or none)
        vals = self._hyper_values(self._pending_step if self.defer_optimizer else self.step_count + 1)
        if self._hyper_ring is None or self._hyper_ring.bufs[0].numel() != len(vals):
            self._hyper_ring = _lib.PinnedRing(len(vals), torch.float32)
        self._hyper_ring.upload(self.hyper[:len(vals)], vals)  # asynchronous: the host keeps queueing steps ahead of the device

    def _slice_norm(self, layer):
        """engine hook: the gradients of `layer` (and of everything above it) are final on the current stream"""
        s = self._norm_slices.get(layer)
        if s is None or self._span.frozen:   # the sliced norm covers the whole buffer: off while anything is frozen
            return
        lo, hi, first, per = s
        m = self.model
        _lib.check(self.lib.ecgvit_grad_sumsq_partial(m._flat_g.data_ptr() + 4 * lo, _lib.F32, hi - lo, self.hyper.data_ptr(),
                                                      self.stats.data_ptr(), first, per,
                                                      torch.cuda.current_stream().cuda_stream), 'grad_sumsq_partial')

    # ---- the step ----------------------------------------------------------------------------------
    def _device_step(self, sample_values, labels):
        m, st = self.model, torch.cuda.current_stream().cuda_stream
        eng = m._engine
        side = eng.side_stream
        # with a frozen prefix the memset, the norm and AdamW cover [lo, n) only
        lo = self._span.lo
        if side is not None:
            # the 342 MB gradient memset does not depend on the forward pass: on the side stream it becomes a parallel
            # branch of the step graph and disappears behind the (tensor-bound) forward kernels
            main = torch.cuda.current_stream()
            fork = torch.cuda.Event()
            fork.record(main)
            side.wait_event(fork)  # after the previous step's AdamW / all-reduce, which read the gradients
            if not self.defer_optimizer:
                with torch.cuda.stream(side):
                    (m._flat_g if lo == 0 else m._flat_g[lo:]).zero_()
                    zeroed = torch.cuda.Event()
                    zeroed.record(side)
        if self.defer_optimizer:
            self._issue_deferred_update(side if side is not None else torch.cuda.current_stream())
        loss, logits = eng.forward(sample_values, labels, m.loss_reduction)
        m._before_layer_forward = None
        if side is not None and not self.defer_optimizer:
            main.wait_event(zeroed)
        if self._reducer is not None:
            self._reducer.begin()
        eng.backward(grad_scale=1.0, zero_grads=side is None and not self.defer_optimizer)
        if self._reducer is not None:
            self._reducer.finish()
        n = m._flat_g.numel()
        # the buffer the exchanged gradients ended up in: the fp32 accumulation buffer, or its bf16 image when the
        # all-reduce ran in bf16
        g, g_code = (m._flat_g, _lib.F32) if self._reducer is None or self._reducer.flat_g16 is None \
            else (self._reducer.flat_g16, _lib.BF16)
        esz = 4 if g_code == _lib.F32 else 2
        if self._norm_slices is not None and not self._span.frozen:
            if side is not None:   # the slice partials were issued on the side stream
                done = torch.cuda.Event()
                done.record(side)
                main.wait_event(done)
            _lib.check(self.lib.ecgvit_grad_sumsq_finalize(self.stats.data_ptr(), self._norm_blocks, st), 'grad_sumsq_finalize')
        elif self._grouped and self._span.frozen:
            # frozen tensors (id 255 in the map) do not count in the norm
            from .model import _ALIGN
            _lib.check(self.lib.ecgvit_grad_sumsq_grouped(g.data_ptr() + esz * lo, g_code, n - lo,
                                                          self._gmap.data_ptr() + lo // _ALIGN, self.hyper.data_ptr(),
                                                          self.stats.data_ptr(), st), 'grad_sumsq_grouped')
        else:
            _lib.check(self.lib.ecgvit_grad_sumsq(g.data_ptr() + esz * lo, g_code, n - lo, self.hyper.data_ptr(),
                                                  self.stats.data_ptr(), st), 'grad_sumsq')
        if not self.defer_optimizer:
            self._adamw(m._flat_p.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(), g.data_ptr(), g_code,
                        _lib.ptr(m._shadow), lo, n - lo, 0, st)
        return loss, logits

    # ---- deferred optimizer --------------------------------------------------------------------------------------
    def _update_slices(self):
        """[(forward position, lo, hi)] of the flat buffers in the order the forward pass needs the weights: -1 = everything
        before block 0 (pos, cls, patch embedding), l = block l, depth = the head"""
        m = self.model
        depth = m.config.num_hidden_layers
        head = 'head.ln.w' if 'head.ln.w' in m._layout else 'recon.ln.w'   # classification or reconstruction head
        starts = [m._layout[f'l{l}.ln1.w'][0] for l in range(depth)] + [m._layout[head][0]]
        n = m._flat_p.numel()
        out = [(-1, 0, starts[0])]
        for l in range(depth):
            out.append((l, starts[l], starts[l + 1]))
        out.append((depth, starts[depth], n))
        return out

    def _apply_update(self, stream, events=None):
        """clip + AdamW of the pending update, slice by slice in forward order on `stream`, each slice followed by the
        zeroing of its gradients (the next backward accumulates into them); events[pos] is recorded after slice pos"""
        m = self.model
        g, g_code = (m._flat_g, _lib.F32) if self._reducer is None or self._reducer.flat_g16 is None \
            else (self._reducer.flat_g16, _lib.BF16)
        with torch.cuda.stream(stream):
            for i, (pos, lo, hi) in enumerate(self._update_slices()):
                flags = _lib.ADAMW_SLICE | (_lib.ADAMW_FIRST_SLICE if i == 0 else 0)
                self._adamw(m._flat_p.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(), g.data_ptr(),
                            g_code, _lib.ptr(m._shadow), lo, hi - lo, flags, stream.cuda_stream)
                m._flat_g[lo:hi].zero_()
                if events is not None:
                    ev = torch.cuda.Event()
                    ev.record(stream)
                    events[pos] = ev

    def _issue_deferred_update(self, side):
        """start of a deferred step: the previous step's update runs on the side stream while the forward pass starts; a
        forward layer waits for the slice holding its own weights"""
        m = self.model
        main = torch.cuda.current_stream()
        events = {}
        if side is not main:
            fork = torch.cuda.Event()
            fork.record(main)
            side.wait_event(fork)   # after the previous step's gradient norm (and all-reduce)
        self._apply_update(side, events)
        if side is not main:
            m._before_layer_forward = lambda pos: main.wait_event(events[pos])

    def flush(self):
        """apply the update a deferred step left pending (no-op otherwise); called before anything reads the weights"""
        if not self.defer_optimizer or self._pending_step is None or not self._state_ready:
            return
        t, self._pending_step = self._pending_step, None
        vals = self._hyper_values(t)
        self._hyper_ring.upload(self.hyper[:len(vals)], vals)
        self._apply_update(torch.cuda.current_stream())

    def step(self, sample_values, labels=None, time_out_spans=None):
        """One optimisation step on device-resident fp32 inputs; returns (loss, logits) device tensors (no sync).

        The returned tensors are views of workspace buffers: valid until the next step.  With an `input_pipeline` on
        the model, `sample_values` are raw records; `time_out_spans` as in `EcgVit.forward`.
        An `EcgVitForMaskedPatchModeling` takes no labels (its masks are drawn on the device) and returns (loss, None)."""
        if self.ema is not None:
            self.ema.check_inactive('step()')
        pretrain = getattr(self.model, 'mask_ratio', None) is not None
        if (labels is None) != pretrain:
            raise ValueError('a masked-patch model trains without labels' if pretrain else 'EcgVit.step needs labels')
        self._ensure_state(sample_values.device)
        self._plan()
        self._upload_hyper()
        pipe = self.model.input_pipeline
        if pipe is not None and pipe.timeout is not None and self.model.training:
            if time_out_spans is None:
                time_out_spans = pipe.draw_spans(sample_values.shape[0], pipe.padded_length(sample_values.shape[2]))
            self.model._engine.set_spans(time_out_spans)  # a persistent device buffer: the captured graph reads it
        if self.model._draws_step_seed():
            self.model._engine.new_dropout_seed()  # a device scalar: the captured graph reads the fresh value
        if self.use_cuda_graph:
            out = self._graph_step(sample_values, labels)
        else:
            out = self._device_step(sample_values, labels)
        self.step_count += 1  # scheduler.step() (train.py:283)
        if self.defer_optimizer:
            self._pending_step = self.step_count   # applied at the start of the next step, or by flush()
            self.model._flush_pending = self.flush
        ev = torch.cuda.Event()
        ev.record()
        self._step_done.append(ev)  # lets stage() reuse an input slot only after the step that read it
        return out

    def _graph_step(self, sample_values, labels):
        lw = self.model.loss_weight
        pipe = self.model.input_pipeline
        cfg = self.model.config
        # everything the capture bakes in: shapes, loss weighting / reduction, train vs eval (dropout on or off and its
        # probabilities, the drop-path rates), the input pipeline, and the flat buffers the kernels point at
        # (a masked-patch model: no labels, and its mask ratio sets how many patches the captured mask draw takes) and the
        # requires_grad flags (which backward kernels run, and over which span the optimizer does)
        key = (self._span.key, tuple(sample_values.shape), None if labels is None else tuple(labels.shape),
               tuple(float(v) for v in lw) if lw else None,
               self.model.training, float(cfg.hidden_dropout_prob), float(cfg.attention_probs_dropout_prob),
               float(getattr(cfg, 'drop_path_rate', 0.0)),
               self.model.loss_reduction, self.model._flat_p.data_ptr(),
               None if pipe is None else (id(pipe), pipe.pad, pipe.timeout), getattr(self.model, 'mask_ratio', None),
               None if self.param_groups is None else tuple(self._group_names),
               None if self._gmap is None else self._gmap.data_ptr())
        if self._graph is None or self._graph_key != key:
            self._static_x = torch.empty_like(sample_values)
            self._static_y = None if labels is None else \
                torch.empty(labels.shape, device=labels.device, dtype=torch.float32)
            self._static_x.copy_(sample_values)
            if labels is not None:
                self._static_y.copy_(labels)
            # eager warm-up (sets function attributes, allocates workspaces) on a side stream, then capture;
            # parameters/optimizer state are snapshotted so the warm-up does not count as a step
            self.flush()   # the warm-up below must not apply a pending update twice
            self._upload_hyper()
            snap = (self.model._flat_p.clone(), self.exp_avg.clone(), self.exp_avg_sq.clone(),
                    None if self.ema is None else self.ema.buf.clone())
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._device_step(self._static_x, self._static_y)
            torch.cuda.current_stream().wait_stream(s)
            self.model._flat_p.copy_(snap[0]); self.exp_avg.copy_(snap[1]); self.exp_avg_sq.copy_(snap[2])
            if self.ema is not None:
                self.ema.buf.copy_(snap[3])
            self.model.sync_shadow(force=True)
            g = torch.cuda.CUDAGraph()
            n0 = _lib.launch_counter[0]
            with torch.cuda.graph(g):
                self._graph_out = self._device_step(self._static_x, self._static_y)
            self.launches_per_step = _lib.launch_counter[0] - n0  # kernels of ours replayed by every graph launch
            self._graph, self._graph_key = g, key
        self._static_x.copy_(sample_values, non_blocking=True)
        if labels is not None:
            self._static_y.copy_(labels, non_blocking=True)
        self._graph.replay()
        return self._graph_out

    # ---- input staging ---------------------------------------------------------------------------------
    def stage(self, sample_values_host, labels_host):
        """Start the host->device copy of the NEXT batch on a side stream (pinned source recommended) and return device
        tensors whose use on the current stream is ordered after the copy.  Two slots alternate, so when calls go
        `cur = stage(); loop: step(*cur); nxt = stage(); ...; cur = nxt` the copy of batch i+1 overlaps the kernels of
        step i (the reference copies synchronously inside the step, train.py:274)."""
        dev = torch.device('cuda', torch.cuda.current_device())
        if getattr(self, '_stage_slots', None) is None or self._stage_slots[0][0].shape != sample_values_host.shape:
            self._copy_stream = torch.cuda.Stream(device=dev)
            self._stage_slots = [(torch.empty(sample_values_host.shape, device=dev, dtype=torch.float32),
                                  torch.empty(labels_host.shape, device=dev, dtype=torch.float32),
                                  torch.cuda.Event()) for _ in range(2)]
            self._stage_next = 0
        xd, yd, copied = self._stage_slots[self._stage_next]
        self._stage_next ^= 1
        cs = self._copy_stream
        # this slot was last read by the step BEFORE the most recently enqueued one (which reads the other slot)
        if len(self._step_done) == 2:
            cs.wait_event(self._step_done[0])
        elif len(self._step_done) == 1 and self.step_count >= 2:
            cs.wait_event(self._step_done[0])
        with torch.cuda.stream(cs):
            xd.copy_(sample_values_host, non_blocking=True)
            yd.copy_(labels_host, non_blocking=True)
            copied.record(cs)
        torch.cuda.current_stream().wait_event(copied)
        return xd, yd

    # ---- host-visible results (these synchronise) ----------------------------------------------------
    def grad_norm(self):
        return float(self.stats[2])

    def check_finite(self):
        """`error_if_nonfinite=True` of clip_grad_norm_ (train.py:281): raises like torch does, at the next poll.  The
        kernels skip an update whose gradient norm is non-finite and COUNT it in a sticky device counter, so polling every
        k steps cannot miss one.  (The host-side step count, hence the LR schedule and AdamW's bias correction, has
        advanced past the skipped update: treat the error as fatal, as the reference does.)"""
        self.flush()
        s = self.stats[:4].tolist()
        if s[3] != 0.0 or s[1] != 0.0 or not math.isfinite(s[2]):
            self.stats[3] = 0.0
            raise RuntimeError(
                'The total norm of order 2.0 for gradients from `parameters` is non-finite, so it cannot be clipped. '
                f'(the fused step skipped {int(s[3]) or 1} update(s))')

    def state_dict(self):
        """optimizer + schedule (+ dropout stream) state for a true resume; the reference saves the model only
        (train.py:297-300), so a restarted run there silently restarts AdamW's moments and the LR schedule"""
        self._ensure_state(next(self.model.parameters()).device)
        self.flush()
        eng = self.model._engine
        return {'step': self.step_count, 'exp_avg': self.exp_avg.clone(), 'exp_avg_sq': self.exp_avg_sq.clone(),
                'dropout_counter': eng._seed_counter, 'dropout_base_seed': eng.base_seed,  # rank-independent
                'schedule': self.schedule, 'n_warmup': self.n_warmup, 'n_step': self.n_step, 'lr': self.lr,
                'weight_decay': self.wd, 'betas': tuple(self.betas), 'eps': self.eps, 'max_grad_norm': self.max_grad_norm,
                **({} if self.param_groups is None else {'param_groups': self._groups_state()}),
                **({} if self.ema is None else {'ema': self.ema.average(self.model).clone(), 'ema_decay': self.ema.decay,
                                                'ema_warmup': self.ema.warmup})}

    def _groups_state(self):
        """the groups as [(parameter names, lr_scale, weight_decay)]"""
        return [(names, g['lr_scale'], g['weight_decay']) for names, g in zip(self._group_names, self.param_groups)]

    def load_state_dict(self, sd):
        mine = None if self.param_groups is None else self._groups_state()
        theirs = sd.get('param_groups')
        theirs = None if theirs is None else [(tuple(n), float(s), None if w is None else float(w)) for n, s, w in theirs]
        if theirs != mine:
            raise ValueError('FusedTrainer.load_state_dict: the checkpoint\'s parameter groups differ from this '
                             'trainer\'s (build the trainer with the same param_groups)')
        if self.ema is not None:
            self.ema.check_inactive('load_state_dict()')
        self._ensure_state(next(self.model.parameters()).device)
        self._pending_step = None
        self.step_count = sd['step']
        self.exp_avg.copy_(sd['exp_avg'])
        self.exp_avg_sq.copy_(sd['exp_avg_sq'])
        eng = self.model._engine
        eng._seed_counter = sd.get('dropout_counter', eng._seed_counter)
        eng.base_seed = sd.get('dropout_base_seed', eng.base_seed)   # the rank offset stays this process's own
        for k, attr in (('schedule', 'schedule'), ('n_warmup', 'n_warmup'), ('n_step', 'n_step'), ('lr', 'lr'),
                        ('weight_decay', 'wd'), ('betas', 'betas'), ('eps', 'eps'), ('max_grad_norm', 'max_grad_norm')):
            if k in sd:
                setattr(self, attr, sd[k])
        if self.ema is not None:
            # a checkpoint without an average (written without EMA): the average starts from the loaded weights
            self.ema.load(self.model, sd.get('ema'))
            if 'ema_decay' in sd:
                self.ema.decay, self.ema.warmup = float(sd['ema_decay']), bool(sd['ema_warmup'])
        self.model.sync_shadow(force=True)

    # ---- the weight moving average -------------------------------------------------------------------------
    @contextlib.contextmanager
    def ema_weights(self):
        """Inside this context the model's weights (fp32 master and bf16 shadow) ARE the moving average: `model(...)`,
        `evaluate`, `Recorder`, `state_dict()` and `encoder_state_dict()` all see it; on exit the weights and the shadow
        are restored bit for bit.  A pending deferred update is applied first.  `step()` inside it and nesting it raise
        `RuntimeError`; without `ema_decay` it raises `ValueError`."""
        ema = self._require_ema()
        self._ensure_state(next(self.model.parameters()).device)
        self.flush()
        with ema.weights(self.model):
            yield

    def ema_state_dict(self):
        """the moving average in the model's own `state_dict()` keys (loads with strict=True into the model's class and
        into the oracle)"""
        ema = self._require_ema()
        self._ensure_state(next(self.model.parameters()).device)
        return ema.state_dict(self.model)

    def _require_ema(self):
        if self.ema is None:
            raise ValueError('the trainer keeps no weight moving average: build it with ema_decay=...')
        return self.ema


    # ---- the reference's outer loop (MyTrainer.train, train.py:263-319), re-hosted -------------------------------------
    def fit(self, train_data, eval_data=None, num_train_epoch=3, train_batch_size=64, eval_batch_size=None,
            do_eval=True, patience=8, save_every_n_epoch=0, output_dir=None, log_every=10, shuffle_seed=0,
            on_log=None, drop_last=False):
        """Epochs of fused steps with the control flow of `MyTrainer.train`: per epoch a shuffled pass over `train_data`
        (`(sample_values [n, C, L], labels [n, n_class])` host tensors -- what the reference's Dataset yields, stacked),
        then `evaluate` on `eval_data`, early stop after `patience` epochs without a better eval loss, a model checkpoint
        every `save_every_n_epoch` epochs and at the end (`model - <tag>.pt`, the reference's format) -- and, which the
        reference does not save, the trainer state next to it (`trainer - <tag>.pt`) so `resume()` restarts the schedule,
        AdamW's moments and the dropout stream where they stopped.

        Unlike the reference nothing here synchronises per step (it calls `.item()` and sklearn every step,
        train.py:278,287-290): batches are staged one step ahead on a copy stream, the loss of every `log_every`-th step
        is copied to pinned memory asynchronously and read one logging interval later; the non-finite check is polled at
        the same cadence.  Returns the list of log records."""
        from .metrics import evaluate
        x_all, y_all = train_data
        n = x_all.shape[0]
        bsz = train_batch_size
        steps_per_epoch = n // bsz if drop_last else (n + bsz - 1) // bsz
        logs, best_eval, n_bad = [], float('inf'), 0
        emit = on_log or (lambda rec: None)
        ring = [(torch.zeros(1).pin_memory(), torch.cuda.Event()) for _ in range(2)]
        pending = None   # (record, slot) whose loss is in flight
        gen = torch.Generator().manual_seed(shuffle_seed + self.step_count)

        def flush():
            nonlocal pending
            if pending is not None:
                rec, slot = pending
                ring[slot][1].synchronize()
                rec['train/loss'] = float(ring[slot][0])
                logs.append(rec)
                emit(rec)
                pending = None

        def batches(perm):
            for i in range(steps_per_epoch):
                idx = perm[i * bsz:(i + 1) * bsz]
                yield x_all[idx].pin_memory(), y_all[idx].pin_memory()

        for epoch in range(1, num_train_epoch + 1):
            self.model.train()
            perm = torch.randperm(n, generator=gen)
            it = batches(perm)
            staged = None
            for i in range(steps_per_epoch):
                if staged is None:
                    staged = self.stage(*next(it))
                xd, yd = staged
                if xd.shape[0] != bsz and self.use_cuda_graph:
                    # the ragged last batch has its own shape: run it outside the captured graph
                    self.use_cuda_graph, saved = False, True
                else:
                    saved = False
                loss, _ = self.step(xd, yd)
                if saved:
                    self.use_cuda_graph = True
                staged = self.stage(*next(it)) if i + 1 < steps_per_epoch else None
                if self.step_count % log_every == 0 or i + 1 == steps_per_epoch:
                    flush()
                    slot = (self.step_count // max(1, log_every)) & 1
                    ring[slot][0].copy_(loss.reshape(1), non_blocking=True)
                    ring[slot][1].record()
                    pending = ({'epoch': epoch, 'step': self.step_count, 'train/learning_rate': self.current_lr()}, slot)
                    self.check_finite()
            flush()
            tag = f'ep{epoch}'
            if output_dir and save_every_n_epoch and epoch % save_every_n_epoch == 0:
                self.save(output_dir, tag)
            if do_eval and eval_data is not None:
                ebsz = eval_batch_size or bsz
                xe, ye = eval_data
                batches_eval = lambda: ({'sample_values': xe[j:j + ebsz], 'labels': ye[j:j + ebsz]}
                                        for j in range(0, xe.shape[0], ebsz))
                d = evaluate(self.model, batches_eval())
                rec = dict(epoch=epoch, step=self.step_count, **d)
                if self.ema is not None:   # the moving average next to the weights; patience watches eval/loss
                    with self.ema_weights():
                        d_ema = evaluate(self.model, batches_eval())
                    rec.update({'eval_ema/' + k[len('eval/'):]: v for k, v in d_ema.items()})
                logs.append(rec)
                emit(rec)
                if d['eval/loss'] < best_eval:   # train.py:304-314
                    best_eval, n_bad = d['eval/loss'], 0
                else:
                    n_bad += 1
                if n_bad >= patience:
                    logs.append({'epoch': epoch, 'early_stop': True, 'patience': patience, 'best_eval_loss': best_eval})
                    break
        if output_dir:
            self.save(output_dir, 'final')
        return logs

    def save(self, output_dir, tag):
        """`model - <tag>.pt` = `model.state_dict()` as the reference saves it (train.py:297-300,319; loadable by its
        `load_trained`), `trainer - <tag>.pt` = optimizer / schedule / dropout-stream state (and the moving average),
        with EMA `model_ema - <tag>.pt` = `ema_state_dict()` in the format of `model - <tag>.pt`"""
        if self.ema is not None:
            self.ema.check_inactive('save()')
        os.makedirs(output_dir, exist_ok=True)
        torch.cuda.synchronize()
        torch.save(self.model.state_dict(), os.path.join(output_dir, f'model - {tag}.pt'))
        torch.save(self.state_dict(), os.path.join(output_dir, f'trainer - {tag}.pt'))
        if self.ema is not None:
            torch.save(self.ema_state_dict(), os.path.join(output_dir, f'model_ema - {tag}.pt'))

    def resume(self, output_dir, tag):
        self.model.load_state_dict(torch.load(os.path.join(output_dir, f'model - {tag}.pt'), map_location='cpu'), strict=True)
        self.load_state_dict(torch.load(os.path.join(output_dir, f'trainer - {tag}.pt'), map_location='cpu'))




def fused_train_step(model, batch, lr=3e-4, **trainer_kwargs):
    """One `zero_grad -> forward -> backward -> clip -> AdamW -> scheduler` step (train.py:271-283) on a batch dict as
    the reference's DataLoader yields it (`sample_values`, `labels`); the `FusedTrainer` behind it is created on first
    use and kept per model.  Returns `ModelOutput(loss, logits)` (device tensors, valid until the next step)."""
    from .model import ModelOutput
    tr = getattr(model, '_fused_trainer', None)   # kept ON the model (a collectable cycle), not in a global registry
    if tr is None:
        tr = FusedTrainer(model, learning_rate=lr, **trainer_kwargs)
        object.__setattr__(model, '_fused_trainer', tr)
    tr.lr = lr
    loss, logits = tr.step(batch['sample_values'].cuda(non_blocking=True), batch['labels'].cuda(non_blocking=True))
    return ModelOutput(loss=loss, logits=logits)
