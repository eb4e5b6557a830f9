"""CPU tier: the weight moving average (ema_decay) -- the decay schedule, hyper[15] as the trainer fills it (double-precision
1 - d_t, skip, the deferred pending step), the rejections, the entry points each configuration selects (and that
ema_decay=None selects today's), the checkpoint keys, the context's guards, and the new C prototypes."""
import os
import types

import numpy as np
import pytest
import torch

from conftest import GOLDEN_CFG, ROOT
from ecg_b200 import EcgVit, EcgVitConfig, FusedAdamW, FusedTrainer, _lib
from ecg_b200.optim import WeightEma

TODAY_KEYS = {'step', 'exp_avg', 'exp_avg_sq', 'dropout_counter', 'dropout_base_seed', 'schedule', 'n_warmup', 'n_step',
              'lr', 'weight_decay', 'betas', 'eps', 'max_grad_norm'}


def model_cpu():
    torch.manual_seed(0)
    return EcgVit(config=EcgVitConfig(compute_dtype='fp32', **GOLDEN_CFG))


def trainer(model=None, **kw):
    """a trainer over host stand-ins of the flat buffers (nothing here touches a device)"""
    model = model or model_cpu()
    tr = FusedTrainer(model, data_parallel=False, **kw)
    model._layout, total = model._flat_layout()
    model._flat_p = torch.zeros(total)
    tr._flat_ptr = model._flat_p.data_ptr()
    return tr


def test_decay_at_constant_and_warmup():
    const = WeightEma(0.9999)
    assert [const.decay_at(t) for t in (1, 10, 10 ** 6)] == [0.9999] * 3
    warm = WeightEma(0.9999, warmup=True)
    for t in (1, 2, 10, 100, 1000, 89990, 89991, 10 ** 6):
        assert warm.decay_at(t) == min(0.9999, (1.0 + t) / (10.0 + t)), t
    assert warm.decay_at(1) == 2.0 / 11.0
    assert warm.decay_at(89991) == 0.9999   # (1 + t) / (10 + t) reaches 0.9999 at t = 89 990
    # the rate is 1 - d_t in double precision; 1 - fp32(d) in fp32 would be 1.7e-4 off relative at d = 0.9999
    assert const.rate(5) == 1.0 - 0.9999
    f32 = float(np.float32(1.0) - np.float32(0.9999))
    assert abs(f32 - (1.0 - 0.9999)) / (1.0 - 0.9999) > 1e-4
    assert abs(float(np.float32(const.rate(5))) - (1.0 - 0.9999)) / (1.0 - 0.9999) < 1e-7


def test_hyper_slot_15_from_the_trainer(monkeypatch):
    tr = trainer(ema_decay=0.999, ema_warmup=True)
    ema = tr.ema
    for t in (1, 2, 50, 5000):
        vals = tr._hyper_values(t)
        assert len(vals) == 16 and vals[14] == 0.0
        assert vals[15] == 1.0 - min(0.999, (1.0 + t) / (10.0 + t)) == ema.rate(t)
    skip = tr._hyper_values(None)
    assert skip[14] == 1.0 and skip[15] == 0.0
    # grouped: the group table stays behind slot 15
    tr._grouped = True
    assert len(tr._hyper_values(3)) == 18 and tr._hyper_values(3)[15] == ema.rate(3)
    tr._grouped = False

    uploaded = []

    class Ring:
        def __init__(self, n, dtype):
            self.bufs = [torch.empty(n, dtype=dtype)]

        def upload(self, dst, vals):
            uploaded.append(list(vals))

    monkeypatch.setattr(_lib, 'PinnedRing', Ring)
    tr.hyper = torch.zeros(16)
    tr.step_count = 6
    tr._upload_hyper()                         # immediate: this step applies update 7
    assert uploaded[-1][15] == ema.rate(7)
    tr.defer_optimizer, tr._pending_step = True, 6
    tr._upload_hyper()                         # deferred: the pending update 6 (the forward of step 7 runs beside it)
    assert uploaded[-1][15] == ema.rate(6)
    tr._pending_step = None
    tr._upload_hyper()                         # nothing pending: skip
    assert uploaded[-1][14] == 1.0


def test_hyper_slot_15_is_zero_without_ema():
    tr = trainer()
    assert tr.ema is None and tr._hyper_values(4)[15] == 0.0
    assert tr._hyper_values(4) == _lib.adamw_hyper(tr.lr, 0.9, 0.999, 1e-8, tr.wd, 4, 1.0, 1.0)


@pytest.mark.parametrize('front', ['trainer', 'adamw'])
def test_rejections(front):
    make = (lambda **kw: FusedTrainer(model_cpu(), **kw)) if front == 'trainer' else \
        (lambda **kw: FusedAdamW(model_cpu(), **kw))
    for bad in (0.0, 1.0, -0.5, 1.5, float('nan')):
        with pytest.raises(ValueError, match='ema_decay'):
            make(ema_decay=bad)
    with pytest.raises(ValueError, match='ema_warmup'):
        make(ema_warmup=True)
    plain = make()
    assert plain.ema is None
    with pytest.raises(ValueError, match='ema_decay'):
        with plain.ema_weights():
            pass
    with pytest.raises(ValueError, match='ema_decay'):
        plain.ema_state_dict()
    assert make(ema_decay=0.5).ema.decay == 0.5


class FakeLib:
    """records the entry point and arguments of every call"""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def fn(*args):
            self.calls.append((name, args))
            return 0
        return fn


@pytest.mark.parametrize('grouped', [False, True])
@pytest.mark.parametrize('ema', [None, 0.99])
def test_adamw_entry_point_selection(ema, grouped):
    tr = trainer(ema_decay=ema)
    tr.lib = FakeLib()
    tr.hyper, tr.stats = torch.zeros(18), torch.zeros(_lib.STATS_FLOATS)
    tr._grouped = grouped
    tr._gmap = torch.zeros(1000, dtype=torch.uint8)
    if ema is not None:
        tr.ema.buf = torch.zeros(tr.model._flat_p.numel())
    lo, n = 128, 640
    tr._adamw(1 << 20, 2 << 20, 3 << 20, 4 << 20, _lib.F32, None, lo, n, _lib.ADAMW_SLICE, None)
    (name, args), = tr.lib.calls
    if ema is None:
        assert name == ('ecgvit_adamw_step_grouped' if grouped else 'ecgvit_adamw_step')
        return
    assert name == 'ecgvit_adamw_step_ema'
    p, m, v, g, code, shadow, e, count, gm, gt, hyper, stats, flags, _ = args
    # the average is offset by lo exactly like p, m and v
    assert (p, m, v, g) == ((1 << 20) + 4 * lo, (2 << 20) + 4 * lo, (3 << 20) + 4 * lo, (4 << 20) + 4 * lo)
    assert e == tr.ema.buf.data_ptr() + 4 * lo and count == n and flags == _lib.ADAMW_SLICE
    if grouped:
        assert gm == tr._gmap.data_ptr() + lo // 64 and gt == tr.hyper.data_ptr() + 64
    else:
        assert gm is None and gt is None


def _fake_engine(model):
    model._engine = types.SimpleNamespace(_seed_counter=3, base_seed=5)


def test_state_dict_keys_with_and_without_ema():
    for kw, extra in (({}, set()), (dict(ema_decay=0.99, ema_warmup=True), {'ema', 'ema_decay', 'ema_warmup'})):
        tr = trainer(**kw)
        _fake_engine(tr.model)
        tr._ensure_state = lambda device: None
        tr.exp_avg = tr.exp_avg_sq = torch.zeros(tr.model._flat_p.numel())
        if tr.ema is not None:
            tr.ema.ensure(tr.model._flat_p)
        sd = tr.state_dict()
        assert set(sd) == TODAY_KEYS | extra
        if extra:
            assert sd['ema_decay'] == 0.99 and sd['ema_warmup'] is True and sd['ema'].shape == tr.model._flat_p.shape
    for kw, flat in (({}, {'step', 'exp_avg', 'exp_avg_sq'}), (dict(ema_decay=0.9), {'step', 'exp_avg', 'exp_avg_sq', 'ema'})):
        assert set(FusedAdamW(model_cpu(), **kw).state_dict()['flat']) == flat


def test_context_guards_nesting_and_step():
    model = model_cpu()
    tr = FusedTrainer(model, ema_decay=0.9, data_parallel=False)
    ema = tr.ema
    with ema.weights(model):    # before the first step there is nothing to swap, the guards hold all the same
        assert ema.active and not ema.swapped
        with pytest.raises(RuntimeError, match='nest'):
            with ema.weights(model):
                pass
        with pytest.raises(RuntimeError, match='step'):
            tr.step(torch.zeros(1, 12, 500), torch.zeros(1, 71))
        with pytest.raises(RuntimeError, match='save'):
            tr.save('unused', 'x')
    assert not ema.active
    opt = FusedAdamW(model, ema_decay=0.9)
    with opt.ema.weights(model):
        with pytest.raises(RuntimeError, match='step'):
            opt.step()


def test_new_prototypes_in_header_and_ctypes_table():
    src = open(os.path.join(ROOT, 'include', 'ecgvit_b200.h')).read()
    for name in ('ecgvit_adamw_step_ema', 'ecgvit_swap_f32_cast'):
        assert f'int {name}(' in src and name in _lib.SIGNATURES
    assert '[15] 1 - d_t' in src
    assert _lib.SIGNATURES['ecgvit_adamw_step_ema'][6] is _lib.c_void_p        # ema sits after the shadow
    assert _lib.SIGNATURES['ecgvit_adamw_step_ema'][7] is _lib.c_int64         # then n
