"""GPU tier: the weight moving average updated inside the AdamW kernel (ema_decay).  The kernel against the plain and
grouped AdamW and an fp64 reference, the fused trainer and the autograd loop against the oracle plus a reference EMA, the
deferred optimizer, frozen tensors, the bf16 bench geometry, the swap context, save / resume, fit and the MAE encoder."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

from conftest import GOLDEN_CFG
from ecg_b200 import (EcgVit, EcgVitConfig, EcgVitForMaskedAutoencoding, FusedAdamW, FusedTrainer, _lib,
                      clip_grad_norm_, param_groups_lrd)
from ecg_b200.optim import group_table
from oracle.ecg_vit_oracle import OracleTrainer, lr_lambda, synthetic_batch

from test_gpu_parity import rel, FP32_TOL
from test_gpu_pretrain import BENCH
from test_gpu_frozen import CFG3, MAE_DEC, make_pair

LIB = None


def lib():
    global LIB
    LIB = LIB or _lib.load()
    return LIB


# ---- 1. the kernel ---------------------------------------------------------------------------------------------------
N = 64 * 4099   # a whole number of 64-element blocks, not of the grid


def buffers(grad_dtype, seed=0):
    gen = torch.Generator(device='cuda').manual_seed(seed)
    r = lambda: torch.randn(N, device='cuda', generator=gen)
    p, g, ema = r(), r() * 1e-2, r()
    m = r() * 1e-3
    v = r().abs() * 1e-5
    return dict(p=p, m=m, v=v, g=g.to(grad_dtype), ema=ema, shadow=p.bfloat16())


def gmap_table(n_groups=3):
    gm = torch.randint(0, n_groups, (N // 64,), generator=torch.Generator().manual_seed(1), dtype=torch.uint8)
    gm[::7] = 255
    table = torch.tensor(group_table([1e-3, 5e-4, 2e-3][:n_groups], [0.05, 0.0, 0.1][:n_groups], 0.9, 3),
                         dtype=torch.float32)
    return gm.cuda(), table.cuda()


def hyper(rate, skip=False, max_norm=1.0):
    return torch.tensor(_lib.adamw_hyper(1e-3, 0.9, 0.999, 1e-8, 0.05, 3, max_norm, 1.0, skip=skip, ema_rate=rate),
                        dtype=torch.float32, device='cuda')


def stats_with_norm(sumsq):
    s = torch.zeros(_lib.STATS_FLOATS, device='cuda')
    s[0] = sumsq
    return s


def launch(b, hyp, st, shadow, grouped, lo, n, flags, ema=True, gm=None, gt=None):
    code = _lib.F32 if b['g'].dtype == torch.float32 else _lib.BF16
    esz = b['g'].element_size()
    args = (b['p'].data_ptr() + 4 * lo, b['m'].data_ptr() + 4 * lo, b['v'].data_ptr() + 4 * lo,
            b['g'].data_ptr() + esz * lo, code, b['shadow'].data_ptr() + 2 * lo if shadow else None)
    gmp = gm.data_ptr() + lo // 64 if grouped else None
    s = torch.cuda.current_stream().cuda_stream
    if ema:
        return lib().ecgvit_adamw_step_ema(*args, b['ema'].data_ptr() + 4 * lo, n, gmp, gt.data_ptr() if grouped else None,
                                           hyp.data_ptr(), st.data_ptr(), flags, s)
    if grouped:
        return lib().ecgvit_adamw_step_grouped(*args, n, gmp, gt.data_ptr(), hyp.data_ptr(), st.data_ptr(), flags, s)
    return lib().ecgvit_adamw_step(*args, n, hyp.data_ptr(), st.data_ptr(), flags, s)


SLICES = {'whole': [(0, N, 0)],
          'slices': [(0, 64 * 1000, _lib.ADAMW_SLICE | _lib.ADAMW_FIRST_SLICE), (64 * 1000, N - 64 * 1000, _lib.ADAMW_SLICE)]}


@pytest.mark.parametrize('slicing', ['whole', 'slices'])
@pytest.mark.parametrize('grouped', [False, True])
@pytest.mark.parametrize('shadow', [False, True])
@pytest.mark.parametrize('grad_dtype', [torch.float32, torch.bfloat16])
def test_kernel_matches_adamw_and_fp64_ema(grad_dtype, shadow, grouped, slicing):
    rate = 1.0 - 0.9999
    hyp, gm_gt = hyper(rate), gmap_table()
    gm, gt = gm_gt
    ref, out, again = buffers(grad_dtype), buffers(grad_dtype), buffers(grad_dtype)
    ema0 = out['ema'].clone()
    st_ref, st_out, st_again = stats_with_norm(4.0), stats_with_norm(4.0), stats_with_norm(4.0)   # norm 2: the clip acts
    for lo, n, flags in SLICES[slicing]:
        assert launch(ref, hyp, st_ref, shadow, grouped, lo, n, flags, ema=False, gm=gm, gt=gt) == 0
        assert launch(out, hyp, st_out, shadow, grouped, lo, n, flags, gm=gm, gt=gt) == 0
        assert launch(again, hyp, st_again, shadow, grouped, lo, n, flags, gm=gm, gt=gt) == 0
    torch.cuda.synchronize()
    for k in ('p', 'm', 'v', 'shadow'):
        assert torch.equal(out[k], ref[k]), k
    assert torch.equal(st_out[:4], st_ref[:4])
    for k in out:
        assert torch.equal(out[k], again[k]), k          # a second launch is bit-identical
    # fp64 reference from the kernel's own p_new and the fp32 rate it reads
    r = float(torch.tensor(rate, dtype=torch.float32))
    e0, pn = ema0.double(), out['p'].double()
    want = e0 + r * (pn - e0)
    bound = 2.0 ** -23 * (want.abs() + (pn - e0).abs())
    touched = torch.ones(N, dtype=torch.bool, device='cuda')
    if grouped:
        touched = (gm != 255).repeat_interleave(64)
        assert torch.equal(out['ema'][~touched], ema0[~touched])     # id 255: untouched
    err = (out['ema'].double() - want).abs()
    assert bool((err[touched] <= bound[touched]).all()), float((err - bound)[touched].max())
    assert not torch.equal(out['ema'], ema0)


@pytest.mark.parametrize('why', ['skip', 'nonfinite'])
def test_skipped_update_leaves_the_ema_untouched(why):
    b = buffers(torch.float32)
    before = {k: v.clone() for k, v in b.items()}
    hyp = hyper(0.5, skip=why == 'skip')
    st = stats_with_norm(float('inf') if why == 'nonfinite' else 4.0)
    assert launch(b, hyp, st, True, False, 0, N, 0) == 0
    torch.cuda.synchronize()
    for k in b:
        assert torch.equal(b[k], before[k]), k
    assert float(st[3]) == (1.0 if why == 'nonfinite' else 0.0)


def test_rejections_write_nothing():
    b = buffers(torch.float32)
    gm, gt = gmap_table()
    before = {k: v.clone() for k, v in b.items()}
    hyp, st = hyper(0.5), stats_with_norm(4.0)
    s = torch.cuda.current_stream().cuda_stream
    P = lambda k, off=0: b[k].data_ptr() + off
    base = [P('p'), P('m'), P('v'), P('g'), _lib.F32, P('shadow'), P('ema'), N, None, None, hyp.data_ptr(),
            st.data_ptr(), 0, s]
    bad = [dict({6: None}),                                # no average
           dict({6: P('ema', 4)}),                         # misaligned average
           dict({0: P('p', 4)}),                           # misaligned weights
           dict({7: N - 2}),                               # n % 4
           dict({8: gm.data_ptr(), 7: N - 4, 9: gt.data_ptr()}),   # n % 64 with a map
           dict({8: gm.data_ptr()}),                       # a map without a table
           dict({4: 7}),                                   # unknown gradient dtype
           dict({7: 0})]
    for change in bad:
        args = list(base)
        for i, v in change.items():
            args[i] = v
        assert lib().ecgvit_adamw_step_ema(*args) != 0, change
        assert 'adamw_step_ema' in _lib.last_error()
    # n % 64 is required only with a map
    torch.cuda.synchronize()
    for k in b:
        assert torch.equal(b[k], before[k]), k
    args = list(base)
    args[7] = N - 4
    assert lib().ecgvit_adamw_step_ema(*args) == 0
    assert lib().ecgvit_swap_f32_cast(P('p', 4), P('ema'), None, 8, s) != 0


@pytest.mark.parametrize('shadow', [False, True])
def test_swap_kernel_exchanges_and_recasts(shadow):
    for n in (N, 1001):
        b = buffers(torch.float32)
        p0, e0 = b['p'].clone(), b['ema'].clone()
        sh0 = b['shadow'].clone()
        s = torch.cuda.current_stream().cuda_stream
        assert lib().ecgvit_swap_f32_cast(b['p'].data_ptr(), b['ema'].data_ptr(), b['shadow'].data_ptr() if shadow else None,
                                          n, s) == 0
        torch.cuda.synchronize()
        assert torch.equal(b['p'][:n], e0[:n]) and torch.equal(b['ema'][:n], p0[:n])
        assert torch.equal(b['p'][n:], p0[n:]) and torch.equal(b['ema'][n:], e0[n:])
        if shadow:
            assert torch.equal(b['shadow'][:n], e0[:n].bfloat16()) and torch.equal(b['shadow'][n:], sh0[n:])
        assert lib().ecgvit_swap_f32_cast(b['p'].data_ptr(), b['ema'].data_ptr(), b['shadow'].data_ptr() if shadow else None,
                                          n, s) == 0
        torch.cuda.synchronize()
        assert torch.equal(b['p'], p0) and torch.equal(b['ema'], e0) and torch.equal(b['shadow'], sh0)


# ---- 2. the fused trainer against the oracle -------------------------------------------------------------------------
def oracle_ema_step(ema_ref, oracle, decay, t):
    with torch.no_grad():
        for name, q in oracle.named_parameters():
            if q.requires_grad:
                ema_ref[name].lerp_(q.detach(), 1.0 - decay.decay_at(t))


def run_trainer_vs_oracle(mode, warmup, pattern='none', steps=3):
    oracle, model, x, y = make_pair(CFG3, pattern)
    kw = dict(learning_rate=1e-3, weight_decay=1e-2, schedule='cosine', n_warmup=1, n_step=3, max_grad_norm=0.05)
    tr = FusedTrainer(model, use_cuda_graph=mode == 'graph', data_parallel=False, ema_decay=0.9, ema_warmup=warmup, **kw)
    ot = OracleTrainer(oracle, **kw)
    ema_ref = {n: q.detach().clone() for n, q in oracle.named_parameters()}
    for t in range(1, steps + 1):
        _, _, o_norm = ot.step(x, y)
        tr.step(x.cuda(), y.cuda())
        assert float(o_norm) > 0.05, 'test must exercise the clip'
        oracle_ema_step(ema_ref, oracle, tr.ema, t)
    tr.check_finite()
    return tr, ema_ref


@pytest.mark.parametrize('warmup', [False, True])
def test_trainer_ema_tracks_the_oracle_eager_and_captured(warmup):
    out = {}
    for mode in ('eager', 'graph'):
        tr, ema_ref = run_trainer_vs_oracle(mode, warmup)
        sd = tr.ema_state_dict()
        for k, v in ema_ref.items():
            assert rel(sd[k], v) < FP32_TOL, (mode, k, rel(sd[k], v))
        out[mode] = tr.ema.buf.clone()   # (a capture warm-up counted as an update would break the parity above)
    assert rel(out['graph'], out['eager']) < FP32_TOL


@pytest.mark.parametrize('pattern', ['last', 'qkv', 'lrd'])
def test_frozen_slots_of_the_ema_stay_put(pattern):
    oracle, model, x, y = make_pair(CFG3, 'prefix' if pattern == 'lrd' else pattern)
    groups = param_groups_lrd(model) if pattern == 'lrd' else None
    tr = FusedTrainer(model, learning_rate=1e-3, data_parallel=False, param_groups=groups, ema_decay=0.5,
                      use_cuda_graph=True)
    start = {n: p.detach().reshape(-1).clone() for n, p in model.named_parameters()}
    for _ in range(3):
        tr.step(x.cuda(), y.cuda())
    torch.cuda.synchronize()
    params = dict(model.named_parameters())
    moved = 0
    for o, n, _, name in model._layout.values():
        if params[name].requires_grad:
            moved += not torch.equal(tr.ema.buf[o:o + n], start[name])
        else:
            assert torch.equal(tr.ema.buf[o:o + n], start[name]), name
    assert moved > 0


def test_deferred_optimizer_ema_is_final_after_flush():
    kw = dict(learning_rate=1e-3, weight_decay=1e-2, schedule='cosine', n_warmup=1, n_step=6, max_grad_norm=0.05,
              data_parallel=False, ema_decay=0.8, ema_warmup=True)
    _, m_now, x, y = make_pair(CFG3, 'none')
    _, m_def, _, _ = make_pair(CFG3, 'none')
    t_now, t_def = FusedTrainer(m_now, **kw), FusedTrainer(m_def, defer_optimizer=True, **kw)
    xd, yd = x.cuda(), y.cuda()
    for _ in range(4):
        t_now.step(xd, yd)
        t_def.step(xd, yd)
    assert t_def._pending_step == 4
    # the pending update applied slice by slice (flush) == the same update applied in one call, bit for bit
    state = lambda: [m_def._flat_p, t_def.exp_avg, t_def.exp_avg_sq, t_def.ema.buf, t_def.stats, m_def._flat_g]
    saved = [b.clone() for b in state()]
    t_def.flush()
    sliced = [b.clone() for b in state()]
    for b, s in zip(state(), saved):
        b.copy_(s)
    t_def._hyper_ring.upload(t_def.hyper[:16], t_def._hyper_values(4))
    t_def._adamw(m_def._flat_p.data_ptr(), t_def.exp_avg.data_ptr(), t_def.exp_avg_sq.data_ptr(),
                 m_def._flat_g.data_ptr(), _lib.F32, None, 0, m_def._flat_p.numel(), 0,
                 torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    for a, b in zip(sliced[:4], state()[:4]):
        assert torch.equal(a, b)
    # and the deferred run is the immediate run
    assert rel(t_def.ema.buf, t_now.ema.buf) < 1e-6 and rel(m_def._flat_p, m_now._flat_p) < 1e-6


def test_bf16_bench_geometry_ema_follows_its_fp64_recomputation():
    torch.manual_seed(3)
    model = EcgVit(config=EcgVitConfig(compute_dtype='bf16', **dict(BENCH, hidden_dropout_prob=0.1))).cuda().train()
    x, y = synthetic_batch(32, seed=3)
    tr = FusedTrainer(model, learning_rate=1e-3, use_cuda_graph=True, data_parallel=False, ema_decay=0.9999,
                      ema_warmup=True)
    model._prepare(x.cuda().device)
    want = model._flat_p.double()          # the average starts as the weights of the first step
    bound = torch.zeros_like(want)
    for t in range(1, 5):
        tr.step(x.cuda(), y.cuda())
        torch.cuda.synchronize()
        p = model._flat_p.double()
        r = float(torch.tensor(tr.ema.rate(t), dtype=torch.float32))
        bound += 2.0 ** -23 * (want.abs() + (p - want).abs())   # one rounding of p - ema and one of the fma per step
        want = want + r * (p - want)
        err = (tr.ema.buf.double() - want).abs()
        assert bool((err <= bound).all()), (t, float((err - bound).max()))
    assert not torch.equal(tr.ema.buf, model._flat_p)
    tr.check_finite()


# ---- 3. the swap context --------------------------------------------------------------------------------------------
@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
def test_ema_weights_context(dtype):
    torch.manual_seed(4)
    cfg = dict(GOLDEN_CFG, hidden_dropout_prob=0.1)
    model = EcgVit(config=EcgVitConfig(compute_dtype=dtype, **cfg)).cuda().train()
    x, y = synthetic_batch(8, length=cfg['max_signal_length'], seed=4)
    tr = FusedTrainer(model, learning_rate=1e-2, data_parallel=False, ema_decay=0.5)
    for _ in range(3):
        tr.step(x.cuda(), y.cuda())
    torch.cuda.synchronize()
    p0 = model._flat_p.clone()
    sh0 = None if model._shadow is None else model._shadow.clone()
    esd = tr.ema_state_dict()
    fresh = EcgVit(config=EcgVitConfig(compute_dtype=dtype, **cfg))
    fresh.load_state_dict(esd, strict=True)
    fresh.cuda().eval()
    model.eval()
    with tr.ema_weights():
        inside = model(x.cuda(), y.cuda()).logits
        sd_inside = model.state_dict()
        for k in esd:
            assert torch.equal(sd_inside[k], esd[k]), k
        with pytest.raises(RuntimeError):
            tr.step(x.cuda(), y.cuda())
        with pytest.raises(RuntimeError):
            with tr.ema_weights():
                pass
    assert torch.equal(inside, fresh(x.cuda(), y.cuda()).logits)
    assert torch.equal(model._flat_p, p0)
    if sh0 is not None:
        assert torch.equal(model._shadow, sh0)
    assert not torch.equal(inside, model(x.cuda(), y.cuda()).logits)


# ---- 4. save / resume, fit -----------------------------------------------------------------------------------------
def test_save_resume_reproduces_the_uninterrupted_ema(tmp_path):
    kw = dict(learning_rate=1e-3, schedule='cosine', n_warmup=1, n_step=4, data_parallel=False, ema_decay=0.7,
              ema_warmup=True)
    oracle, m_ref, x, y = make_pair(CFG3, 'none')
    _, m_a, _, _ = make_pair(CFG3, 'none')
    t_ref, t_a = FusedTrainer(m_ref, **kw), FusedTrainer(m_a, **kw)
    xs, ys = x.cuda(), y.cuda()
    for _ in range(4):
        t_ref.step(xs, ys)
    for _ in range(2):
        t_a.step(xs, ys)
    t_a.save(str(tmp_path), 'mid')
    _, m_b, _, _ = make_pair(CFG3, 'none', seed=99)
    t_b = FusedTrainer(m_b, **dict(kw, ema_decay=0.3, ema_warmup=False))
    t_b.resume(str(tmp_path), 'mid')
    assert (t_b.ema.decay, t_b.ema.warmup) == (0.7, True)
    for _ in range(2):
        t_b.step(xs, ys)
    assert rel(t_b.ema.buf, t_ref.ema.buf) < 1e-5
    ema_file = torch.load(os.path.join(str(tmp_path), 'model_ema - mid.pt'))
    EcgVit(config=EcgVitConfig(compute_dtype='fp32', **CFG3)).load_state_dict(ema_file, strict=True)
    oracle.load_state_dict(ema_file, strict=True)
    # a checkpoint written without EMA: the average starts from the loaded weights; a trainer without EMA ignores it
    t_plain = FusedTrainer(m_b, **dict(kw, ema_decay=None, ema_warmup=False))
    sd_plain = t_plain.state_dict()
    assert 'ema' not in sd_plain
    t_b.load_state_dict(sd_plain)
    assert torch.equal(t_b.ema.buf, m_b._flat_p)
    t_plain.load_state_dict(t_b.state_dict())


def test_fit_logs_eval_ema(tmp_path):
    torch.manual_seed(5)
    model = EcgVit(config=EcgVitConfig(compute_dtype='bf16', **GOLDEN_CFG)).cuda()
    x, y = synthetic_batch(40, length=GOLDEN_CFG['max_signal_length'], seed=5)
    tr = FusedTrainer(model, learning_rate=1e-3, data_parallel=False, ema_decay=0.9, ema_warmup=True)
    logs = tr.fit((x, y), (x[:16], y[:16]), num_train_epoch=2, train_batch_size=8, output_dir=str(tmp_path))
    evals = [r for r in logs if 'eval/loss' in r]
    assert len(evals) == 2
    for r in evals:
        assert 'eval_ema/loss' in r and 'eval_ema/macro_auc' in r and r['eval_ema/loss'] != r['eval/loss']
    assert os.path.exists(os.path.join(str(tmp_path), 'model_ema - final.pt'))


# ---- 5. the autograd loop ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('groups', [False, True])
def test_fused_adamw_ema_against_torch_adamw(groups):
    oracle, model, x, y = make_pair(CFG3, 'none')
    sched = lambda s: lr_lambda('cosine', s, 1, 3)
    g = param_groups_lrd(model, weight_decay=0.05, layer_decay=0.75) if groups else None
    make = lambda: FusedAdamW(model, lr=2e-3, weight_decay=1e-2, param_groups=g, ema_decay=0.8, ema_warmup=True)
    opt = make()
    if groups:
        names = {id(p): n for n, p in model.named_parameters()}
        op = dict(oracle.named_parameters())
        oopt = torch.optim.AdamW([{'params': [op[names[id(p)]] for p in gg['params']], 'lr': 2e-3 * gg['lr_scale'],
                                   'weight_decay': gg['weight_decay']} for gg in g], lr=2e-3)
    else:
        oopt = torch.optim.AdamW(oracle.parameters(), lr=2e-3, weight_decay=1e-2)
    s1, s2 = torch.optim.lr_scheduler.LambdaLR(opt, sched), torch.optim.lr_scheduler.LambdaLR(oopt, sched)
    ema_ref = {n: q.detach().clone() for n, q in oracle.named_parameters()}
    for t in range(1, 4):
        opt.zero_grad()
        model(x.cuda(), y.cuda()).loss.backward()
        clip_grad_norm_(model, max_norm=0.05)
        oopt.zero_grad()
        oracle(x, y).loss.backward()
        torch.nn.utils.clip_grad_norm_(oracle.parameters(), max_norm=0.05)
        opt.step()
        oopt.step()
        s1.step()
        s2.step()
        oracle_ema_step(ema_ref, oracle, opt.ema, t)
    sd = opt.ema_state_dict()
    for k, v in ema_ref.items():
        assert rel(sd[k], v) < FP32_TOL, (k, rel(sd[k], v))
    flat = opt.state_dict()['flat']['ema']
    assert torch.equal(flat, opt.ema.buf)
    with opt.ema_weights():
        assert torch.equal(model._flat_p, flat)
        with pytest.raises(RuntimeError):
            opt.step()
    opt2 = make()
    opt2.load_state_dict(opt.state_dict())
    assert torch.equal(opt2.ema.buf, flat)


# ---- 6. pre-training ------------------------------------------------------------------------------------------------
def test_mae_ema_encoder_loads_into_a_mean_pooled_classifier():
    cfg = dict(GOLDEN_CFG, num_hidden_layers=3)
    torch.manual_seed(9)
    pre = EcgVitForMaskedAutoencoding(EcgVitConfig(compute_dtype='bf16', **cfg), **MAE_DEC).cuda().train()
    x, _ = synthetic_batch(8, length=cfg['max_signal_length'], seed=9)
    tr = FusedTrainer(pre, learning_rate=1e-3, use_cuda_graph=True, ema_decay=0.5)
    for _ in range(3):
        tr.step(x.cuda())
    torch.cuda.synchronize()
    with tr.ema_weights():
        enc = {k: v.detach().clone() for k, v in pre.encoder_state_dict().items()}
    esd = tr.ema_state_dict()
    for k, v in enc.items():
        assert torch.equal(v, esd[k]), k
    assert not torch.equal(tr.ema.buf, pre._flat_p)
    probe = EcgVit(config=EcgVitConfig(compute_dtype='bf16', pool='mean', **cfg))
    missing = probe.load_state_dict(enc, strict=False).missing_keys
    assert missing and all(k.startswith('vit.mlp_head.') for k in missing)
    pre.load_state_dict(esd, strict=True)
