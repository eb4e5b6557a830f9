"""GPU tier: fine-tuning support -- the grouped AdamW kernel against torch.optim.AdamW, FusedAdamW / FusedTrainer with
parameter groups against the CPU oracle trainer with the same groups, and the mean-pooled classification head
(pool='mean') forward and backward against the oracle."""
import pytest
import torch
from torch import nn

pytestmark = pytest.mark.gpu

from conftest import GOLDEN_CFG
from ecg_b200 import (EcgVit, EcgVitConfig, EcgVitForMaskedAutoencoding, FusedAdamW, FusedTrainer, param_groups_lrd,
                      _lib)
from oracle.ecg_vit_oracle import OracleConfig, OracleEcgVit, OracleTrainer, lr_lambda, synthetic_batch

from test_gpu_parity import rel, cosine, FP32_TOL, BF16_TOL, BF16_GRAD_COS
from test_gpu_pretrain import BENCH, PER_LEAD, PER_LEAD_SHORT
from test_gpu_dropout import inject


def stream():
    return torch.cuda.current_stream().cuda_stream


def lib():
    return _lib.load()


# ---- the grouped AdamW kernel ---------------------------------------------------------------------------------------
# a flat buffer of "tensors" at 64-element offsets, as the model lays its parameters out; sizes not multiples of 64
SIZES = [1000, 64, 3, 4096, 700, 129, 2500, 60, 8192, 33]
GROUPS = [0, 1, 255, 2, 0, 1, 2, 255, 3, 3]          # 255: in no group
LR = [1e-2, 3e-3, 5e-4, 2e-2]
WD = [0.05, 0.0, 0.1, 0.02]


def layout():
    offs, o = [], 0
    for n in SIZES:
        offs.append(o)
        o += (n + 63) // 64 * 64
    return offs, o


def group_map_of(offs, groups):
    gm = torch.full((layout()[1] // 64,), 255, dtype=torch.uint8)
    for o, n, g in zip(offs, SIZES, groups):
        gm[o // 64:(o + n + 63) // 64] = g
    return gm.cuda()


def grouped_step(p, m, v, g, g_code, shadow, gmap, vals, stats, slices=None):
    hyper = torch.tensor(vals, dtype=torch.float32, device='cuda')
    n = p.numel()
    esz = 4 if g_code == _lib.F32 else 2
    for i, (lo, hi) in enumerate(slices or [(0, n)]):
        flags = 0 if slices is None else _lib.ADAMW_SLICE | (_lib.ADAMW_FIRST_SLICE if i == 0 else 0)
        _lib.check(lib().ecgvit_adamw_step_grouped(
            p.data_ptr() + 4 * lo, m.data_ptr() + 4 * lo, v.data_ptr() + 4 * lo, g.data_ptr() + esz * lo, g_code,
            None if shadow is None else shadow.data_ptr() + 2 * lo, hi - lo, gmap.data_ptr() + lo // 64,
            hyper.data_ptr() + 64, hyper.data_ptr(), stats.data_ptr(), flags, stream()), 'adamw_step_grouped')


def hyper_vals(t, gscale, lrs=LR, wds=WD, skip=False):
    from ecg_b200.optim import group_table
    return _lib.adamw_hyper(0.0, 0.9, 0.999, 1e-8, 0.0, t, 0.0, gscale, skip=skip) + group_table(lrs, wds, 0.9, t)


@pytest.mark.parametrize('grad_dtype', ['fp32', 'bf16'])
@pytest.mark.parametrize('shadow', [False, True])
@pytest.mark.parametrize('sliced', [False, True])
def test_grouped_adamw_matches_torch_adamw(grad_dtype, shadow, sliced):
    """three steps against torch.optim.AdamW with the same groups; bf16 gradients scaled by 1/world (world 2), as the
    data-parallel bf16 all-reduce leaves them"""
    offs, total = layout()
    gen = torch.Generator().manual_seed(11)
    p0 = torch.zeros(total)
    for o, n in zip(offs, SIZES):
        p0[o:o + n] = torch.randn(n, generator=gen)
    ref = [nn.Parameter(p0[o:o + n].clone().double()) for o, n in zip(offs, SIZES)]
    opt = torch.optim.AdamW([{'params': [ref[i] for i in range(len(SIZES)) if GROUPS[i] == k], 'lr': LR[k],
                              'weight_decay': WD[k]} for k in range(4)], betas=(0.9, 0.999), eps=1e-8)
    p, m, v = p0.cuda(), torch.zeros(total, device='cuda'), torch.zeros(total, device='cuda')
    sh = p.bfloat16() if shadow else None
    gmap = group_map_of(offs, GROUPS)
    stats = torch.zeros(_lib.STATS_FLOATS, device='cuda')
    g_code, gscale = (_lib.F32, 1.0) if grad_dtype == 'fp32' else (_lib.BF16, 0.5)
    slices = [(0, offs[3]), (offs[3], offs[6]), (offs[6], total)] if sliced else None
    for t in range(1, 4):
        g = torch.zeros(total)
        for o, n in zip(offs, SIZES):
            g[o:o + n] = torch.randn(n, generator=gen)
        gd = g.cuda() if grad_dtype == 'fp32' else g.cuda().bfloat16()
        for r, o, n in zip(ref, offs, SIZES):
            r.grad = gd[o:o + n].double().cpu() * gscale
        opt.step()
        grouped_step(p, m, v, gd, g_code, sh, gmap, hyper_vals(t, gscale), stats, slices)
    torch.cuda.synchronize()
    for i, (r, o, n) in enumerate(zip(ref, offs, SIZES)):
        got = p[o:o + n].cpu()
        if GROUPS[i] == 255:
            assert torch.equal(got, p0[o:o + n]), i   # untouched, moments too
            assert float(m[o:o + n].abs().max()) == 0.0 and float(v[o:o + n].abs().max()) == 0.0
        else:
            assert rel(got, r.detach()) < 1e-5, (i, rel(got, r.detach()))
    if shadow:
        assert torch.equal(sh, p.bfloat16())
    assert float(stats[3]) == 0.0


@pytest.mark.parametrize('grad_dtype', ['fp32', 'bf16'])
def test_single_group_equals_plain_adamw_bit_for_bit(grad_dtype):
    n = 64 * 4099
    gen = torch.Generator(device='cuda').manual_seed(3)
    p = torch.randn(n, device='cuda', generator=gen)
    g = torch.randn(n, device='cuda', generator=gen)
    g_code = _lib.F32
    if grad_dtype == 'bf16':
        g, g_code = g.bfloat16(), _lib.BF16
    a = [p.clone(), torch.zeros(n, device='cuda'), torch.zeros(n, device='cuda'), p.bfloat16()]
    b = [p.clone(), torch.zeros(n, device='cuda'), torch.zeros(n, device='cuda'), p.bfloat16()]
    gmap = torch.zeros(n // 64, dtype=torch.uint8, device='cuda')
    stats_a, stats_b = torch.zeros(_lib.STATS_FLOATS, device='cuda'), torch.zeros(_lib.STATS_FLOATS, device='cuda')
    for t in range(1, 4):
        vals = _lib.adamw_hyper(3e-3, 0.9, 0.999, 1e-8, 0.05, t, 0.0, 0.5)
        hyper = torch.tensor(vals, device='cuda')
        _lib.check(lib().ecgvit_adamw_step(a[0].data_ptr(), a[1].data_ptr(), a[2].data_ptr(), g.data_ptr(), g_code,
                                           a[3].data_ptr(), n, hyper.data_ptr(), stats_a.data_ptr(), 0, stream()))
        grouped_step(b[0], b[1], b[2], g, g_code, b[3], gmap, hyper_vals(t, 0.5, [3e-3], [0.05]), stats_b)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_grouped_adamw_skip_flag_and_nonfinite_counter():
    offs, total = layout()
    gen = torch.Generator(device='cuda').manual_seed(5)
    p = torch.randn(total, device='cuda', generator=gen)
    m, v = torch.rand(total, device='cuda', generator=gen), torch.rand(total, device='cuda', generator=gen)
    g = torch.randn(total, device='cuda', generator=gen)
    gmap = group_map_of(offs, GROUPS)
    before = (p.clone(), m.clone(), v.clone())
    stats = torch.zeros(_lib.STATS_FLOATS, device='cuda')
    # skip: a deferred-update slot with nothing pending
    grouped_step(p, m, v, g, _lib.F32, None, gmap, hyper_vals(1, 1.0, skip=True), stats)
    assert all(torch.equal(x, y) for x, y in zip((p, m, v), before)) and float(stats[3]) == 0.0
    # a non-finite norm: nothing changes, the sticky counter counts, and only the first slice counts
    stats[0] = float('inf')
    grouped_step(p, m, v, g, _lib.F32, None, gmap, hyper_vals(1, 1.0), stats)
    grouped_step(p, m, v, g, _lib.F32, None, gmap, hyper_vals(1, 1.0), stats,
                 slices=[(0, offs[3]), (offs[3], total)])
    assert all(torch.equal(x, y) for x, y in zip((p, m, v), before))
    assert float(stats[3]) == 2.0
    # a finite update leaves the ungrouped tensors alone, moments included
    stats.zero_()
    grouped_step(p, m, v, g, _lib.F32, None, gmap, hyper_vals(1, 1.0), stats)
    for o, n, k in zip(offs, SIZES, GROUPS):
        same = torch.equal(p[o:o + n], before[0][o:o + n]) and torch.equal(m[o:o + n], before[1][o:o + n])
        assert same == (k == 255)


# ---- optimizer front ends with groups against the oracle ------------------------------------------------------------
def oracle_groups(oracle, model_groups, model, lr):
    """the same groups over the oracle's parameters (same names), lr = lr * lr_scale as FusedAdamW defaults it"""
    names = {id(p): n for n, p in model.named_parameters()}
    op = dict(oracle.named_parameters())
    return [{'params': [op[names[id(p)]] for p in g['params']], 'lr': lr * g['lr_scale'],
             'weight_decay': g['weight_decay']} for g in model_groups]


def make_pair(cfg, dtype, batch, pool='cls', seed=77):
    torch.manual_seed(seed)
    oracle = OracleEcgVit(config=OracleConfig(**cfg)).train()
    oracle.vit.pool = pool            # the restated vit_pytorch ViT reads `pool` at forward
    model = EcgVit(config=EcgVitConfig(compute_dtype=dtype, pool=pool, **cfg))
    model.load_state_dict(oracle.state_dict(), strict=True)
    model.cuda().train()
    x, y = synthetic_batch(batch, num_channels=cfg['num_channels'], length=cfg['max_signal_length'], seed=seed)
    return oracle, model, x, y


def grouped_oracle_trainer(oracle, groups, lr, schedule, n_warmup, n_step):
    ot = OracleTrainer(oracle, learning_rate=lr, schedule=schedule, n_warmup=n_warmup, n_step=n_step)
    ot.optimizer = torch.optim.AdamW(groups, lr=lr)
    ot.scheduler = torch.optim.lr_scheduler.LambdaLR(ot.optimizer, lambda s: lr_lambda(schedule, s, n_warmup, n_step))
    return ot


def test_fused_adamw_groups_with_lambdalr_track_torch_adamw():
    oracle, model, x, y = make_pair(GOLDEN_CFG, 'fp32', 4, pool='mean')
    groups = param_groups_lrd(model, weight_decay=0.05, layer_decay=0.6)
    opt = FusedAdamW(model, lr=2e-3, param_groups=groups)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda s: 1.0 / (1 + s))
    oopt = torch.optim.AdamW(oracle_groups(oracle, groups, model, 2e-3), lr=2e-3)
    osched = torch.optim.lr_scheduler.LambdaLR(oopt, lambda s: 1.0 / (1 + s))
    for _ in range(3):
        opt.zero_grad()
        model(x.cuda(), y.cuda()).loss.backward()
        opt.step()
        sched.step()
        oopt.zero_grad()
        oracle(x, y).loss.backward()
        oopt.step()
        osched.step()
    for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()):
        assert rel(p, q) < FP32_TOL, (k, rel(p, q))
    # the optimizer state round-trips the groups
    opt2 = FusedAdamW(model, lr=2e-3, param_groups=param_groups_lrd(model, weight_decay=0.05, layer_decay=0.6))
    opt2.load_state_dict(opt.state_dict())
    assert [(g['lr'], g['lr_scale'], g['weight_decay']) for g in opt2.param_groups] == \
        [(g['lr'], g['lr_scale'], g['weight_decay']) for g in opt.param_groups]
    assert torch.equal(opt2._v, opt._v) and opt2._step == 3


@pytest.mark.parametrize('mode', ['eager', 'graph', 'deferred'])
def test_trainer_groups_track_the_oracle(mode):
    oracle, model, x, y = make_pair(GOLDEN_CFG, 'fp32', 4)
    groups = param_groups_lrd(model, weight_decay=0.05, layer_decay=0.75)
    kw = dict(learning_rate=2e-3, schedule='cosine', n_warmup=0, n_step=5)
    tr = FusedTrainer(model, use_cuda_graph=mode == 'graph', defer_optimizer=mode == 'deferred', data_parallel=False,
                      param_groups=groups, **kw)
    ot = grouped_oracle_trainer(oracle, oracle_groups(oracle, groups, model, 2e-3), 2e-3, 'cosine', 0, 5)
    for _ in range(3):
        o_loss, _, o_norm = ot.step(x, y)
        loss, _ = tr.step(x.cuda(), y.cuda())
        assert rel(loss, o_loss) < FP32_TOL
    tr.check_finite()
    for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()):
        assert rel(p, q) < FP32_TOL, (k, rel(p, q))
    if mode == 'graph':
        plain = FusedTrainer(EcgVit(config=EcgVitConfig(compute_dtype='fp32', **GOLDEN_CFG)).cuda().train(),
                             use_cuda_graph=True, data_parallel=False, **kw)
        plain.step(x.cuda(), y.cuda())
        assert tr.launches_per_step == plain.launches_per_step   # the grouped update is one launch, as the plain one


def test_trainer_groups_save_resume_continues_the_run(tmp_path):
    kw = dict(learning_rate=1e-3, schedule='cosine', n_warmup=1, n_step=8, use_cuda_graph=True, data_parallel=False)
    _, m_ref, x, y = make_pair(GOLDEN_CFG, 'fp32', 4, pool='mean')
    _, m_a, _, _ = make_pair(GOLDEN_CFG, 'fp32', 4, pool='mean')
    xs, ys = x.cuda(), y.cuda()
    t_ref = FusedTrainer(m_ref, param_groups=param_groups_lrd(m_ref), **kw)
    t_a = FusedTrainer(m_a, param_groups=param_groups_lrd(m_a), **kw)
    for _ in range(4):
        t_ref.step(xs, ys)
    for _ in range(2):
        t_a.step(xs, ys)
    t_a.save(str(tmp_path), 'mid')
    m_b = EcgVit(config=EcgVitConfig(compute_dtype='fp32', pool='mean', **GOLDEN_CFG)).cuda().train()
    t_b = FusedTrainer(m_b, param_groups=param_groups_lrd(m_b), **kw)
    t_b.resume(str(tmp_path), 'mid')
    for _ in range(2):
        t_b.step(xs, ys)
    assert t_b.step_count == 4
    # the weight-gradient GEMMs accumulate with atomics: the two runs agree to fp32 rounding, as test_gpu_parity's resume
    assert rel(m_b._flat_p, m_ref._flat_p) < 1e-5
    assert rel(t_b.exp_avg_sq, t_ref.exp_avg_sq) < 1e-4
    # a trainer with other groups, or none, refuses the checkpoint
    m_c = EcgVit(config=EcgVitConfig(compute_dtype='fp32', pool='mean', **GOLDEN_CFG)).cuda().train()
    with pytest.raises(ValueError):
        FusedTrainer(m_c, **kw).resume(str(tmp_path), 'mid')
    with pytest.raises(ValueError):
        FusedTrainer(m_c, param_groups=param_groups_lrd(m_c, layer_decay=0.5), **kw).resume(str(tmp_path), 'mid')


# ---- mean pooling ---------------------------------------------------------------------------------------------------
GEOMETRY = {'golden': (GOLDEN_CFG, 4), 'bench': (BENCH, 2), 'per_lead': (PER_LEAD, 2),
            'per_lead_short': (PER_LEAD_SHORT, 3)}


@pytest.mark.parametrize('geometry', ['golden', 'bench', 'per_lead_short'])
def test_mean_pool_fp32_matches_oracle(geometry):
    cfg, batch = GEOMETRY[geometry]
    oracle, model, x, y = make_pair(cfg, 'fp32', batch, pool='mean')
    o = oracle(sample_values=x, labels=y)
    o.loss.backward()
    out = model(sample_values=x.cuda(), labels=y.cuda())
    out.loss.backward()
    assert rel(out.logits, o.logits) < FP32_TOL and rel(out.loss, o.loss) < FP32_TOL
    for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()):
        assert rel(p.grad, q.grad) < FP32_TOL, (k, rel(p.grad, q.grad))


@pytest.mark.parametrize('geometry,res', [('golden', 'bf16'), ('bench', 'bf16'), ('per_lead', 'bf16'),
                                          ('golden', 'fp32'), ('bench', 'fp32')])
def test_mean_pool_bf16_matches_oracle(geometry, res):
    cfg, batch = GEOMETRY[geometry]
    torch.manual_seed(77)
    oracle = OracleEcgVit(config=OracleConfig(**cfg)).train()
    oracle.vit.pool = 'mean'
    model = EcgVit(config=EcgVitConfig(compute_dtype='bf16', residual_dtype=res, pool='mean', **cfg))
    model.load_state_dict(oracle.state_dict(), strict=True)
    model.cuda().train()
    assert model._res_f32 == (res == 'fp32')
    x, y = synthetic_batch(batch, num_channels=cfg['num_channels'], length=cfg['max_signal_length'], seed=77)
    o = oracle(sample_values=x, labels=y)
    o.loss.backward()
    out = model(sample_values=x.cuda(), labels=y.cuda())
    out.loss.backward()
    assert rel(out.logits, o.logits) < BF16_TOL and rel(out.loss, o.loss) < BF16_TOL
    worst = min((cosine(p.grad, q.grad), k) for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()))
    assert worst[0] >= BF16_GRAD_COS, worst


@pytest.mark.parametrize('dtype,tol', [('fp32', FP32_TOL), ('bf16', BF16_TOL)])
def test_mean_pool_with_dropout_matches_oracle(dtype, tol):
    cfg = dict(GOLDEN_CFG, hidden_size=128, num_attention_heads=4, intermediate_size=256, hidden_dropout_prob=0.1,
               attention_probs_dropout_prob=0.2)
    oracle, model, x, y = make_pair(cfg, dtype, 6, pool='mean', seed=3)
    out = model(sample_values=x.cuda(), labels=y.cuda())
    out.loss.backward()
    inject(oracle, int(model._engine.rng[0]), cfg['attention_probs_dropout_prob'], cfg['hidden_dropout_prob'])
    ref = oracle(sample_values=x, labels=y)
    ref.loss.backward()
    assert rel(out.logits, ref.logits) < tol and rel(out.loss, ref.loss) < tol
    for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()):
        if dtype == 'fp32':
            assert rel(p.grad, q.grad) < 5e-4, (k, rel(p.grad, q.grad))   # test_gpu_dropout's bar with masks on
        else:
            assert cosine(p.grad, q.grad) > BF16_GRAD_COS, (k, cosine(p.grad, q.grad))


def test_mean_pool_eval_recorder_and_unreduced_loss():
    from ecg_b200 import Recorder, evaluate
    oracle, model, x, y = make_pair(GOLDEN_CFG, 'fp32', 4, pool='mean')
    oracle.eval(), model.eval()
    model.loss_reduction = oracle.loss_reduction = 'none'
    with torch.no_grad():
        o = oracle(sample_values=x, labels=y)
        out = model(sample_values=x.cuda(), labels=y.cuda())
    assert out.loss.shape == (4, 71) and rel(out.loss, o.loss) < FP32_TOL
    model.loss_reduction = 'mean'
    logits, attns = Recorder(model.vit)(x.cuda().unsqueeze(2))
    assert rel(logits, o.logits) < FP32_TOL and attns.shape[1] == GOLDEN_CFG['num_hidden_layers']
    d = evaluate(model, [{'sample_values': x, 'labels': y}])
    assert abs(d['eval/loss'] - float(nn.functional.binary_cross_entropy_with_logits(o.logits, y))) < 1e-5


@pytest.mark.parametrize('dtype', [_lib.F32, _lib.BF16, _lib.BF16_RES32])
def test_token_mean_kernels_against_torch_and_bit_identical(dtype):
    B, N, d = 7, 241, 768
    gen = torch.Generator(device='cuda').manual_seed(9)
    tdt = torch.bfloat16 if dtype == _lib.BF16 else torch.float32
    tok = torch.randn(B, N, d, device='cuda', generator=gen).to(tdt)
    outs = []
    for _ in range(2):
        out = torch.full((B, d), float('nan'), device='cuda')
        _lib.check(lib().ecgvit_token_mean(tok.data_ptr(), out.data_ptr(), B, N, d, dtype, stream()), 'token_mean')
        outs.append(out)
    assert torch.equal(outs[0], outs[1])
    assert rel(outs[0], tok.double().mean(1)) < 1e-6
    dpool = torch.randn(B, d, device='cuda', generator=gen)
    gdt = torch.float32 if dtype == _lib.F32 else torch.bfloat16   # the token gradient is bf16 in both bf16 modes
    grads = []
    for _ in range(2):
        dtok = torch.full((B, N, d), float('nan'), device='cuda', dtype=gdt)
        _lib.check(lib().ecgvit_token_mean_bwd(dpool.data_ptr(), dtok.data_ptr(), B, N, d, dtype, stream()))
        grads.append(dtok)
    assert torch.equal(grads[0], grads[1])
    assert torch.equal(grads[0], (dpool / N).unsqueeze(1).expand(B, N, d).to(gdt))


def test_mae_encoder_fine_tunes_with_mean_pool_and_lrd():
    """the user path: MAE pre-training -> encoder_state_dict() -> EcgVit(pool='mean') -> three captured FusedTrainer
    steps with layer-wise LR decay, tracking the oracle with the same groups"""
    cfg = dict(GOLDEN_CFG)
    torch.manual_seed(21)
    pre = EcgVitForMaskedAutoencoding(EcgVitConfig(compute_dtype='fp32', **cfg), decoder_hidden_size=32,
                                      decoder_num_hidden_layers=2, decoder_num_attention_heads=2,
                                      decoder_intermediate_size=64).cuda().train()
    x, y = synthetic_batch(4, length=cfg['max_signal_length'], seed=5)
    pt = FusedTrainer(pre, learning_rate=1e-3, data_parallel=False)
    for _ in range(2):
        pt.step(x.cuda())
    model = EcgVit(config=EcgVitConfig(compute_dtype='fp32', pool='mean', **cfg))
    missing, unexpected = model.load_state_dict(pre.encoder_state_dict(), strict=False)
    assert sorted(missing) == ['vit.mlp_head.0.bias', 'vit.mlp_head.0.weight', 'vit.mlp_head.1.bias',
                               'vit.mlp_head.1.weight'] and not unexpected
    oracle = OracleEcgVit(config=OracleConfig(**cfg)).train()
    oracle.vit.pool = 'mean'
    oracle.load_state_dict({k: v.cpu() for k, v in model.state_dict().items()}, strict=True)
    model.cuda().train()
    groups = param_groups_lrd(model, weight_decay=0.05, layer_decay=0.75)
    tr = FusedTrainer(model, learning_rate=1e-3, use_cuda_graph=True, data_parallel=False, param_groups=groups)
    ot = grouped_oracle_trainer(oracle, oracle_groups(oracle, groups, model, 1e-3), 1e-3, 'constant', 0, 1000)
    for _ in range(3):
        o_loss, _, _ = ot.step(x, y)
        loss, _ = tr.step(x.cuda(), y.cuda())
        assert rel(loss, o_loss) < FP32_TOL
    for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()):
        assert rel(p, q) < FP32_TOL, (k, rel(p, q))
