"""GPU tier: stochastic depth (`EcgVitConfig.drop_path_rate`).  The three drop-path kernel variants against torch
compositions, then whole models against the CPU oracle with the kernels' per-record keeps injected through forward hooks
on its PreNorm modules (tests/drop_path_oracle.py), and dropout masks injected as in test_gpu_dropout.py."""
import ctypes

import pytest
import torch
from torch import nn

pytestmark = pytest.mark.gpu

from conftest import GOLDEN_CFG
import ecg_b200
from ecg_b200 import (EcgVit, EcgVitConfig, EcgVitForMaskedAutoencoding, EcgVitForMaskedPatchModeling, FusedTrainer,
                      param_groups_lrd, _lib)
from oracle.ecg_vit_oracle import OracleConfig, OracleEcgVit, OracleTrainer, synthetic_batch
from oracle.mae_oracle import OracleMaskedAutoencoder
from oracle.mpm_oracle import OracleMaskedPatchModel

from drop_path_oracle import inject_drop_path, keeps, path_keep
from test_gpu_dropout import inject as inject_dropout
from test_gpu_finetune import grouped_oracle_trainer, oracle_groups
from test_gpu_mae import DEC
from test_gpu_parity import rel, cosine, FP32_TOL, BF16_GRAD_COS
from test_gpu_pretrain import PER_LEAD_SHORT


def stream():
    return torch.cuda.current_stream().cuda_stream


def lib():
    return _lib.load()


SEED = 0x1234567
MAE_N = 3    # an MAE encoder's token count n_vis + 1 (golden geometry: 10 patches, 8 masked -> 2 visible + CLS)


def seed_buf(seed=SEED):
    return torch.tensor([seed, 0], dtype=torch.int32, device='cuda')


def row_factor(rate, site, M, N, seed=SEED):
    return path_keep(seed, site, rate, M // N).repeat_interleave(N).cuda()


def elem_mask(p, site, M, d, seed=SEED):
    return _lib.dropout_keep_mask(seed, site, p, torch.arange(M * d).reshape(M, d)).cuda()


# ---- kernels ---------------------------------------------------------------------------------------------------------
def run_gemm(A, W, bias, aux, out, epi, dtype, p, site, seed, path=None):
    M, K = A.shape
    N = W.shape[0]
    g = _lib.GemmArgs(M, N, K, A.data_ptr(), K, 1, W.data_ptr(), K, 1, epi, out.data_ptr(), N, None, aux.data_ptr(),
                      bias.data_ptr(), dtype, 1, site, p, seed.data_ptr())
    if path is None:
        return lib().ecgvit_gemm(ctypes.byref(g), stream())
    return lib().ecgvit_gemm_drop_path(ctypes.byref(g), path[0], path[1], path[2], stream())


@pytest.mark.parametrize('mode', ['fp32', 'bf16', 'bf16_res32'])
@pytest.mark.parametrize('p', [0.0, 0.2])
@pytest.mark.parametrize('n_tok', [51, MAE_N, 2401])
def test_gemm_drop_path_against_torch(mode, p, n_tok):
    torch.manual_seed(n_tok)
    B = 6 if n_tok < 2401 else 2
    M, K, N = B * n_tok, 128, 64
    T = torch.float32 if mode == 'fp32' else torch.bfloat16
    RT = torch.bfloat16 if mode == 'bf16' else torch.float32
    dtype = _lib.F32 if mode == 'fp32' else _lib.BF16
    epi = _lib.EPI_BIAS_RES_F32 if mode == 'bf16_res32' else _lib.EPI_BIAS_RES
    A = torch.randn(M, K, device='cuda').to(T)
    W = (torch.randn(N, K, device='cuda') / K ** 0.5).to(T)
    bias = torch.randn(N, device='cuda')
    aux = torch.randn(M, N, device='cuda').to(RT)
    seed = seed_buf()
    rate, site = 0.5, 37
    out = torch.empty(M, N, device='cuda', dtype=RT)
    _lib.check(run_gemm(A, W, bias, aux, out, epi, dtype, p, 5, seed, (rate, site, n_tok)), 'gemm_drop_path')
    s = row_factor(rate, site, M, n_tok)
    assert (s == 0).any() and (s > 0).any()
    branch = (A.float() @ W.float().t() + bias) * elem_mask(p, 5, M, N)
    want = s[:, None] * branch + aux.float()
    dropped = s == 0
    # a dropped record's rows are its residual, exactly
    assert torch.equal(out[dropped], aux[dropped])
    tol = 1e-5 if mode == 'fp32' else 1e-2
    assert rel(out[~dropped].float(), want[~dropped]) < tol
    # rate 0 is the plain entry point, bit for bit
    ref, got = torch.empty_like(out), torch.empty_like(out)
    _lib.check(run_gemm(A, W, bias, aux, ref, epi, dtype, p, 5, seed), 'gemm')
    _lib.check(run_gemm(A, W, bias, aux, got, epi, dtype, p, 5, seed, (0.0, site, n_tok)), 'gemm_drop_path')
    assert torch.equal(ref, got)


def test_gemm_drop_path_rejections():
    A = torch.zeros(64, 64, device='cuda', dtype=torch.bfloat16)
    W = torch.zeros(64, 64, device='cuda', dtype=torch.bfloat16)
    bias = torch.zeros(64, device='cuda')
    aux = torch.zeros(64, 64, device='cuda', dtype=torch.bfloat16)
    out = torch.full((64, 64), 7.0, device='cuda', dtype=torch.bfloat16)
    seed = seed_buf()
    for epi in (_lib.EPI_STORE, _lib.EPI_BIAS_GELU, _lib.EPI_DGELU):
        assert run_gemm(A, W, bias, aux, out, epi, _lib.BF16, 0.0, 0, seed, (0.1, 40, 8)) != 0
        assert 'drop path' in _lib.last_error()
    assert run_gemm(A, W, bias, aux, out, _lib.EPI_BIAS_RES, _lib.BF16, 0.0, 0, seed, (0.1, 40, 0)) != 0
    assert run_gemm(A, W, bias, aux, out, _lib.EPI_BIAS_RES, _lib.BF16, 0.0, 0, seed, (1.0, 40, 8)) != 0
    g = _lib.GemmArgs(64, 64, 64, A.data_ptr(), 64, 1, W.data_ptr(), 64, 1, _lib.EPI_BIAS_RES, out.data_ptr(), 64, None,
                      aux.data_ptr(), bias.data_ptr(), _lib.BF16, 1, 0, 0.0, None)
    assert lib().ecgvit_gemm_drop_path(ctypes.byref(g), 0.1, 40, 8, stream()) != 0   # no seed
    torch.cuda.synchronize()
    assert bool((out == 7.0).all()), 'a rejected call must not launch'


@pytest.mark.parametrize('mode', ['fp32', 'bf16', 'bf16_res32'])
@pytest.mark.parametrize('p', [0.0, 0.2])
@pytest.mark.parametrize('n_tok', [51, MAE_N, 2401])
def test_layernorm_bwd_drop_path_against_plain_and_torch(mode, p, n_tok):
    torch.manual_seed(n_tok + 1)
    B = 4 if n_tok < 2401 else 2
    M, d = B * n_tok, 128
    T = torch.float32 if mode == 'fp32' else torch.bfloat16
    XT = torch.bfloat16 if mode == 'bf16' else torch.float32
    code = {'fp32': _lib.F32, 'bf16': _lib.BF16, 'bf16_res32': _lib.BF16_RES32}[mode]
    dy = torch.randn(M, d, device='cuda').to(T)
    x = torch.randn(M, d, device='cuda').to(XT)
    dres = torch.randn(M, d, device='cuda').to(T)
    gamma = 1 + 0.1 * torch.randn(d, device='cuda')
    xf = x.float()
    mean = xf.mean(1)
    rstd = (xf.var(1, unbiased=False) + 1e-5).rsqrt()
    scratch = torch.empty(int(lib().ecgvit_layernorm_bwd_scratch_floats(d)), device='cuda')
    seed = seed_buf()
    rate, site = 0.5, 41

    def call(path):
        dx, dxm = torch.empty(M, d, device='cuda', dtype=T), torch.empty(M, d, device='cuda', dtype=T)
        dg, db, dc = (torch.zeros(d, device='cuda') for _ in range(3))
        args = (dy.data_ptr(), x.data_ptr(), gamma.data_ptr(), mean.data_ptr(), rstd.data_ptr(), dres.data_ptr(),
                dx.data_ptr(), dg.data_ptr(), db.data_ptr(), dc.data_ptr(), scratch.data_ptr(), dxm.data_ptr(), p, 9,
                seed.data_ptr(), M, d, 0, code)
        if path is None:
            _lib.check(lib().ecgvit_layernorm_bwd(*args, stream()), 'layernorm_bwd')
        else:
            _lib.check(lib().ecgvit_layernorm_bwd_drop_path(*args, path, site, n_tok, stream()), 'layernorm_bwd')
        return dx, dxm, dg, db, dc

    dx0, _, dg0, db0, _ = call(None)
    dx, dxm, dg, db, dc = call(rate)
    assert torch.equal(dx, dx0) and torch.equal(dg, dg0) and torch.equal(db, db0)
    s = row_factor(rate, site, M, n_tok)
    want = dx.float() * elem_mask(p, 9, M, d) * s[:, None]
    assert torch.equal(dxm[s == 0], torch.zeros_like(dxm[s == 0]))
    assert rel(dxm.float(), want) < (1e-6 if mode == 'fp32' else 1e-2)
    assert rel(dc, want.double().sum(0)) < (1e-5 if mode == 'fp32' else 1e-2)
    # rate 0 is the plain entry point (which leaves dxm unwritten without dropout)
    out0, plain = call(0.0), call(None)
    for i, (a, b) in enumerate(zip(out0, plain)):
        if i != 1 or p > 0:
            assert torch.equal(a, b)


@pytest.mark.parametrize('mode', ['fp32', 'bf16'])
@pytest.mark.parametrize('p', [0.0, 0.2])
@pytest.mark.parametrize('n_tok', [51, MAE_N, 2401])
def test_dropout_bwd_copy_drop_path_against_torch(mode, p, n_tok):
    torch.manual_seed(n_tok + 2)
    B = 4 if n_tok < 2401 else 2
    M, d = B * n_tok, 128
    T = torch.float32 if mode == 'fp32' else torch.bfloat16
    code = _lib.F32 if mode == 'fp32' else _lib.BF16
    dy = torch.randn(M, d, device='cuda').to(T)
    seed = seed_buf()
    rate, site = 0.5, 43
    dym = torch.empty_like(dy)
    dc = torch.zeros(d, device='cuda')
    _lib.check(lib().ecgvit_dropout_bwd_copy_drop_path(dy.data_ptr(), dym.data_ptr(), dc.data_ptr(), M, d, d, p, 7,
                                                        seed.data_ptr(), code, rate, site, n_tok, stream()),
               'dropout_bwd_copy')
    s = row_factor(rate, site, M, n_tok)
    want = (dy.float() * elem_mask(p, 7, M, d) * s[:, None]).to(T)
    assert torch.equal(dym, want)
    assert rel(dc, want.double().sum(0)) < 1e-5
    if p > 0:   # rate 0 is the plain entry point
        a, b = torch.empty_like(dy), torch.empty_like(dy)
        _lib.check(lib().ecgvit_dropout_bwd_copy(dy.data_ptr(), a.data_ptr(), None, M, d, d, p, 7, seed.data_ptr(), code,
                                                 stream()), 'dropout_bwd_copy')
        _lib.check(lib().ecgvit_dropout_bwd_copy_drop_path(dy.data_ptr(), b.data_ptr(), None, M, d, d, p, 7,
                                                            seed.data_ptr(), code, 0.0, site, n_tok, stream()),
                   'dropout_bwd_copy')
        assert torch.equal(a, b)
    # rejections: bad rate, bad record length, no seed (nothing launched)
    keep = dym.clone()
    assert lib().ecgvit_dropout_bwd_copy_drop_path(dy.data_ptr(), dym.data_ptr(), None, M, d, d, p, 7, seed.data_ptr(),
                                                   code, 1.5, site, n_tok, stream()) != 0
    assert lib().ecgvit_dropout_bwd_copy_drop_path(dy.data_ptr(), dym.data_ptr(), None, M, d, d, p, 7, seed.data_ptr(),
                                                   code, rate, site, 0, stream()) != 0
    assert lib().ecgvit_dropout_bwd_copy_drop_path(dy.data_ptr(), dym.data_ptr(), None, M, d, d, 0.0, 7, None, code,
                                                   rate, site, n_tok, stream()) != 0
    torch.cuda.synchronize()
    assert torch.equal(dym, keep)


# ---- whole models against the oracle ---------------------------------------------------------------------------------
RATE = 0.5
CFG3 = dict(GOLDEN_CFG, num_hidden_layers=3)


def assert_some_drop(seed, depth, B):
    ks = keeps(seed, depth, RATE, B)
    assert any(bool((a == 0).any() or (f == 0).any()) for a, f in ks), 'no record was dropped'
    assert all(bool((a > 0).any() and (f > 0).any()) for a, f in ks), 'no record was kept'


def check_grads(model, oracle, dtype):
    for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()):
        if q.grad is None or float(q.grad.norm()) == 0:
            continue
        if dtype == 'fp32':
            assert rel(p.grad, q.grad) < 5e-4, (k, rel(p.grad, q.grad))
        else:
            assert cosine(p.grad, q.grad) > BF16_GRAD_COS, (k, cosine(p.grad, q.grad))


@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
@pytest.mark.parametrize('pool', ['cls', 'mean'])
@pytest.mark.parametrize('p', [0.0, 0.1])
def test_ecgvit_matches_oracle_with_injected_keeps(dtype, pool, p):
    cfg = dict(CFG3, hidden_dropout_prob=p, attention_probs_dropout_prob=p)
    torch.manual_seed(5)
    oracle = OracleEcgVit(config=OracleConfig(**cfg)).train()
    oracle.vit.pool = pool
    model = EcgVit(config=EcgVitConfig(compute_dtype=dtype, pool=pool, drop_path_rate=RATE, **cfg))
    model.load_state_dict(oracle.state_dict(), strict=True)
    model.cuda().train()
    x, y = synthetic_batch(6, length=500, seed=11)
    out = model(sample_values=x.cuda(), labels=y.cuda())
    out.loss.backward()
    seed = int(model._engine.rng[0])
    assert_some_drop(seed, 3, 6)
    if p > 0:
        inject_dropout(oracle, seed, p, p)
    hs = inject_drop_path(oracle.vit.transformer, seed, RATE)
    ref = oracle(sample_values=x, labels=y)
    ref.loss.backward()
    for h in hs:
        h.remove()
    if dtype == 'fp32':
        assert rel(out.logits, ref.logits) < FP32_TOL and rel(out.loss, ref.loss) < FP32_TOL
    else:
        assert cosine(out.logits, ref.logits) > 0.999
    check_grads(model, oracle, dtype)


def test_ecgvit_per_lead_bf16_matches_oracle():
    cfg = dict(PER_LEAD_SHORT)
    torch.manual_seed(6)
    oracle = OracleEcgVit(config=OracleConfig(**cfg)).train()
    model = EcgVit(config=EcgVitConfig(compute_dtype='bf16', drop_path_rate=RATE, **cfg))
    model.load_state_dict(oracle.state_dict(), strict=True)
    model.cuda().train()
    x, y = synthetic_batch(6, num_channels=cfg['num_channels'], length=cfg['max_signal_length'], seed=12)
    out = model(sample_values=x.cuda(), labels=y.cuda())
    out.loss.backward()
    seed = int(model._engine.rng[0])
    hs = inject_drop_path(oracle.vit.transformer, seed, RATE)
    ref = oracle(sample_values=x, labels=y)
    ref.loss.backward()
    for h in hs:
        h.remove()
    assert cosine(out.logits, ref.logits) > 0.999
    check_grads(model, oracle, 'bf16')


@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
def test_masked_patch_model_matches_oracle(dtype):
    torch.manual_seed(7)
    oracle = OracleMaskedPatchModel(OracleConfig(**CFG3)).train()
    model = EcgVitForMaskedPatchModeling(config=EcgVitConfig(compute_dtype=dtype, drop_path_rate=RATE, **CFG3))
    model.load_state_dict(oracle.state_dict(), strict=True)
    model.cuda().train()
    x, _ = synthetic_batch(6, length=500, seed=13)
    out = model(x.cuda())
    out.loss.backward()
    seed = int(model._engine.rng[0])
    assert_some_drop(seed, 3, 6)
    hs = inject_drop_path(oracle.vit.transformer, seed, RATE)
    o_loss, _ = oracle(x, out.bool_masked_pos.cpu())
    o_loss.backward()
    for h in hs:
        h.remove()
    assert rel(out.loss, o_loss) < (FP32_TOL if dtype == 'fp32' else 1e-2)
    check_grads(model, oracle, dtype)


@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
def test_mae_encoder_matches_oracle_at_visible_token_count(dtype):
    torch.manual_seed(8)
    oracle = OracleMaskedAutoencoder(OracleConfig(**CFG3), **DEC['golden']).train()
    model = EcgVitForMaskedAutoencoding(config=EcgVitConfig(compute_dtype=dtype, drop_path_rate=RATE, **CFG3),
                                        **DEC['golden'])
    model.load_state_dict(oracle.state_dict(), strict=True)
    model.cuda().train()
    x, _ = synthetic_batch(6, length=500, seed=14)
    out = model(x.cuda())
    out.loss.backward()
    assert model._engine._cur.N == MAE_N
    seed = int(model._engine.rng[0])
    assert_some_drop(seed, 3, 6)
    hs = inject_drop_path(oracle.vit.transformer, seed, RATE)   # the encoder only: the decoder never drops paths
    o_loss, _ = oracle(x, out.bool_masked_pos.cpu())
    o_loss.backward()
    for h in hs:
        h.remove()
    assert rel(out.loss, o_loss) < (FP32_TOL if dtype == 'fp32' else 1e-2)
    check_grads(model, oracle, dtype)


def test_eval_mode_is_bit_equal_to_rate_zero():
    torch.manual_seed(9)
    a = EcgVit(config=EcgVitConfig(compute_dtype='bf16', drop_path_rate=0.3, **CFG3)).cuda().eval()
    b = EcgVit(config=EcgVitConfig(compute_dtype='bf16', **CFG3))
    b.load_state_dict(a.state_dict())
    b.cuda().eval()
    x, _ = synthetic_batch(6, length=500, seed=15)
    with torch.no_grad():
        assert torch.equal(a(x.cuda()).logits, b(x.cuda()).logits)


@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
def test_activation_checkpointing_recomputes_the_same_blocks(dtype):
    """the recompute in backward reproduces every activation of the dropped / kept branches bit for bit (the keeps are a
    function of the step's seed); the loss is identical and the gradients agree up to the order of the split-K
    weight-gradient and bias column-sum atomics, which differs from run to run with or without checkpointing"""
    depth = 5
    cfg = dict(GOLDEN_CFG, num_hidden_layers=depth, hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1)
    torch.manual_seed(10)
    x, y = synthetic_batch(6, length=500, seed=16)
    base = EcgVit(config=EcgVitConfig(compute_dtype=dtype, drop_path_rate=RATE, **cfg)).state_dict()
    runs = []
    for ckpt in (False, True):
        m = EcgVit(config=EcgVitConfig(compute_dtype=dtype, drop_path_rate=RATE, activation_checkpointing=ckpt, **cfg))
        m.load_state_dict(base)
        m.cuda().train()
        out = m(sample_values=x.cuda(), labels=y.cuda())
        out.loss.backward()
        w = m._engine._cur
        assert w.ckpt == ckpt
        # with checkpointing, the two rotating activation sets end up holding the recompute of layers 0 and 1
        acts = [[t.clone() for t in (w.ln1[l], w.qkv[l], w.o[l], w.y[l], w.ln2[l], w.u[l], w.h[l])] for l in (0, 1)]
        runs.append((out.loss.clone(), [(k, p.grad.clone()) for k, p in m.named_parameters()], int(m._engine.rng[0]),
                     acts))
    seed = runs[0][2]
    assert runs[1][2] == seed
    a1, f1 = keeps(seed, depth, RATE, 6)[1]
    assert bool((a1 == 0).any() and (f1 == 0).any()), 'layer 1 must drop a record in both branches'
    assert torch.equal(runs[0][0], runs[1][0])
    for l in (0, 1):
        for t0, t1 in zip(runs[0][3][l], runs[1][3][l]):
            assert torch.equal(t0, t1), l
    tol = 1e-6 if dtype == 'fp32' else 1e-5
    for (k, g0), (_, g1) in zip(runs[0][1], runs[1][1]):
        assert rel(g1, g0) < tol, (k, rel(g1, g0))


def test_captured_trainer_tracks_oracle_and_rebuilds_on_rate_change():
    cfg = dict(CFG3, hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1)
    torch.manual_seed(11)
    oracle = OracleEcgVit(config=OracleConfig(**cfg)).train()
    model = EcgVit(config=EcgVitConfig(compute_dtype='fp32', drop_path_rate=RATE, **cfg))
    model.load_state_dict(oracle.state_dict(), strict=True)
    model.cuda().train()
    x, y = synthetic_batch(6, length=500, seed=17)
    ot = OracleTrainer(oracle, learning_rate=1e-3, weight_decay=1e-2)
    tr = FusedTrainer(model, learning_rate=1e-3, weight_decay=1e-2, max_grad_norm=1.0, use_cuda_graph=True)
    patterns = []
    for _ in range(3):
        loss, _ = tr.step(x.cuda(), y.cuda())
        seed = int(model._engine.rng[0])
        patterns.append(tuple(tuple(k.tolist()) for pair in keeps(seed, 3, RATE, 6) for k in pair))
        inject_dropout(oracle, seed, 0.1, 0.1)
        hs = inject_drop_path(oracle.vit.transformer, seed, RATE)
        o_loss, _, _ = ot.step(x, y)
        for h in hs:
            h.remove()
        assert rel(loss, o_loss) < FP32_TOL
    assert len(set(patterns)) == 3, 'every step must draw new keeps'
    for k, v in model.state_dict().items():
        assert rel(v, oracle.state_dict()[k]) < 2e-5, k
    graph = tr._graph
    model.config.drop_path_rate = 0.2
    tr.step(x.cuda(), y.cuda())
    assert tr._graph is not graph, 'a new drop_path_rate must rebuild the captured step'


def test_mae_encoder_fine_tunes_with_drop_path_mean_pool_and_lrd():
    """MAE pre-training -> encoder_state_dict() -> EcgVit(pool='mean', drop_path_rate=0.1) -> captured FusedTrainer
    steps with layer-wise LR decay, tracking the oracle with the same groups and injected keeps"""
    cfg = dict(CFG3)
    torch.manual_seed(21)
    pre = EcgVitForMaskedAutoencoding(EcgVitConfig(compute_dtype='fp32', drop_path_rate=0.1, **cfg),
                                      **DEC['golden']).cuda().train()
    x, y = synthetic_batch(6, length=cfg['max_signal_length'], seed=5)
    pt = FusedTrainer(pre, learning_rate=1e-3, data_parallel=False)
    for _ in range(2):
        pt.step(x.cuda())
    model = EcgVit(config=EcgVitConfig(compute_dtype='fp32', pool='mean', drop_path_rate=0.1, **cfg))
    missing, unexpected = model.load_state_dict(pre.encoder_state_dict(), strict=False)
    assert len(missing) == 4 and not unexpected
    oracle = OracleEcgVit(config=OracleConfig(**cfg)).train()
    oracle.vit.pool = 'mean'
    oracle.load_state_dict({k: v.cpu() for k, v in model.state_dict().items()}, strict=True)
    model.cuda().train()
    groups = param_groups_lrd(model, weight_decay=0.05, layer_decay=0.75)
    tr = FusedTrainer(model, learning_rate=1e-3, use_cuda_graph=True, data_parallel=False, param_groups=groups)
    ot = grouped_oracle_trainer(oracle, oracle_groups(oracle, groups, model, 1e-3), 1e-3, 'constant', 0, 1000)
    for _ in range(3):
        loss, _ = tr.step(x.cuda(), y.cuda())
        seed = int(model._engine.rng[0])
        hs = inject_drop_path(oracle.vit.transformer, seed, 0.1)
        o_loss, _, _ = ot.step(x, y)
        for h in hs:
            h.remove()
        assert rel(loss, o_loss) < FP32_TOL
    for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()):
        assert rel(p, q) < 2e-5, (k, rel(p, q))
