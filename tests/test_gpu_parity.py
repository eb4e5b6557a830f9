"""GPU tier: the whole hot path (forward, backward, clip + AdamW, 3 steps) against the CPU oracle and the committed
golden vectors.  Tolerances are BASELINE.json's: fp32 logits/loss <= 1e-5 relative; bf16 <= 1e-2 relative with
per-parameter gradient cosine >= 0.999; patch indexing bit-exact (test_gpu_kernels.py)."""
import numpy as np
import pytest
import torch
from torch import nn

pytestmark = pytest.mark.gpu

from conftest import GOLDEN_CFG, golden_sample
import ecg_b200
from ecg_b200 import EcgVit, EcgVitConfig, FusedTrainer, FusedAdamW, clip_grad_norm_
from oracle.ecg_vit_oracle import OracleConfig, OracleEcgVit, OracleTrainer, synthetic_batch

FP32_TOL = 1e-5       # north_star: fp32 logits and loss within 1e-5 relative
BF16_TOL = 1e-2       # north_star: bf16 within 1e-2 relative
BF16_GRAD_COS = 0.999  # north_star: per-parameter gradient cosine


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def cosine(a, b):
    a, b = a.detach().double().cpu().flatten(), b.detach().double().cpu().flatten()
    return float((a @ b) / (a.norm() * b.norm()).clamp_min(1e-300))


def make_pair(cfg, dtype, batch, seed=77, length=None):
    torch.manual_seed(seed)
    oracle = OracleEcgVit(config=OracleConfig(**cfg)).train()
    model = EcgVit(config=EcgVitConfig(compute_dtype=dtype, **cfg))
    model.load_state_dict(oracle.state_dict(), strict=True)
    model.cuda().train()
    x, y = synthetic_batch(batch, length=length or cfg['max_signal_length'], seed=seed)
    return oracle, model, x, y


def golden_model(golden, dtype):
    model = EcgVit(config=EcgVitConfig(compute_dtype=dtype, **GOLDEN_CFG))
    model.load_state_dict({k[5:]: torch.from_numpy(v) for k, v in golden.items() if k.startswith('init/')}, strict=True)
    return model.cuda().train()


# ---- golden vectors (generated through the reference's own wrapper) ------------------------------------------
def test_fp32_matches_golden_forward_backward(golden):
    model = golden_model(golden, 'fp32')
    x, y = torch.from_numpy(golden['x']).cuda(), torch.from_numpy(golden['y']).cuda()
    out = model(sample_values=x, labels=y)
    assert isinstance(out, ecg_b200.ModelOutput)
    out.loss.backward()
    assert rel(out.logits, torch.from_numpy(golden['logits'])) < FP32_TOL
    assert abs(float(out.loss) - float(golden['loss'])) < FP32_TOL * float(golden['loss'])
    for k, p in model.named_parameters():
        got, g = golden_sample(p.grad), torch.from_numpy(golden['grad/' + k])
        assert rel(got, g) < 2e-4, (k, rel(got, g))
        assert cosine(got, g) > 0.999999, k


def test_fp32_matches_golden_three_steps(golden):
    model = golden_model(golden, 'fp32')
    x, y = torch.from_numpy(golden['x']).cuda(), torch.from_numpy(golden['y']).cuda()
    tr = FusedTrainer(model, learning_rate=3e-4, weight_decay=1e-2, schedule='constant', max_grad_norm=1.0)
    for step in (1, 2, 3):
        loss, _ = tr.step(x, y)
        assert abs(float(loss) - float(golden[f'loss{step}'])) < FP32_TOL * float(golden[f'loss{step}'])
        assert abs(tr.grad_norm() - float(golden[f'norm{step}'])) < 1e-4 * float(golden[f'norm{step}'])
        if step in (1, 3):
            for k, v in model.state_dict().items():
                got = golden_sample(v) if step == 1 else v
                assert rel(got, torch.from_numpy(golden[f'step{step}/' + k])) < FP32_TOL, (step, k)
    tr.check_finite()


def test_eval_loss_none_matches_golden(golden):
    model = EcgVit(config=EcgVitConfig(compute_dtype='fp32', **GOLDEN_CFG), loss_reduction='none')
    model.load_state_dict({k[6:]: torch.from_numpy(v) for k, v in golden.items() if k.startswith('step3/')}, strict=True)
    model.cuda().eval()
    with torch.no_grad():
        out = model(torch.from_numpy(golden['x']).cuda(), torch.from_numpy(golden['y']).cuda())
    assert out.loss.shape == (4, 71)
    assert rel(out.loss, torch.from_numpy(golden['eval_loss_none'])) < FP32_TOL
    assert rel(out.logits, torch.from_numpy(golden['eval_logits'])) < FP32_TOL
    assert model(torch.from_numpy(golden['x']).cuda()).loss is None


# ---- oracle on the same seeded inputs -------------------------------------------------------------------------
CFG1 = dict(max_signal_length=2500, patch_size=50, num_channels=12, hidden_size=256, num_hidden_layers=4,
            num_attention_heads=8, intermediate_size=1024, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
CFG_MID = dict(max_signal_length=2500, patch_size=50, num_channels=12, hidden_size=384, num_hidden_layers=3,
               num_attention_heads=6, intermediate_size=1536, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
CFG_REFDEFAULT = dict(max_signal_length=2560, patch_size=64, num_channels=12, hidden_size=128, num_hidden_layers=2,
                      num_attention_heads=4, intermediate_size=512, hidden_dropout_prob=0.0,
                      attention_probs_dropout_prob=0.0)


@pytest.mark.parametrize('cfg,batch', [(CFG1, 8), (CFG_REFDEFAULT, 5)])
def test_fp32_parity_with_oracle_cfg1(cfg, batch):
    """cfg1 of BASELINE.json (d=256, 4 layers, 8 heads, patch 50, 12x2500) and the reference's default 2560/64 geometry"""
    oracle, model, x, y = make_pair(cfg, 'fp32', batch)
    o = oracle(sample_values=x, labels=y)
    o.loss.backward()
    out = model(sample_values=x.cuda(), labels=y.cuda())
    out.loss.backward()
    assert rel(out.logits, o.logits) < FP32_TOL and rel(out.loss, o.loss) < FP32_TOL
    for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()):
        assert rel(p.grad, q.grad) < 5e-4, (k, rel(p.grad, q.grad))
        assert cosine(p.grad, q.grad) > 0.99999, k


def test_fp32_three_steps_with_clipping_active():
    oracle, model, x, y = make_pair(CFG_REFDEFAULT, 'fp32', 6, seed=5)
    ot = OracleTrainer(oracle, learning_rate=1e-3, weight_decay=1e-2, schedule='cosine', n_warmup=1, n_step=3,
                       max_grad_norm=0.05)
    tr = FusedTrainer(model, learning_rate=1e-3, weight_decay=1e-2, schedule='cosine', n_warmup=1, n_step=3,
                      max_grad_norm=0.05)
    for _ in range(3):
        o_loss, _, o_norm = ot.step(x, y)
        loss, _ = tr.step(x.cuda(), y.cuda())
        assert float(o_norm) > 0.05, 'test must exercise the clip'
        assert rel(loss, o_loss) < FP32_TOL and abs(tr.grad_norm() - float(o_norm)) < 1e-4 * float(o_norm)
    for k, v in model.state_dict().items():
        assert rel(v, oracle.state_dict()[k]) < FP32_TOL, k


def test_shorter_signal_uses_pos_embedding_slice():
    """vit_pytorch slices pos_embedding[:, :n+1], so inputs shorter than max_signal_length are legal"""
    oracle, model, x, y = make_pair(CFG_REFDEFAULT, 'fp32', 3, length=1280)
    o = oracle(sample_values=x, labels=y)
    out = model(sample_values=x.cuda(), labels=y.cuda())
    assert rel(out.logits, o.logits) < FP32_TOL
    o.loss.backward()
    out.loss.backward()
    g, go = model.vit.pos_embedding.grad, oracle.vit.pos_embedding.grad
    assert rel(g, go) < 1e-4 and float(g[0, 21:].abs().max()) == 0.0


@pytest.mark.parametrize('cfg,batch', [(CFG1, 16), (CFG_MID, 8), (GOLDEN_CFG, 4)])
def test_bf16_parity_with_oracle(cfg, batch):
    oracle, model, x, y = make_pair(cfg, 'bf16', batch)
    o = oracle(sample_values=x, labels=y)
    o.loss.backward()
    out = model(sample_values=x.cuda(), labels=y.cuda())
    out.loss.backward()
    assert rel(out.logits, o.logits) < BF16_TOL, rel(out.logits, o.logits)
    assert rel(out.loss, o.loss) < BF16_TOL
    worst = min((cosine(p.grad, q.grad), k) for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()))
    assert worst[0] >= BF16_GRAD_COS, worst


# bf16 tolerance: 1e-2 (north_star) for every named size.  Up to 12 layers the residual stream is stored in bf16; its
# rounding error random-walks with depth, so deeper models ('large': 24 layers) keep the stream in fp32
# (EcgVitConfig.residual_dtype = 'auto'; ECGVIT_BF16_RES32 / ECGVIT_EPI_BIAS_RES_F32 in the C ABI).
@pytest.mark.parametrize('size,batch,tol', [('debug', 6, BF16_TOL), ('tiny', 4, BF16_TOL), ('small', 3, BF16_TOL),
                                            ('base', 3, BF16_TOL), ('large', 2, BF16_TOL)])
def test_named_sizes_reference_geometry(size, batch, tol):
    """the reference's own named sizes at its default geometry (12 x 2560, patch 64 -> 41 tokens; ecg_vit.py:31-32,56-92);
    'large' is BASELINE.json configs[4]'s model (d=1024, 24 layers, 16 heads)"""
    torch.manual_seed(1)
    oc = OracleConfig.from_defined(f'ecg-vit-{size}')
    oc.hidden_dropout_prob = oc.attention_probs_dropout_prob = 0.0
    oracle = OracleEcgVit(config=oc).train()
    conf = EcgVitConfig.from_defined(f'ecg-vit-{size}')
    conf.hidden_dropout_prob = conf.attention_probs_dropout_prob = 0.0
    model = EcgVit(config=conf)
    assert model.to_str() == f'EcgVit, {size}'
    assert model._res_f32 == (size == 'large')
    model.load_state_dict(oracle.state_dict(), strict=True)
    model.cuda().train()
    x, y = synthetic_batch(batch, length=2560, seed=21)
    o = oracle(sample_values=x, labels=y)
    o.loss.backward()
    out = model(sample_values=x.cuda(), labels=y.cuda())
    out.loss.backward()
    assert rel(out.logits, o.logits) < tol, rel(out.logits, o.logits)
    assert rel(out.loss, o.loss) < BF16_TOL
    worst = min((cosine(p.grad, q.grad), k) for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()))
    assert worst[0] >= BF16_GRAD_COS, worst


def test_bf16_three_steps_track_the_oracle():
    oracle, model, x, y = make_pair(CFG1, 'bf16', 16)
    ot, tr = OracleTrainer(oracle), FusedTrainer(model)
    for _ in range(3):
        o_loss, _, o_norm = ot.step(x, y)
        loss, _ = tr.step(x.cuda(), y.cuda())
        assert rel(loss, o_loss) < BF16_TOL
        assert abs(tr.grad_norm() - float(o_norm)) < 3e-2 * float(o_norm)
    tr.check_finite()
    # the bf16 shadow the next forward reads is exactly the rounded fp32 master
    assert torch.equal(model._shadow, model._flat_p.bfloat16())


# ---- reference-style loop through the drop-in API ---------------------------------------------------------------
def test_reference_style_loop_equals_fused_step():
    """zero_grad / model(**inputs) / loss.backward() / clip_grad_norm_ / optimizer.step() / scheduler.step()
    (train.py:271-283) through the nn.Module API gives the same parameters as FusedTrainer.step"""
    from transformers import get_cosine_schedule_with_warmup
    _, m1, x, y = make_pair(GOLDEN_CFG, 'fp32', 4)
    _, m2, _, _ = make_pair(GOLDEN_CFG, 'fp32', 4)
    inputs = dict(sample_values=x.cuda(), labels=y.cuda())
    opt = FusedAdamW(m1, lr=3e-4, weight_decay=1e-2)
    sch = get_cosine_schedule_with_warmup(opt, num_warmup_steps=1, num_training_steps=4)
    tr = FusedTrainer(m2, learning_rate=3e-4, weight_decay=1e-2, schedule='cosine', n_warmup=1, n_step=4)
    for _ in range(3):
        opt.zero_grad()
        out = m1(**inputs)
        loss, logits = out  # tuple-unpack like EcgVitTrainModule (train.py:49)
        loss.backward()
        clip_grad_norm_(m1, max_norm=1.0, error_if_nonfinite=True)
        opt.step()
        sch.step()
        tr.step(**inputs)
    for (k, a), (_, b) in zip(m1.state_dict().items(), m2.state_dict().items()):
        assert rel(a, b) < 1e-6, k


def test_stock_torch_optimizer_also_works_and_shadow_follows():
    """a user may keep torch.optim.AdamW + nn.utils.clip_grad_norm_: parameters stay views of the flat buffer and the
    bf16 shadow is refreshed when their version counters move"""
    oracle, model, x, y = make_pair(GOLDEN_CFG, 'bf16', 4)
    opt = torch.optim.AdamW(model.parameters(), lr=1e-2, weight_decay=1e-2)
    for _ in range(2):
        opt.zero_grad()
        model(sample_values=x.cuda(), labels=y.cuda()).loss.backward()
        nn.utils.clip_grad_norm_(model.parameters(), 1.0, error_if_nonfinite=True)
        opt.step()
    out = model(sample_values=x.cuda(), labels=y.cuda())
    assert torch.equal(model._shadow, model._flat_p.bfloat16())
    oracle.load_state_dict(model.state_dict())
    assert rel(out.logits, oracle(x, y).logits) < BF16_TOL


def test_gradient_accumulation_semantics():
    _, model, x, y = make_pair(GOLDEN_CFG, 'fp32', 4)
    inputs = dict(sample_values=x.cuda(), labels=y.cuda())
    model(**inputs).loss.backward()
    g1 = [p.grad.clone() for p in model.parameters()]
    model(**inputs).loss.backward()  # no zero_grad in between: autograd semantics are "accumulate"
    for p, g in zip(model.parameters(), g1):
        assert rel(p.grad, 2 * g) < 1e-5


def test_cuda_graph_step_matches_eager_step():
    _, m1, x, y = make_pair(GOLDEN_CFG, 'bf16', 4)
    _, m2, _, _ = make_pair(GOLDEN_CFG, 'bf16', 4)
    t1, t2 = FusedTrainer(m1, use_cuda_graph=False), FusedTrainer(m2, use_cuda_graph=True)
    xs, ys = x.cuda(), y.cuda()
    for i in range(4):
        xi = xs * (1.0 + 0.1 * i)
        l1, _ = t1.step(xi, ys)
        l2, _ = t2.step(xi, ys)
        assert abs(float(l1) - float(l2)) < 1e-3 * abs(float(l1))  # fp32 atomics reorder between runs
    assert rel(m2._flat_p, m1._flat_p) < 1e-4


# ---- full-size properties (cfg2 geometry; the oracle would take minutes on CPU) -----------------------------------
def test_base_model_full_batch_properties():
    cfg = dict(max_signal_length=2500, patch_size=50, num_channels=12, hidden_size=768, num_hidden_layers=12,
               num_attention_heads=12, intermediate_size=3072, hidden_dropout_prob=0.0,
               attention_probs_dropout_prob=0.0)
    torch.manual_seed(0)
    model = EcgVit(config=EcgVitConfig(compute_dtype='bf16', **cfg)).cuda().train()
    x, y = synthetic_batch(256)
    x, y = x.cuda(), y.cuda()
    with torch.no_grad():
        full = model(sample_values=x, labels=y).logits
        # samples are independent: any sub-batch reproduces its rows of the full-batch logits
        part = model(sample_values=x[64:96], labels=y[64:96]).logits
        # permutation equivariance over the batch
        perm = torch.randperm(256, device='cuda')
        shuf = model(sample_values=x[perm], labels=y[perm]).logits
    assert rel(part, full[64:96]) < 2e-3
    assert rel(shuf, full[perm]) < 2e-3
    # a training step leaves everything finite and moves the loss down on the same batch
    tr = FusedTrainer(model, learning_rate=3e-4)
    l0 = float(tr.step(x, y)[0])
    for _ in range(4):
        l = float(tr.step(x, y)[0])
    tr.check_finite()
    assert np.isfinite(l) and l < l0
    assert torch.equal(model._shadow, model._flat_p.bfloat16())


# ---- Recorder slow path + checkpoint round trip (SURVEY 8f rank 3) ---------------------------------------------------
@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
def test_recorder_attention_maps_match_oracle(dtype):
    from oracle.vit_restated import Recorder as OracleRecorder
    oracle, model, x, _ = make_pair(GOLDEN_CFG, dtype, 2)
    oracle.eval(), model.eval()
    rec_o = OracleRecorder(oracle.vit)
    with torch.no_grad():
        want_logits, want_attn = rec_o(x.unsqueeze(-2))                 # the call of ecg_vit.py:177-179
    rec_o.eject()
    rec = ecg_b200.Recorder(model.vit)
    logits, attn = rec(x.cuda().unsqueeze(-2))
    assert attn.shape == want_attn.shape                                # (b, layers, heads, n, n)
    tol = FP32_TOL if dtype == 'fp32' else BF16_TOL
    assert rel(attn, want_attn) < tol and rel(logits, want_logits) < tol
    assert float((attn.sum(-1) - 1).abs().max()) < 1e-5
    # the roll-out of EcgVitVisualizer.__call__ (ecg_vit.py:184-193) on top of both
    def rollout(a):
        a = a[0].double().cpu().mean(dim=0)
        a = a + torch.eye(a.size(1), dtype=a.dtype)
        a = a / a.sum(dim=-1, keepdim=True)
        res = torch.empty_like(a)
        res[0] = a[0]
        for i in range(1, a.size(0)):
            res[i] = a[i] @ a[i - 1]
        res = res[:, 0, 1:]
        return res / res.max()
    assert rel(rollout(attn), rollout(want_attn)) < tol
    assert rec.eject() is model.vit
    with pytest.raises(AssertionError):
        rec(x.cuda().unsqueeze(-2))
    out = model(sample_values=x.cuda())                                 # the fused path is untouched afterwards
    assert rel(out.logits, want_logits) < tol


def test_reference_format_checkpoint_round_trip(tmp_path):
    """train.py:297-300 saves `model.state_dict()`; ecg_vit.py:152-161 loads it with strict=True"""
    oracle, model, x, y = make_pair(GOLDEN_CFG, 'fp32', 2)
    path = tmp_path / 'model - reference format.pt'
    torch.save(oracle.state_dict(), path)                               # what the reference trainer writes
    fresh = EcgVit(config=EcgVitConfig(compute_dtype='fp32', **GOLDEN_CFG))
    fresh.load_state_dict(torch.load(path, map_location='cpu'), strict=True)
    fresh.cuda().eval()
    oracle.eval()
    with torch.no_grad():
        want = oracle(sample_values=x, labels=y)
    got = fresh(sample_values=x.cuda(), labels=y.cuda())
    assert rel(got.logits, want.logits) < FP32_TOL
    # and back: a checkpoint written by the fused model (after a fused step) loads into the reference-side module
    tr = FusedTrainer(fresh.train(), use_cuda_graph=False, data_parallel=False)
    tr.step(x.cuda(), y.cuda())
    path2 = tmp_path / 'model - fused.pt'
    torch.save(fresh.state_dict(), path2)
    sd = torch.load(path2, map_location='cpu')
    assert list(sd.keys()) == list(oracle.state_dict().keys())
    oracle.load_state_dict(sd, strict=True)
    oracle.eval(), fresh.eval()
    with torch.no_grad():
        want = oracle(sample_values=x, labels=y)
    got = fresh(sample_values=x.cuda(), labels=y.cuda())
    assert rel(got.logits, want.logits) < FP32_TOL


@pytest.mark.parametrize('reduction', ['mean', 'none'])
def test_loss_weight_matches_reference_formula(reduction):
    """ecg_vit.py:144-147: BCEWithLogitsLoss(weight=tensor(loss_weight)[labels.long()], reduction)"""
    oracle, model, x, y = make_pair(GOLDEN_CFG, 'fp32', 4)
    lw = [0.25, 4.0]
    model.loss_weight = lw
    model.loss_reduction = reduction
    out = model(sample_values=x.cuda(), labels=y.cuda())
    with torch.no_grad():
        logits = oracle(sample_values=x).logits
    want = nn.BCEWithLogitsLoss(weight=torch.tensor(lw)[y.long()], reduction=reduction)(input=logits, target=y)
    assert rel(out.loss, want) < FP32_TOL
    if reduction == 'mean':
        out.loss.backward()
        oracle.zero_grad()
        lo = oracle(sample_values=x).logits
        nn.BCEWithLogitsLoss(weight=torch.tensor(lw)[y.long()])(input=lo, target=y).backward()
        for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()):
            assert rel(p.grad, q.grad) < 2e-4 and cosine(p.grad, q.grad) > 0.999999, k
        # the fused trainer picks the table up too (and re-captures when it changes)
        tr = FusedTrainer(model, use_cuda_graph=True, data_parallel=False)
        l1 = float(tr.step(x.cuda(), y.cuda())[0])   # the returned tensors are views of workspace buffers
        assert abs(l1 - float(want)) < FP32_TOL * float(want)
        model.loss_weight = None
        l2 = float(tr.step(x.cuda(), y.cuda())[0])
        assert abs(l2 - l1) > 0.1 * l1


def test_resume_from_saved_optimizer_state_and_fused_train_step():
    """SURVEY 8f rank 4: model + FusedTrainer state saved after 2 steps, loaded into fresh objects, 2 more steps ==
    4 uninterrupted steps (cosine schedule with warm-up and dropout on, so step counter, moments and the dropout
    stream all matter)"""
    cfg = dict(GOLDEN_CFG, hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1)
    kw = dict(learning_rate=1e-3, weight_decay=1e-2, schedule='cosine', n_warmup=2, n_step=8, use_cuda_graph=True,
              data_parallel=False)
    _, m_ref, x, y = make_pair(cfg, 'fp32', 4)
    _, m_a, _, _ = make_pair(cfg, 'fp32', 4)
    xs, ys = x.cuda(), y.cuda()
    t_ref, t_a = FusedTrainer(m_ref, **kw), FusedTrainer(m_a, **kw)
    for _ in range(4):
        t_ref.step(xs, ys)
    for _ in range(2):
        t_a.step(xs, ys)
    saved = {'model': {k: v.cpu() for k, v in m_a.state_dict().items()},
             'trainer': {k: (v.cpu() if torch.is_tensor(v) else v) for k, v in t_a.state_dict().items()}}
    m_b = EcgVit(config=EcgVitConfig(compute_dtype='fp32', **cfg))
    m_b.load_state_dict(saved['model'], strict=True)
    m_b.cuda().train()
    t_b = FusedTrainer(m_b, **kw)
    t_b.load_state_dict(saved['trainer'])
    for _ in range(2):
        t_b.step(xs, ys)
    assert t_b.step_count == 4
    assert rel(m_b._flat_p, m_ref._flat_p) < 1e-5
    assert rel(t_b.exp_avg_sq, t_ref.exp_avg_sq) < 1e-4
    # without the optimizer state the run diverges visibly (what the reference's model-only checkpoint gives)
    m_c = EcgVit(config=EcgVitConfig(compute_dtype='fp32', **cfg))
    m_c.load_state_dict(saved['model'], strict=True)
    m_c.cuda().train()
    t_c = FusedTrainer(m_c, **kw)
    for _ in range(2):
        t_c.step(xs, ys)
    assert rel(m_c._flat_p, m_ref._flat_p) > 10 * rel(m_b._flat_p, m_ref._flat_p)
    # the functional entry point of SURVEY 8b
    out = ecg_b200.fused_train_step(m_c, dict(sample_values=x, labels=y), lr=1e-3)
    assert isinstance(out, ecg_b200.ModelOutput) and out.logits.shape == (4, 71) and float(out.loss) > 0


@pytest.mark.parametrize('cfg,batch', [(CFG1, 8), (CFG_MID, 4)])
def test_fp32_residual_stream_mode_matches_oracle(cfg, batch):
    """residual_dtype='fp32' forced on small models: forward, backward and three fused steps (CUDA graph)"""
    torch.manual_seed(77)
    oracle = OracleEcgVit(config=OracleConfig(**cfg)).train()
    model = EcgVit(config=EcgVitConfig(compute_dtype='bf16', residual_dtype='fp32', **cfg))
    model.load_state_dict(oracle.state_dict(), strict=True)
    model.cuda().train()
    assert model._res_f32
    x, y = synthetic_batch(batch, length=cfg['max_signal_length'])
    o = oracle(sample_values=x, labels=y)
    o.loss.backward()
    out = model(sample_values=x.cuda(), labels=y.cuda())
    out.loss.backward()
    assert model._engine._cur.x[0].dtype == torch.float32 and model._engine._cur.ln1[0].dtype == torch.bfloat16
    assert rel(out.logits, o.logits) < BF16_TOL and rel(out.loss, o.loss) < BF16_TOL
    worst = min((cosine(p.grad, q.grad), k) for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()))
    assert worst[0] >= BF16_GRAD_COS, worst
    # same model with the bf16 stream: the fp32 stream must not be further from the oracle
    model16 = EcgVit(config=EcgVitConfig(compute_dtype='bf16', residual_dtype='bf16', **cfg))
    model16.load_state_dict(oracle.state_dict(), strict=True)
    model16.cuda().train()
    out16 = model16(sample_values=x.cuda(), labels=y.cuda())
    assert rel(out.logits, o.logits) <= 1.5 * rel(out16.logits, o.logits) + 1e-4
    oracle.zero_grad()
    ot, tr = OracleTrainer(oracle), FusedTrainer(model, use_cuda_graph=True, data_parallel=False)
    for _ in range(3):
        o_loss, _, o_norm = ot.step(x, y)
        loss, _ = tr.step(x.cuda(), y.cuda())
        assert rel(loss, o_loss) < BF16_TOL
    tr.check_finite()


def test_fp32_residual_stream_with_dropout_masks():
    """the fp32-stream epilogue applies the same counter-based dropout as the bf16 one"""
    from test_gpu_dropout import inject
    cfg = dict(CFG_MID, hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1)
    torch.manual_seed(5)
    oracle = OracleEcgVit(config=OracleConfig(**cfg)).train()
    model = EcgVit(config=EcgVitConfig(compute_dtype='bf16', residual_dtype='fp32', **cfg))
    model.load_state_dict(oracle.state_dict(), strict=True)
    model.cuda().train()
    x, y = synthetic_batch(4, length=cfg['max_signal_length'], seed=3)
    got = model(sample_values=x.cuda(), labels=y.cuda())
    got.loss.backward()
    inject(oracle, int(model._engine.rng[0]), cfg['attention_probs_dropout_prob'], cfg['hidden_dropout_prob'])
    want = oracle(sample_values=x, labels=y)
    want.loss.backward()
    assert rel(got.logits, want.logits) < BF16_TOL
    for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()):
        assert cosine(p.grad, q.grad) > BF16_GRAD_COS, (k, cosine(p.grad, q.grad))


@pytest.mark.parametrize('p_drop,res', [(0.0, 'bf16'), (0.1, 'bf16'), (0.1, 'fp32')])
def test_activation_checkpointing_reproduces_the_stored_activation_step(p_drop, res):
    """BASELINE.json configs[4] asks for activation checkpointing: with `activation_checkpointing=True` only the block
    inputs are kept and every block is recomputed in backward (dropout masks regenerate from the counter).  Same loss,
    same gradients (up to the order of the split-K red.adds), same three optimisation steps as the default path, and
    still inside the bf16 bar against the oracle."""
    cfg = dict(CFG_MID, num_hidden_layers=5, hidden_dropout_prob=p_drop, attention_probs_dropout_prob=p_drop)
    torch.manual_seed(77)
    oracle = OracleEcgVit(config=OracleConfig(**cfg)).train()
    models = []
    for ckpt in (False, True):
        m = EcgVit(config=EcgVitConfig(compute_dtype='bf16', residual_dtype=res, activation_checkpointing=ckpt, **cfg))
        m.load_state_dict(oracle.state_dict(), strict=True)
        m.cuda().train()
        m._prepare(torch.device('cuda', torch.cuda.current_device()))
        models.append(m)
    x, y = synthetic_batch(6, length=cfg['max_signal_length'])
    xd, yd = x.cuda(), y.cuda()
    outs = []
    for m in models:
        m._engine.new_dropout_seed(seed=4242)
        loss, logits = m._engine.forward(xd, yd, 'mean')
        loss, logits = loss.clone(), logits.clone()
        m._engine.backward()
        outs.append((loss, logits, m._flat_g.clone()))
    assert models[1]._engine._cur.ckpt and not models[0]._engine._cur.ckpt
    assert models[1]._engine._cur.ln1[0] is models[1]._engine._cur.ln1[2]          # shared buffer sets
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    assert rel(outs[1][2], outs[0][2]) < 1e-5
    if p_drop == 0.0:
        o = oracle(sample_values=x, labels=y)
        assert rel(outs[1][1], o.logits) < BF16_TOL
    trainers = [FusedTrainer(m, use_cuda_graph=True, data_parallel=False) for m in models]
    for step in range(3):
        for m, tr in zip(models, trainers):
            m._engine._seed_counter = 100 + step          # both draw the same masks
            tr.step(xd, yd)
    assert rel(models[1]._flat_p, models[0]._flat_p) < 1e-6
