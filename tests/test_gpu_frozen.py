"""GPU tier: frozen parameters (requires_grad=False) -- linear probing and partial fine-tuning.  The fused trainer and the
autograd loop against the CPU oracle with the same flags, the truncated backward against the full one, the kernels a
frozen prefix no longer runs, the lean activation workspace, gradual unfreezing, save / resume, and the pre-training
models."""
import re

import pytest
import torch

pytestmark = pytest.mark.gpu

from conftest import GOLDEN_CFG
from ecg_b200 import (EcgVit, EcgVitConfig, EcgVitForMaskedAutoencoding, FusedAdamW, FusedTrainer, clip_grad_norm_,
                      param_groups_lrd)
from oracle.ecg_vit_oracle import OracleConfig, OracleEcgVit, OracleTrainer, lr_lambda, synthetic_batch

from test_gpu_parity import rel, FP32_TOL
from test_gpu_pretrain import BENCH, PER_LEAD, PER_LEAD_SHORT

CFG3 = dict(GOLDEN_CFG, num_hidden_layers=3)
EMBEDDING = ('vit.to_patch_embedding.', 'vit.pos_embedding', 'vit.cls_token', 'vit.mask_token')
MAE_DEC = dict(decoder_hidden_size=64, decoder_num_hidden_layers=2, decoder_num_attention_heads=2,
               decoder_intermediate_size=128)


def block_of(name):
    return int(name.split('.')[3]) if name.startswith('vit.transformer.layers.') else None


def freeze(model, pattern):
    """head_only: the linear probe; last: the last block and the head (MAE's partial fine-tuning with k = 1); prefix:
    the embedding and the lower half of the blocks; pos: the positional table; qkv: one block's to_qkv weight"""
    depth = model.config.num_hidden_layers
    for name, p in model.named_parameters():
        b = block_of(name)
        frozen = {'head_only': name.startswith('vit.') and not name.startswith('vit.mlp_head.'),
                  'last': name.startswith(EMBEDDING) or (b is not None and b < depth - 1),
                  'prefix': name.startswith(EMBEDDING) or (b is not None and b < depth // 2),
                  'pos': name == 'vit.pos_embedding',
                  'qkv': name == 'vit.transformer.layers.1.0.fn.to_qkv.weight',
                  'none': False}[pattern]
        p.requires_grad_(not frozen)
    return model


def make_pair(cfg, pattern, seed=77, batch=4):
    torch.manual_seed(seed)
    oracle = OracleEcgVit(config=OracleConfig(**cfg)).train()
    model = EcgVit(config=EcgVitConfig(compute_dtype='fp32', **cfg))
    model.load_state_dict(oracle.state_dict(), strict=True)
    freeze(model, pattern).cuda().train()
    flags = {n: p.requires_grad for n, p in model.named_parameters()}
    for n, p in oracle.named_parameters():
        p.requires_grad_(flags[n])
    x, y = synthetic_batch(batch, num_channels=cfg['num_channels'], length=cfg['max_signal_length'], seed=seed)
    return oracle, model, x, y


def assert_frozen_untouched(model, start, moments=()):
    for key, (o, n, _, name) in model._layout.items():
        p = dict(model.named_parameters())[name]
        if p.requires_grad:
            continue
        assert torch.equal(model._flat_p[o:o + n].cpu(), start[name].reshape(-1)), name
        for m in moments:
            assert not bool(m[o:o + n].any()), name


# ---- 1. the fused trainer against the oracle --------------------------------------------------------------------------
@pytest.mark.parametrize('mode', ['eager', 'graph'])
@pytest.mark.parametrize('pattern', ['head_only', 'last', 'pos', 'qkv', 'lrd'])
def test_trainer_with_frozen_tensors_tracks_the_oracle(pattern, mode):
    oracle, model, x, y = make_pair(CFG3, 'prefix' if pattern == 'lrd' else pattern)
    start = {n: p.detach().cpu().clone() for n, p in model.named_parameters()}
    kw = dict(learning_rate=1e-3, weight_decay=1e-2, schedule='cosine', n_warmup=1, n_step=3, max_grad_norm=0.05)
    if pattern == 'lrd':
        groups = param_groups_lrd(model, weight_decay=0.05, layer_decay=0.75)
        tr = FusedTrainer(model, use_cuda_graph=mode == 'graph', data_parallel=False, param_groups=groups, **kw)
        names = {id(p): n for n, p in model.named_parameters()}
        op = dict(oracle.named_parameters())
        ogroups = [{'params': [op[names[id(p)]] for p in g['params']], 'lr': 1e-3 * g['lr_scale'],
                    'weight_decay': g['weight_decay']} for g in groups]
        ot = OracleTrainer(oracle, max_grad_norm=0.05)
        ot.optimizer = torch.optim.AdamW(ogroups, lr=1e-3)
        ot.scheduler = torch.optim.lr_scheduler.LambdaLR(ot.optimizer, lambda s: lr_lambda('cosine', s, 1, 3))
    else:
        tr = FusedTrainer(model, use_cuda_graph=mode == 'graph', data_parallel=False, **kw)
        ot = OracleTrainer(oracle, **kw)
    for _ in range(3):
        o_loss, _, o_norm = ot.step(x, y)
        loss, _ = tr.step(x.cuda(), y.cuda())
        # clipping is active: a frozen gradient leaking into the norm would change every update
        assert float(o_norm) > 0.05, 'test must exercise the clip'
        assert rel(loss, o_loss) < FP32_TOL
        assert abs(tr.grad_norm() - float(o_norm)) < 1e-4 * float(o_norm), (tr.grad_norm(), float(o_norm))
    tr.check_finite()
    for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()):
        assert rel(p, q) < FP32_TOL, (k, rel(p, q))
    assert_frozen_untouched(model, start, (tr.exp_avg, tr.exp_avg_sq))


def test_nothing_to_train_and_deferred_optimizer_raise():
    _, model, x, y = make_pair(GOLDEN_CFG, 'head_only')
    with pytest.raises(ValueError, match='defer_optimizer'):
        FusedTrainer(model, defer_optimizer=True).step(x.cuda(), y.cuda())
    for p in model.parameters():
        p.requires_grad_(False)
    with pytest.raises(ValueError, match='nothing to train'):
        FusedTrainer(model).step(x.cuda(), y.cuda())


# ---- 2. truncated backward == full backward on the trainable tensors ---------------------------------------------------
def engine_grads(model, x, y, seed):
    eng = model._engine
    eng.upload_seed(seed, 1)
    if isinstance(model, EcgVitForMaskedAutoencoding):
        eng.forward(x)
    else:
        eng.forward(x, y, 'mean')
    eng.backward()
    torch.cuda.synchronize()
    return {k: v.clone() for k, v in model._grads_f32().items()}


def check_truncated_equals_full(model, x, y, patterns):
    model.cuda().train()
    model._prepare(x.device)
    full = engine_grads(model, x, y, 4321)
    for pattern in patterns:
        freeze(model, pattern)
        part = engine_grads(model, x, y, 4321)
        frozen = model.trainable_span().frozen
        for k, g in part.items():
            if k in frozen or model.trainable_span().lo > model._layout[k][0]:
                continue
            # the only difference is the order of the split-K / column-sum atomics
            assert rel(g, full[k]) < 1e-5, (pattern, k, rel(g, full[k]))
    freeze(model, 'none')


@pytest.mark.parametrize('ckpt', [False, True])
@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
@pytest.mark.parametrize('geometry', ['bench', 'per_lead'])
def test_truncated_backward_equals_full_backward(geometry, dtype, ckpt):
    # per-lead in fp32: the short geometry (the fp32 attention holds the whole sequence in shared memory)
    per_lead = PER_LEAD if dtype == 'bf16' else PER_LEAD_SHORT
    cfg, batch = {'bench': (BENCH, 16), 'per_lead': (dict(per_lead, num_hidden_layers=4), 4)}[geometry]
    cfg = dict(cfg, hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1)
    torch.manual_seed(5)
    model = EcgVit(config=EcgVitConfig(compute_dtype=dtype, drop_path_rate=0.1, activation_checkpointing=ckpt, **cfg))
    x, y = synthetic_batch(batch, num_channels=cfg['num_channels'], length=cfg['max_signal_length'], seed=5)
    check_truncated_equals_full(model, x.cuda(), y.cuda(), ['last', 'prefix', 'qkv', 'pos'])


def test_mae_frozen_encoder_prefix_matches_full_backward():
    cfg = dict(GOLDEN_CFG, num_hidden_layers=4, hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1)
    torch.manual_seed(6)
    model = EcgVitForMaskedAutoencoding(EcgVitConfig(compute_dtype='bf16', drop_path_rate=0.1, **cfg), **MAE_DEC)
    x, _ = synthetic_batch(8, length=cfg['max_signal_length'], seed=6)
    check_truncated_equals_full(model, x.cuda(), None, ['prefix', 'last', 'head_only'])


# ---- 3. kernels a frozen prefix no longer runs -----------------------------------------------------------------------
BWD_RE = re.compile(r'attn_tc_bwd|attn_tc_dot|attn_tc_dq|attention_bwd|flash_bwd|layernorm_bwd')   # per block
COPY_RE = re.compile(r'dropout_bwd')   # the masked copies (the top block's gradient, from the head)
WGRAD_RE = re.compile(r'gemm_tc2_kernel<\s*\d+\s*,\s*(true|false)\s*,\s*(true|false)\s*,\s*4\s*,')


def captured_step_kernels(pattern):
    cfg = dict(GOLDEN_CFG, num_hidden_layers=4, hidden_size=256, num_attention_heads=8, intermediate_size=1024,
               hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1)
    torch.manual_seed(7)
    model = freeze(EcgVit(config=EcgVitConfig(compute_dtype='bf16', **cfg)), pattern).cuda().train()
    x, y = synthetic_batch(64, length=cfg['max_signal_length'], seed=7)
    tr = FusedTrainer(model, use_cuda_graph=True, data_parallel=False)
    tr.step(x.cuda(), y.cuda())
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        tr.step(x.cuda(), y.cuda())
        torch.cuda.synchronize()
    return [e.name for e in prof.events()], tr.launches_per_step


def test_frozen_prefix_runs_no_encoder_backward_kernels():
    full, n_full = captured_step_kernels('none')
    last, n_last = captured_step_kernels('last')
    probe, n_probe = captured_step_kernels('head_only')
    count = lambda names, rx: sum(1 for n in names if rx.search(n))
    assert count(full, BWD_RE) > 0 and count(full, WGRAD_RE) >= 4 * 4   # four per block (and the embedding's)
    assert count(probe, BWD_RE) == 0 and count(probe, WGRAD_RE) == 0 and count(probe, COPY_RE) == 0
    # exactly one block's backward
    assert count(last, BWD_RE) * 4 == count(full, BWD_RE)
    assert count(last, WGRAD_RE) == 4
    assert n_probe < n_last < n_full


# ---- 4. the lean activation workspace --------------------------------------------------------------------------------
def test_head_only_workspace_saves_the_frozen_block_sets():
    cfg, B = BENCH, 256
    d, mlp, H, depth = cfg['hidden_size'], cfg['intermediate_size'], cfg['num_attention_heads'], cfg['num_hidden_layers']
    x, y = synthetic_batch(B, seed=8)
    x, y = x.cuda(), y.cuda()
    used = {}
    for pattern in ('none', 'head_only'):
        torch.manual_seed(8)
        model = freeze(EcgVit(config=EcgVitConfig(compute_dtype='bf16', **cfg)), pattern).cuda().train()
        model._prepare(x.device)
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        model._engine.forward(x, y, 'mean')
        torch.cuda.synchronize()
        used[pattern] = torch.cuda.memory_allocated() - before
        del model
        torch.cuda.empty_cache()
    N = cfg['max_signal_length'] // cfg['patch_size'] + 1
    M = B * N
    # one block's activation set (_alloc_stack): ln1, ln2, o, y, qkv, u, h in bf16, the row statistics and lse in fp32
    block_set = 2 * M * (4 * d + 3 * d + 2 * mlp) + 4 * (4 * M + B * H * N)
    assert used['none'] - used['head_only'] >= (depth - 1) * block_set, (used, block_set)


# ---- 5. the autograd path ------------------------------------------------------------------------------------------
def test_autograd_loop_with_frozen_prefix_tracks_torch_adamw():
    oracle, model, x, y = make_pair(CFG3, 'prefix')
    start = {n: p.detach().cpu().clone() for n, p in model.named_parameters()}
    opt = FusedAdamW(model, lr=2e-3, weight_decay=1e-2)
    oopt = torch.optim.AdamW(oracle.parameters(), lr=2e-3, weight_decay=1e-2)
    for step in range(3):
        opt.zero_grad()
        model(x.cuda(), y.cuda()).loss.backward()
        norm = clip_grad_norm_(model, max_norm=0.05)
        oopt.zero_grad()
        oracle(x, y).loss.backward()
        o_norm = torch.nn.utils.clip_grad_norm_(oracle.parameters(), max_norm=0.05)
        assert abs(float(norm) - float(o_norm)) < 1e-4 * float(o_norm)
        for n, p in model.named_parameters():
            assert (p.grad is None) == (not p.requires_grad), n
        if step == 2:
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                opt.step()
                torch.cuda.synchronize()
            names = [e.name for e in prof.events()]
            # the frozen slices are left out by the group map: no device-to-device copies, no copy kernels
            assert not any('DtoD' in n or 'copy_kernel' in n for n in names), names
        else:
            opt.step()
        oopt.step()
    for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()):
        assert rel(p, q) < FP32_TOL, (k, rel(p, q))
    assert_frozen_untouched(model, start, (opt._m, opt._v))


# ---- 6. gradual unfreezing ----------------------------------------------------------------------------------------
def test_unfreezing_mid_run_recaptures_and_trains_the_new_tensors():
    _, model, x, y = make_pair(CFG3, 'head_only')
    tr = FusedTrainer(model, learning_rate=1e-3, use_cuda_graph=True, data_parallel=False)
    for _ in range(2):
        tr.step(x.cuda(), y.cuda())
    g1, n1 = tr._graph, tr.launches_per_step
    top = model.vit.transformer.layers[2]
    before = {n: p.detach().clone() for n, p in top.named_parameters()}
    for p in top.parameters():
        p.requires_grad_(True)
    tr.step(x.cuda(), y.cuda())
    torch.cuda.synchronize()
    assert tr._graph is not g1 and tr.launches_per_step > n1
    for n, p in top.named_parameters():
        assert not torch.equal(p.detach(), before[n]), n
    assert not any(p.requires_grad for p in model.vit.transformer.layers[0].parameters())


# ---- 7. save and resume ---------------------------------------------------------------------------------------------
def test_save_resume_with_frozen_prefix_continues_the_run(tmp_path):
    _, m_ref, x, y = make_pair(CFG3, 'last')
    _, m_a, _, _ = make_pair(CFG3, 'last')
    kw = dict(learning_rate=1e-3, schedule='cosine', n_warmup=1, n_step=4, data_parallel=False)
    t_ref, t_a = FusedTrainer(m_ref, **kw), FusedTrainer(m_a, **kw)
    xs, ys = x.cuda(), y.cuda()
    for _ in range(4):
        t_ref.step(xs, ys)
    for _ in range(2):
        t_a.step(xs, ys)
    t_a.save(str(tmp_path), 'mid')
    _, m_b, _, _ = make_pair(CFG3, 'last', seed=99)
    t_b = FusedTrainer(m_b, **kw)
    t_b.resume(str(tmp_path), 'mid')
    for _ in range(2):
        t_b.step(xs, ys)
    assert rel(m_b._flat_p, m_ref._flat_p) < 1e-5
    assert rel(t_b.exp_avg_sq, t_ref.exp_avg_sq) < 1e-4
    lo = m_b.trainable_span().lo
    assert torch.equal(m_b._flat_p[:lo], m_ref._flat_p[:lo])


# ---- 8. pre-trained encoder, linear probe ------------------------------------------------------------------------------
def test_mae_encoder_linear_probe_keeps_the_encoder_bit_identical():
    cfg = dict(GOLDEN_CFG, num_hidden_layers=3)
    torch.manual_seed(9)
    pre = EcgVitForMaskedAutoencoding(EcgVitConfig(compute_dtype='bf16', **cfg), **MAE_DEC).cuda().train()
    x, y = synthetic_batch(8, length=cfg['max_signal_length'], seed=9)
    FusedTrainer(pre, learning_rate=1e-3, use_cuda_graph=True).step(x.cuda())
    enc = {k: v.detach().clone() for k, v in pre.encoder_state_dict().items()}
    probe = EcgVit(config=EcgVitConfig(compute_dtype='bf16', pool='mean', **cfg))
    missing = probe.load_state_dict(enc, strict=False).missing_keys
    assert all(k.startswith('vit.mlp_head.') for k in missing)
    freeze(probe, 'head_only').cuda().train()
    head0 = probe.vit.mlp_head[1].weight.detach().clone()
    tr = FusedTrainer(probe, learning_rate=1e-3, use_cuda_graph=True, param_groups=param_groups_lrd(probe))
    for _ in range(3):
        tr.step(x.cuda(), y.cuda())
    tr.check_finite()
    for k, v in probe.state_dict().items():
        if k in enc:
            assert torch.equal(v, enc[k]), k
    assert not torch.equal(probe.vit.mlp_head[1].weight.detach(), head0)
