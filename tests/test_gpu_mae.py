"""GPU tier: MAE-style pre-training (EcgVitForMaskedAutoencoding) -- the index build, row gather, visible assemble and
unshuffle kernels against torch, and the whole forward / backward / training step against the CPU oracle
(oracle/mae_oracle.py) with the GPU's mask injected."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from conftest import GOLDEN_CFG
from ecg_b200 import EcgVitConfig, EcgVitForMaskedAutoencoding, FusedAdamW, FusedTrainer, MaskedPatchOutput, _lib
from oracle.ecg_vit_oracle import OracleConfig, synthetic_batch
from oracle.mae_oracle import OracleMaskedAutoencoder
from oracle.mpm_oracle import OracleMaskedPatchTrainer

from test_gpu_parity import rel, cosine, FP32_TOL, BF16_TOL, BF16_GRAD_COS
from test_gpu_pretrain import BENCH, PER_LEAD, PER_LEAD_SHORT

# decoder dims per geometry: head dim 16 at golden / per-lead-short, 64 (tcgen05 attention in bf16) at bench / per-lead
DEC = {'golden': dict(decoder_hidden_size=32, decoder_num_hidden_layers=2, decoder_num_attention_heads=2,
                      decoder_intermediate_size=64),
       'bench': dict(decoder_hidden_size=128, decoder_num_hidden_layers=2, decoder_num_attention_heads=2,
                     decoder_intermediate_size=256),
       'per_lead': dict(decoder_hidden_size=128, decoder_num_hidden_layers=2, decoder_num_attention_heads=2,
                        decoder_intermediate_size=256),
       'per_lead_short': dict(decoder_hidden_size=32, decoder_num_hidden_layers=2, decoder_num_attention_heads=2,
                              decoder_intermediate_size=64)}


def stream():
    return torch.cuda.current_stream().cuda_stream


def lib():
    return _lib.load()


def equal_count_mask(B, n, k, g, first_last=True):
    mask = torch.zeros(B, n, dtype=torch.bool, device='cuda')
    for b in range(B):
        mask[b, torch.randperm(n, device='cuda', generator=g)[:k]] = True
    if first_last and B >= 2:
        mask[0] = torch.arange(n, device='cuda') < k        # first patch masked
        mask[1] = torch.arange(n, device='cuda') >= n - k   # last patch masked
    return mask


def index_build(mask, n_vis):
    B, n = mask.shape
    vis = torch.full((B, n_vis), -7, device='cuda', dtype=torch.int32)
    slot = torch.full((B, n), -7, device='cuda', dtype=torch.int32)
    m8 = mask.to(torch.uint8).contiguous()
    _lib.check(lib().ecgvit_mae_index(m8.data_ptr(), B, n, n_vis, vis.data_ptr(), slot.data_ptr(), stream()))
    return vis, slot


# ---- kernels ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('n', [50, 2400])
def test_index_build_equals_nonzero(n):
    g = torch.Generator(device='cuda').manual_seed(1)
    B = 5
    for k in (1, n // 2, n - 1):
        mask = equal_count_mask(B, n, k, g)
        vis, slot = index_build(mask, n - k)
        for b in range(B):
            want = torch.nonzero(~mask[b]).flatten().to(torch.int32)
            assert torch.equal(vis[b], want), (n, k, b)
            s = torch.full((n,), -1, device='cuda', dtype=torch.int32)
            s[want.long()] = torch.arange(n - k, device='cuda', dtype=torch.int32)
            assert torch.equal(slot[b], s), (n, k, b)


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16])
def test_row_gather(dtype):
    g = torch.Generator(device='cuda').manual_seed(2)
    B, n, k, Kp = 4, 50, 38, 600
    src = torch.randn(B * n, Kp, device='cuda', generator=g).to(dtype)
    mask = equal_count_mask(B, n, k, g)
    vis, _ = index_build(mask, n - k)
    dst = torch.empty(B * (n - k), Kp, device='cuda', dtype=dtype)
    code = _lib.F32 if dtype == torch.float32 else _lib.BF16
    _lib.check(lib().ecgvit_row_gather(src.data_ptr(), dst.data_ptr(), vis.data_ptr(), B, n, n - k, Kp, code,
                                       stream()))
    want = torch.gather(src.view(B, n, Kp), 1, vis.long()[..., None].expand(-1, -1, Kp)).reshape(-1, Kp)
    assert torch.equal(dst, want)


def _visible_case(p, n):
    g = torch.Generator(device='cuda').manual_seed(3)
    B, k, d = 6, 3 * n // 4, 64
    nv = n - k
    mask = equal_count_mask(B, n, k, g)
    vis, slot = index_build(mask, nv)
    e = torch.randn(B * nv, d, device='cuda', generator=g)
    cls, pos = torch.randn(d, device='cuda', generator=g), torch.randn(n + 1, d, device='cuda', generator=g)
    seed = torch.tensor([4242, 0], device='cuda', dtype=torch.int32)
    keep = _lib.dropout_keep_mask(4242, 0, p, torch.arange(B * (nv + 1) * d)).view(B, nv + 1, d).cuda()
    return B, n, nv, d, vis, slot, e, cls, pos, seed, keep


@pytest.mark.parametrize('n', [40, 600])   # one / five chunks of the fixed-order bias fold
@pytest.mark.parametrize('p', [0.0, 0.1])
def test_visible_assemble_forward_backward_against_torch(p, n):
    B, n, nv, d, vis, slot, e, cls, pos, seed, keep = _visible_case(p, n)
    sp = seed.data_ptr() if p > 0 else None
    tok = torch.empty(B * (nv + 1), d, device='cuda')
    _lib.check(lib().ecgvit_embed_assemble_visible(e.data_ptr(), cls.data_ptr(), pos.data_ptr(), vis.data_ptr(),
                                                   tok.data_ptr(), B, nv, d, p, 0, sp, _lib.F32, stream()))
    body = e.view(B, nv, d) + pos[1 + vis.long()]
    want = torch.cat([(cls + pos[0]).expand(B, 1, d), body], 1) * keep
    if p == 0:
        assert torch.equal(tok.view(B, nv + 1, d), want)
    else:   # the same dropped elements; the kept ones scaled by the kernel's fp32 1 / (1 - p)
        assert torch.equal(tok.view(B, nv + 1, d) == 0, want == 0) and rel(tok.view(B, nv + 1, d), want) < 1e-6
    dtok = torch.randn(B * (nv + 1), d, device='cuda', generator=torch.Generator(device='cuda').manual_seed(5))
    outs = []
    for _ in range(2):
        de = torch.full((B * nv, d), 7.0, device='cuda')
        dcls, dpos, db = torch.zeros(d, device='cuda'), torch.zeros(n + 1, d, device='cuda'), torch.zeros(d, device='cuda')
        scratch = torch.empty(n * d, device='cuda')
        _lib.check(lib().ecgvit_embed_assemble_visible_bwd(dtok.data_ptr(), slot.data_ptr(), de.data_ptr(),
                                                           dcls.data_ptr(), dpos.data_ptr(), db.data_ptr(),
                                                           scratch.data_ptr(), B, n, nv, d, p, 0, sp, _lib.F32,
                                                           stream()), 'embed_assemble_visible_bwd')
        outs.append((de, dcls, dpos, db))
    for a, b in zip(*outs):
        assert torch.equal(a, b)   # fixed summation order: bit-identical launches
    de, dcls, dpos, db = outs[0]
    gt = dtok.view(B, nv + 1, d) * keep
    if p == 0:
        assert torch.equal(de.view(B, nv, d), gt[:, 1:])
    else:
        assert torch.equal(de.view(B, nv, d) == 0, gt[:, 1:] == 0) and rel(de.view(B, nv, d), gt[:, 1:]) < 1e-6
    want_pos = torch.zeros(n + 1, d, device='cuda', dtype=torch.float64)
    want_pos[0] = gt[:, 0].double().sum(0)
    want_pos.index_add_(0, (1 + vis.long()).flatten(), gt[:, 1:].double().reshape(-1, d))
    assert rel(dpos, want_pos) < 1e-6 and rel(dcls, gt[:, 0].double().sum(0)) < 1e-6
    assert rel(db, gt[:, 1:].double().sum((0, 1))) < 1e-6


@pytest.mark.parametrize('out_dtype', ['fp32', 'bf16_res32'])
def test_unshuffle_forward_backward_against_torch(out_dtype):
    g = torch.Generator(device='cuda').manual_seed(6)
    B, n, k, d = 5, 600, 450, 128   # five chunks of the fixed-order mask-token fold
    nv = n - k
    mask = equal_count_mask(B, n, k, g)
    vis, slot = index_build(mask, nv)
    T = torch.float32 if out_dtype == 'fp32' else torch.bfloat16
    code = _lib.F32 if out_dtype == 'fp32' else _lib.BF16_RES32
    t = torch.randn(B * (nv + 1), d, device='cuda', generator=g).to(T)
    mt, pos = torch.randn(d, device='cuda', generator=g), torch.randn(n + 1, d, device='cuda', generator=g)
    u = torch.empty(B * (n + 1), d, device='cuda')
    _lib.check(lib().ecgvit_mae_unshuffle(t.data_ptr(), mt.data_ptr(), pos.data_ptr(), slot.data_ptr(), u.data_ptr(), B,
                                          n, nv, d, code, stream()))
    tv = t.float().view(B, nv + 1, d)
    body = mt.expand(B, n, d).clone()
    body.scatter_(1, vis.long()[..., None].expand(-1, -1, d), tv[:, 1:])
    want = torch.cat([tv[:, :1], body], 1) + pos
    assert torch.equal(u.view(B, n + 1, d), want)
    if out_dtype != 'fp32':
        return
    du = torch.randn(B * (n + 1), d, device='cuda', generator=g)
    outs = []
    for _ in range(2):
        dt = torch.full((B * (nv + 1), d), 9.0, device='cuda')
        dpos, dmt, scratch = torch.zeros(n + 1, d, device='cuda'), torch.zeros(d, device='cuda'), torch.empty(n * d, device='cuda')
        _lib.check(lib().ecgvit_mae_unshuffle_bwd(du.data_ptr(), slot.data_ptr(), dt.data_ptr(), dpos.data_ptr(),
                                                  dmt.data_ptr(), scratch.data_ptr(), B, n, nv, d, _lib.F32, stream()),
                   'mae_unshuffle_bwd')
        outs.append((dt, dpos, dmt))
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    dt, dpos, dmt = outs[0]
    g3 = du.view(B, n + 1, d)
    want_dt = torch.cat([g3[:, :1], torch.gather(g3[:, 1:], 1, vis.long()[..., None].expand(-1, -1, d))], 1)
    assert torch.equal(dt.view(B, nv + 1, d), want_dt)
    assert rel(dpos, g3.double().sum(0)) < 1e-6
    assert rel(dmt, (g3[:, 1:].double() * mask[..., None]).sum((0, 1))) < 1e-6


# ---- whole model against the oracle ----------------------------------------------------------------------------
def make(cfg, dec, dtype, batch, seed=77, mask_ratio=0.75, **kw):
    torch.manual_seed(seed)
    oracle = OracleMaskedAutoencoder(OracleConfig(**cfg), **dec).train()
    with torch.no_grad():   # non-zero mask token and LayerNorm weights, so their gradients are exercised
        oracle.decoder.mask_token.normal_()
        oracle.recon_head[0].weight.add_(0.1 * torch.randn_like(oracle.recon_head[0].weight))
        oracle.decoder.norm.weight.add_(0.1 * torch.randn_like(oracle.decoder.norm.weight))
    model = EcgVitForMaskedAutoencoding(config=EcgVitConfig(compute_dtype=dtype, **cfg, **kw), mask_ratio=mask_ratio,
                                        **dec)
    model.load_state_dict(oracle.state_dict(), strict=True)
    model.cuda().train()
    x, _ = synthetic_batch(batch, num_channels=cfg['num_channels'], length=cfg['max_signal_length'], seed=seed)
    return oracle, model, x


def check_grads(model, oracle, dtype):
    worst = 0.0
    for (k, p), (_, q) in zip(model.named_parameters(), oracle.named_parameters()):
        if dtype == 'fp32':
            e = rel(p.grad, q.grad)
            worst = max(worst, e)
            assert e < FP32_TOL, (k, e)
        else:
            assert cosine(p.grad, q.grad) > BF16_GRAD_COS, (k, cosine(p.grad, q.grad))
    return worst


@pytest.mark.parametrize('geometry,dtype', [(g, t) for g in ('golden', 'bench', 'per_lead_short') for t in ('fp32', 'bf16')]
                         + [('per_lead', 'bf16'), ('golden_res32', 'bf16')])
def test_forward_backward_against_oracle(geometry, dtype):
    cfg, batch = {'golden': (GOLDEN_CFG, 4), 'bench': (BENCH, 2), 'per_lead': (PER_LEAD, 2),
                  'per_lead_short': (PER_LEAD_SHORT, 3), 'golden_res32': (GOLDEN_CFG, 4)}[geometry]
    kw = dict(residual_dtype='fp32') if geometry == 'golden_res32' else {}
    dec = DEC[geometry.replace('_res32', '')]
    oracle, model, x = make(cfg, dec, dtype, batch, **kw)
    out = model(x.cuda())
    assert isinstance(out, MaskedPatchOutput)
    n = model.vit.pos_embedding.shape[1] - 1
    k = round(0.75 * n)
    assert out.bool_masked_pos.shape == (batch, n) and (out.bool_masked_pos.sum(1) == k).all()
    assert model._engine._cur.N == n - k + 1 and model._engine._cur.dec.N == n + 1
    out.loss.backward()
    o_loss, o_pred = oracle(x, out.bool_masked_pos.cpu())
    o_loss.backward()
    tol = FP32_TOL if dtype == 'fp32' else BF16_TOL
    assert rel(out.loss, o_loss) < tol and rel(out.reconstruction, o_pred) < tol
    worst = check_grads(model, oracle, dtype)
    print(f'{geometry}/{dtype}: encoder N {n - k + 1} decoder N {n + 1}: loss rel {rel(out.loss, o_loss):.2e} '
          f'recon rel {rel(out.reconstruction, o_pred):.2e} worst grad rel {worst:.2e}')


def test_user_mask_counts_eval_mask_and_fresh_training_masks():
    oracle, model, x = make(GOLDEN_CFG, DEC['golden'], 'fp32', 3)
    mask = torch.zeros(3, 10, dtype=torch.bool)
    mask[0, [0, 5, 9]] = True
    mask[1, [2, 3, 4]] = True
    mask[2, [1, 7, 8]] = True
    out = model(x.cuda(), bool_masked_pos=mask.cuda())
    assert torch.equal(out.bool_masked_pos.cpu(), mask)
    out.loss.backward()
    o_loss, o_pred = oracle(x, mask)
    o_loss.backward()
    assert rel(out.loss, o_loss) < FP32_TOL and rel(out.reconstruction, o_pred) < FP32_TOL
    check_grads(model, oracle, 'fp32')
    bad = mask.clone()
    bad[2, 1] = False
    with pytest.raises(ValueError, match='same number'):
        model(x.cuda(), bool_masked_pos=bad.cuda())
    with pytest.raises(ValueError, match='same number'):
        model(x.cuda(), bool_masked_pos=torch.zeros(3, 10, dtype=torch.bool, device='cuda'))
    model.eval()
    with torch.no_grad():
        a, b = model(x.cuda()), model(x.cuda())
    assert torch.equal(a.bool_masked_pos, b.bool_masked_pos) and torch.equal(a.loss, b.loss)
    model.train()
    with torch.no_grad():
        c, d = model(x.cuda()), model(x.cuda())
    assert not torch.equal(c.bool_masked_pos, d.bool_masked_pos)


def test_encoder_activation_checkpointing_gives_identical_results():
    cfg = dict(GOLDEN_CFG, num_hidden_layers=4, hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1)
    runs = []
    for ckpt in (False, True):
        _, model, x = make(cfg, DEC['golden'], 'fp32', 4, activation_checkpointing=ckpt)
        model._prepare(x.cuda().device)
        model._engine.base_seed = 11
        out = model(x.cuda())
        out.loss.backward()
        assert model._engine._cur.ckpt == ckpt and not model._engine._cur.dec.ckpt
        runs.append((out.loss.clone(), out.bool_masked_pos, [p.grad.clone() for p in model.parameters()]))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    for a, b in zip(runs[0][2], runs[1][2]):
        assert rel(a, b) < 1e-6


def test_fused_adamw_through_the_autograd_bridge():
    oracle, model, x = make(GOLDEN_CFG, DEC['golden'], 'fp32', 4)
    opt = FusedAdamW(model, lr=1e-3, weight_decay=1e-2)
    oopt = torch.optim.AdamW(oracle.parameters(), lr=1e-3, weight_decay=1e-2)
    out = model(x.cuda())
    out.loss.backward()
    opt.step()
    o_loss, _ = oracle(x, out.bool_masked_pos.cpu())
    o_loss.backward()
    oopt.step()
    for k, v in model.state_dict().items():
        assert rel(v, oracle.state_dict()[k]) < FP32_TOL, k


@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
def test_three_captured_trainer_steps_track_the_oracle_trainer(dtype):
    oracle, model, x = make(GOLDEN_CFG, DEC['golden'], dtype, 4, seed=5)
    ot = OracleMaskedPatchTrainer(oracle, learning_rate=1e-3, max_grad_norm=1.0)
    tr = FusedTrainer(model, learning_rate=1e-3, max_grad_norm=1.0, use_cuda_graph=True)
    xc = x.cuda()
    masks = []
    for _ in range(3):
        loss, second = tr.step(xc)
        assert second is None
        mask = model._engine.mask().cpu()
        masks.append(mask)
        o_loss, _, o_norm = ot.step(x, mask)
        tol = FP32_TOL if dtype == 'fp32' else BF16_TOL
        assert rel(loss, o_loss) < tol, (dtype, rel(loss, o_loss))
        assert abs(tr.grad_norm() - float(o_norm)) < (1e-4 if dtype == 'fp32' else 2e-2) * float(o_norm)
    assert not torch.equal(masks[0], masks[1])   # every replay draws a new mask
    tr.check_finite()
    if dtype == 'fp32':
        for k, v in model.state_dict().items():
            assert rel(v, oracle.state_dict()[k]) < FP32_TOL, k
    sd = tr.state_dict()
    tr2 = FusedTrainer(model, learning_rate=1e-3, max_grad_norm=1.0)
    tr2.load_state_dict(sd)
    assert tr2.step_count == 3 and torch.equal(tr2.exp_avg, tr.exp_avg)
    tr.use_cuda_graph = False
    loss, _ = tr.step(xc)
    assert torch.isfinite(loss)


def test_deferred_optimizer_ends_equal_to_the_immediate_update():
    _, m_now, x = make(GOLDEN_CFG, DEC['golden'], 'fp32', 4, seed=8)
    _, m_def, _ = make(GOLDEN_CFG, DEC['golden'], 'fp32', 4, seed=8)
    kw = dict(learning_rate=1e-3, max_grad_norm=0.05, use_cuda_graph=True)
    t_now, t_def = FusedTrainer(m_now, **kw), FusedTrainer(m_def, defer_optimizer=True, **kw)
    xc = x.cuda()
    for _ in range(3):
        l_now, _ = t_now.step(xc)
        l_def, _ = t_def.step(xc)
        assert torch.equal(m_now._engine.mask(), m_def._engine.mask())
        assert rel(l_def, l_now) < 1e-6
    t_def.flush()
    assert rel(m_def._flat_p, m_now._flat_p) < 1e-6
