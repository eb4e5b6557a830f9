"""GPU tier: masked-patch pre-training (EcgVitForMaskedPatchModeling) -- the mask draw bit-exact against its host
replica, the new kernels against torch, the row-square GEMM epilogue, and the whole forward / backward / training step
against the CPU oracle (oracle/mpm_oracle.py) with the GPU's mask injected."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from conftest import GOLDEN_CFG
from ecg_b200 import (EcgVitConfig, EcgVitForMaskedPatchModeling, FusedAdamW, FusedTrainer, MaskedPatchOutput, _lib)
from oracle.ecg_vit_oracle import OracleConfig, synthetic_batch
from oracle.mpm_oracle import OracleMaskedPatchModel, OracleMaskedPatchTrainer

from test_gpu_parity import rel, cosine, FP32_TOL, BF16_TOL, BF16_GRAD_COS

BENCH = dict(max_signal_length=2500, patch_size=50, num_channels=12, hidden_size=768, num_hidden_layers=12,
             num_attention_heads=12, intermediate_size=3072, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
PER_LEAD = dict(max_signal_length=500, patch_size=25, num_channels=12, hidden_size=128, num_hidden_layers=2,
                num_attention_heads=2, intermediate_size=128, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0,
                per_lead_tokens=True)   # N = 12 * 20 + 1 = 241, patch_dim 25 -> padded to 32
# fp32 parity mode keeps whole sequences in shared memory (N = 241 does not fit): per-lead tokens at N = 37
PER_LEAD_SHORT = dict(PER_LEAD, max_signal_length=300, num_channels=3, hidden_size=64, num_attention_heads=4)


def stream():
    return torch.cuda.current_stream().cuda_stream


def lib():
    return _lib.load()


# ---- kernels ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('n', [50, 2400])
def test_mask_kernel_matches_host_replica(n):
    B, site = 6, 49
    seed = torch.tensor([123457, 0], device='cuda', dtype=torch.int32)
    for k in (1, n - 1, n // 2):
        mask = torch.zeros(B * n, device='cuda', dtype=torch.uint8)
        counts = torch.zeros(B, device='cuda', dtype=torch.int32)
        _lib.check(lib().ecgvit_mpm_mask(seed.data_ptr(), B, n, k, site, mask.data_ptr(), counts.data_ptr(), stream()))
        want = _lib.mpm_mask(123457, B, n, k, site)
        assert torch.equal(mask.view(B, n).bool().cpu(), want), (n, k)
        assert counts.cpu().tolist() == [k] * B
    # a caller's mask is only counted
    user = torch.rand(B, n, device='cuda') < 0.3
    mask = user.to(torch.uint8).reshape(-1).contiguous()
    _lib.check(lib().ecgvit_mpm_mask(None, B, n, 0, site, mask.data_ptr(), counts.data_ptr(), stream()))
    assert counts.cpu().tolist() == user.sum(1).cpu().tolist()
    assert torch.equal(mask.view(B, n).bool(), user)


def test_masked_assemble_forward_backward_against_torch():
    B, n, d = 3, 10, 64
    g = torch.Generator(device='cuda').manual_seed(1)
    e = torch.randn(B * n, d, device='cuda', generator=g)
    cls, pos = torch.randn(d, device='cuda', generator=g), torch.randn(n + 1, d, device='cuda', generator=g)
    mt = torch.randn(d, device='cuda', generator=g)
    m = torch.rand(B, n, device='cuda', generator=g) < 0.5
    mask = m.to(torch.uint8).reshape(-1).contiguous()
    tok = torch.empty(B * (n + 1), d, device='cuda')
    _lib.check(lib().ecgvit_embed_assemble_masked(e.data_ptr(), cls.data_ptr(), pos.data_ptr(), mt.data_ptr(),
                                                  mask.data_ptr(), tok.data_ptr(), B, n, d, 0.0, 0, None, _lib.F32,
                                                  stream()))
    ew = torch.where(m[..., None], mt.expand(B, n, d), e.view(B, n, d))
    want = torch.cat([cls.expand(B, 1, d), ew], 1) + pos
    assert torch.equal(tok.view(B, n + 1, d), want)
    dtok = torch.randn(B * (n + 1), d, device='cuda', generator=g)
    de = torch.full((B * n, d), 7.0, device='cuda')
    dcls, dpos, db, dmt = (torch.zeros(d, device='cuda'), torch.zeros(n + 1, d, device='cuda'),
                           torch.zeros(d, device='cuda'), torch.zeros(d, device='cuda'))
    _lib.check(lib().ecgvit_embed_assemble_masked_bwd(dtok.data_ptr(), mask.data_ptr(), de.data_ptr(), dcls.data_ptr(),
                                                      dpos.data_ptr(), db.data_ptr(), dmt.data_ptr(), B, n, d, 0.0, 0,
                                                      None, _lib.F32, stream()))
    gt = dtok.view(B, n + 1, d)
    gp = gt[:, 1:]
    assert torch.equal(de.view(B, n, d), torch.where(m[..., None], torch.zeros_like(gp), gp))
    torch.testing.assert_close(dpos, gt.sum(0), rtol=1e-6, atol=1e-5)
    torch.testing.assert_close(dcls, gt[:, 0].sum(0), rtol=1e-6, atol=1e-5)
    torch.testing.assert_close(db, (gp * (~m)[..., None]).sum((0, 1)), rtol=1e-6, atol=1e-5)
    torch.testing.assert_close(dmt, (gp * m[..., None]).sum((0, 1)), rtol=1e-6, atol=1e-5)


@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
def test_patch_row_layernorm_forward_backward_against_torch(dtype):
    B, n, d = 4, 50, 768
    code, T = (_lib.F32, torch.float32) if dtype == 'fp32' else (_lib.BF16, torch.bfloat16)
    tol = dict(rtol=1e-5, atol=1e-5) if dtype == 'fp32' else dict(rtol=2e-2, atol=2e-2)
    g = torch.Generator(device='cuda').manual_seed(2)
    tok = torch.randn(B * (n + 1), d, device='cuda', generator=g).to(T)
    gamma, beta = 1 + 0.1 * torch.randn(d, device='cuda', generator=g), 0.1 * torch.randn(d, device='cuda', generator=g)
    y = torch.empty(B * n, d, device='cuda', dtype=T)
    st = torch.empty(2, B * n, device='cuda')
    _lib.check(lib().ecgvit_layernorm_patch_fwd(tok.data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(),
                                                st[0].data_ptr(), st[1].data_ptr(), B, n, d, 1e-5, code, stream()))
    xp = tok.float().view(B, n + 1, d)[:, 1:].reshape(B * n, d).requires_grad_(True)
    gm, bt = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    ref = torch.nn.functional.layer_norm(xp, (d,), gm, bt, 1e-5)
    torch.testing.assert_close(y.float(), ref, **tol)
    dy = torch.randn(B * n, d, device='cuda', generator=g).to(T)
    ref.backward(dy.float())
    dtok = torch.full((B * (n + 1), d), 3.0, device='cuda', dtype=T)
    dgam, dbet, dcol = torch.zeros(d, device='cuda'), torch.zeros(d, device='cuda'), torch.zeros(d, device='cuda')
    scratch = torch.empty(int(lib().ecgvit_layernorm_bwd_scratch_floats(d)), device='cuda')
    _lib.check(lib().ecgvit_layernorm_patch_bwd(dy.data_ptr(), tok.data_ptr(), gamma.data_ptr(), st[0].data_ptr(),
                                                st[1].data_ptr(), dtok.data_ptr(), dgam.data_ptr(), dbet.data_ptr(),
                                                dcol.data_ptr(), scratch.data_ptr(), B, n, d, code, stream()))
    dt = dtok.float().view(B, n + 1, d)
    assert float(dt[:, 0].abs().max()) == 0.0
    torch.testing.assert_close(dt[:, 1:].reshape(B * n, d), xp.grad, **tol)
    torch.testing.assert_close(dgam, gm.grad, **tol)
    torch.testing.assert_close(dbet, bt.grad, **tol)
    # the column sums are taken before dtok is rounded to dtype
    torch.testing.assert_close(dcol, xp.grad.sum(0), rtol=1e-4, atol=1e-3 if dtype == 'fp32' else 0.2)


@pytest.mark.parametrize('dtype', ['fp32', 'bf16'])
@pytest.mark.parametrize('N', [600, 32])
def test_row_square_epilogue_against_torch(dtype, N):
    M, K = 1000, 768
    code, T = (_lib.F32, torch.float32) if dtype == 'fp32' else (_lib.BF16, torch.bfloat16)
    g = torch.Generator(device='cuda').manual_seed(3)
    A = torch.randn(M, K, device='cuda', generator=g).to(T)
    W = (torch.randn(N, K, device='cuda', generator=g) / K ** 0.5).to(T)
    bias = torch.randn(N, device='cuda', generator=g)
    tgt = torch.randn(M, N, device='cuda', generator=g).to(T)
    out = torch.empty(M, N, device='cuda', dtype=T)
    G = (N + 63) // 64
    rowsq = torch.empty(G, M, device='cuda')
    eng_args = lambda: _lib.GemmArgs(M, N, K, A.data_ptr(), K, 1, W.data_ptr(), K, 1, _lib.EPI_BIAS_SUB_ROWSQ,
                                     out.data_ptr(), N, rowsq.data_ptr(), tgt.data_ptr(), bias.data_ptr(), code, 1, 0,
                                     0.0, None)
    import ctypes
    _lib.check(lib().ecgvit_gemm(ctypes.byref(eng_args()), stream()), 'gemm')
    r = A.float() @ W.float().t() + bias - tgt.float()
    tol = dict(rtol=1e-5, atol=1e-4) if dtype == 'fp32' else dict(rtol=2e-2, atol=3e-2)
    torch.testing.assert_close(out.float(), r, **tol)
    want = torch.stack([(r[:, 64 * i:64 * (i + 1)] ** 2).sum(1) for i in range(G)])
    torch.testing.assert_close(rowsq, want, rtol=1e-4 if dtype == 'fp32' else 2e-2, atol=1e-3)
    # the loss fold is bit-identical from launch to launch
    mask = (torch.rand(M, device='cuda', generator=g) < 0.5).to(torch.uint8)
    counts = torch.tensor([int(mask.sum())], device='cuda', dtype=torch.int32)
    losses = []
    for _ in range(2):
        _lib.check(lib().ecgvit_gemm(ctypes.byref(eng_args()), stream()), 'gemm')
        loss, cnt = torch.zeros(1, device='cuda'), torch.zeros(1, device='cuda')
        _lib.check(lib().ecgvit_mpm_loss(rowsq.data_ptr(), G, mask.data_ptr(), counts.data_ptr(), 1, M, N,
                                         loss.data_ptr(), cnt.data_ptr(), stream()))
        losses.append(loss.clone())
    assert torch.equal(losses[0], losses[1])
    want_loss = (r[mask.bool()] ** 2).sum() / (float(mask.sum()) * N)
    assert rel(losses[0], want_loss.reshape(1)) < (1e-5 if dtype == 'fp32' else 2e-2)


# ---- whole model against the oracle ----------------------------------------------------------------------------
def make(cfg, dtype, batch, seed=77, **kw):
    torch.manual_seed(seed)
    oracle = OracleMaskedPatchModel(OracleConfig(**cfg)).train()
    with torch.no_grad():   # a non-zero mask token and recon LayerNorm, so their gradients are exercised
        oracle.vit.mask_token.normal_()
        oracle.recon_head[0].weight.add_(0.1 * torch.randn_like(oracle.recon_head[0].weight))
    model = EcgVitForMaskedPatchModeling(config=EcgVitConfig(compute_dtype=dtype, **cfg, **kw))
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
    # golden_res32: bf16 with the fp32 residual stream (the token matrix the assembly writes and the recon LayerNorm
    # reads is fp32)
    kw = dict(residual_dtype='fp32') if geometry == 'golden_res32' else {}
    oracle, model, x = make(cfg, dtype, batch, **kw)
    assert model._res_f32 == (geometry == 'golden_res32')
    out = model(x.cuda())
    assert isinstance(out, MaskedPatchOutput)
    n = model.vit.pos_embedding.shape[1] - 1
    assert out.bool_masked_pos.shape == (batch, n) and (out.bool_masked_pos.sum(1) == round(0.5 * n)).all()
    out.loss.backward()
    o_loss, o_pred = oracle(x, out.bool_masked_pos.cpu())
    o_loss.backward()
    tol = FP32_TOL if dtype == 'fp32' else BF16_TOL
    assert rel(out.loss, o_loss) < tol and rel(out.reconstruction, o_pred) < tol
    worst = check_grads(model, oracle, dtype)
    print(f'{geometry}/{dtype}: loss rel {rel(out.loss, o_loss):.2e} recon rel {rel(out.reconstruction, o_pred):.2e} '
          f'worst grad rel {worst:.2e}')


def test_user_mask_with_unequal_counts_and_eval_mask_is_fixed():
    oracle, model, x = make(GOLDEN_CFG, 'fp32', 3)
    mask = torch.zeros(3, 10, dtype=torch.bool)
    mask[0, [0, 5, 9]] = True
    mask[1, 2] = True
    mask[2, :8] = True
    out = model(x.cuda(), bool_masked_pos=mask.cuda())
    assert torch.equal(out.bool_masked_pos.cpu(), mask)
    out.loss.backward()
    o_loss, o_pred = oracle(x, mask)
    o_loss.backward()
    assert rel(out.loss, o_loss) < FP32_TOL and rel(out.reconstruction, o_pred) < FP32_TOL
    check_grads(model, oracle, 'fp32')
    model.eval()
    with torch.no_grad():
        a, b = model(x.cuda()), model(x.cuda())
    assert torch.equal(a.bool_masked_pos, b.bool_masked_pos) and torch.equal(a.loss, b.loss)
    model.train()
    with torch.no_grad():
        c, d = model(x.cuda()), model(x.cuda())
    assert not torch.equal(c.bool_masked_pos, d.bool_masked_pos)   # a fresh mask every training forward


def test_activation_checkpointing_gives_identical_gradients():
    """same masks, same dropout, same forward; gradients equal up to the order of the split-K weight-gradient adds"""
    cfg = dict(GOLDEN_CFG, num_hidden_layers=4, hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1)
    runs = []
    for ckpt in (False, True):
        _, model, x = make(cfg, 'fp32', 4, activation_checkpointing=ckpt)
        model._prepare(x.cuda().device)
        model._engine.base_seed = 11
        out = model(x.cuda())
        out.loss.backward()
        runs.append((out.loss.clone(), out.bool_masked_pos, [p.grad.clone() for p in model.parameters()]))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    for a, b in zip(runs[0][2], runs[1][2]):
        assert rel(a, b) < 1e-6


def test_fused_adamw_through_the_autograd_bridge():
    oracle, model, x = make(GOLDEN_CFG, 'fp32', 4)
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
    oracle, model, x = make(GOLDEN_CFG, dtype, 4, seed=5)
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
    # the trainer state round-trips
    sd = tr.state_dict()
    tr2 = FusedTrainer(model, learning_rate=1e-3, max_grad_norm=1.0)
    tr2.load_state_dict(sd)
    assert tr2.step_count == 3 and torch.equal(tr2.exp_avg, tr.exp_avg)
    # and the same trainer keeps working without a graph
    tr.use_cuda_graph = False
    loss, _ = tr.step(xc)
    assert torch.isfinite(loss)
