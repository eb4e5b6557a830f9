"""CPU tier of the attention conformance suite: the host replica of the dispatch (`attention_oracle.plan`) pinned to
hand-worked values at the shapes the models run, and the element-wise checker shown to reject planted faults of the
kinds an attention kernel gets wrong (a padded key in the row sum, a mis-indexed dropout mask, swapped problems,
unscaled or doubled gradients, D from the undropped probabilities, writes past the end)."""
import inspect
import math

import pytest
import torch

from ecg_b200 import _lib as L
from ecg_b200.model import EcgVitForMaskedAutoencoding
import attention_oracle as O

BF, F32 = L.BF16, L.F32


# ---- plan ---------------------------------------------------------------------------------------------------------
def mae_visible_tokens():
    """tokens the MAE encoder attends over at the default mask ratio: CLS + the visible patches of the 12 x 2500,
    patch-50 geometry (n = 50 patches)"""
    ratio = inspect.signature(EcgVitForMaskedAutoencoding.__init__).parameters['mask_ratio'].default
    n = 2500 // 50
    return n - int(round(ratio * n)) + 1


def test_plan_model_shapes():
    # cfg2 (base, 12 heads of 64, N = 51) and cfg3 (per-lead tokens, N = 2401)
    assert O.plan(BF, 51, 64) == O.Plan('tc_packed', ('true',), ['attn_tc_fwd_kernel<true>'],
                                        ['attn_tc_bwd_kernel<true>'], 0)
    p = O.plan(BF, 2401, 64, B=2, H=12)
    assert p.family == 'tc_long' and p.fwd == ['attn_tc_fwd_kernel<false>']
    assert p.bwd == ['attn_tc_dot_kernel', 'attn_tc_bwd_kernel<false>', 'attn_tc_dq_convert_kernel']
    # D [2 * 12 * 2401 = 57624 -> 57664, a multiple of 64] + the fp32 dQ accumulator [2 * 2401, 12 * 64]
    assert p.scratch_floats == 57664 + 2 * 2401 * 768
    # the MAE encoder over its visible tokens (13 at mask ratio 0.75) and the decoder (256 wide, 4 heads of 64)
    nv = mae_visible_tokens()
    assert nv == 13
    assert O.plan(BF, nv, 64).family == 'tc_packed' and O.plan(BF, 51, 256 // 4).family == 'tc_packed'
    # cfg1 dims (d = 256, 8 heads: dh 32, N = 51): mma<32, 4> in bf16, SIMT float in fp32
    assert O.plan(BF, 51, 32) == O.Plan('mma', (32, 4), ['attention_fwd_mma_kernel<32,4>'],
                                        ['attention_bwd_mma_kernel<32,4>'], 0)
    assert O.plan(F32, 51, 32) == O.Plan('simt', ('float',), ['attention_fwd_simt_kernel<float>'],
                                         ['attention_bwd_simt_kernel<float>'], 0)
    # debug at its default geometry: 2560 / 64 = 40 patches + CLS = 41 tokens, 64 / 4 heads = dh 16
    assert O.plan(BF, 2560 // 64 + 1, 64 // 4).targs == (16, 3)
    # dh 16 past one tile: nothing but SIMT serves it
    assert O.plan(BF, 65, 16).family == 'simt' and O.plan(BF, 65, 16).targs == ('bf16',)
    # dh 32 per-lead: flash<32> with its D scratch
    p = O.plan(BF, 2401, 32, B=3, H=8)
    assert p == O.Plan('flash', (32,), ['flash_fwd_kernel<32>'],
                       ['flash_bwd_dot_kernel<32>', 'flash_bwd_dq_kernel<32>', 'flash_bwd_dkv_kernel<32>'], 3 * 8 * 2401)
    # fp32 never takes a tensor-core path
    assert O.plan(F32, 51, 64).family == 'simt' and O.plan(F32, 2401, 32).family == 'simt'


def test_plan_bf16_dh64_is_tcgen05_at_every_length():
    for N in range(1, 2402):
        assert O.plan(BF, N, 64).family == ('tc_packed' if N <= 64 else 'tc_long'), N


@pytest.mark.parametrize('N,nt', [(1, 1), (16, 1), (17, 2), (32, 2), (33, 3), (48, 3), (49, 4), (64, 4)])
def test_plan_nt_boundaries(N, nt):
    for dh in (16, 32):
        assert O.plan(BF, N, dh).targs == (dh, nt)
    assert O.plan(BF, N, 64).family == 'tc_packed'
    assert O.plan(BF, N, 64, B=7, H=3).scratch_floats == 0


def test_kernel_inventory():
    ks = O.all_kernels()
    assert len(ks) == 32 and len(set(ks)) == 32
    names = set(ks)
    for dt in (BF, F32):
        for N in (1, 17, 64, 65, 300, 2401):
            for dh in (8, 16, 24, 32, 64):
                p = O.plan(dt, N, dh)
                assert set(p.fwd + p.bwd) <= names, (dt, N, dh)


def test_simt_length_limit():
    for dh in (8, 16, 32, 64):
        for bwd in (False, True):
            n = O.simt_max_len(dh, bwd)
            assert O.simt_smem(n, dh, bwd) <= 227 * 1024 < O.simt_smem(n + 1, dh, bwd)
    assert O.simt_max_len(16, True) < 2560 // 64 * 12 + 1      # per-lead debug tokens are refused today


# ---- the checker rejects planted faults -------------------------------------------------------------------------------
def unheads(x, B, N, H, dh):
    return x.reshape(B, H, N, dh).permute(0, 2, 1, 3).reshape(B * N, H * dh)


def faithful(case):
    """(reference, outputs of a kernel that rounds the exact results to the stored types) of a CPU case; the stored o /
    lse that backward reads are the forward's"""
    B, N, H, dh = case.B, case.N, case.H, case.dh
    fwd = O.reference(case, bwd=False)
    case.o.copy_(unheads(fwd['o'][0], B, N, H, dh).to(case.td))
    case.lse.copy_(fwd['lse'][0].view(B, H, N).float())
    ref = O.reference(case)
    got = {k: (r.float() if k == 'lse' else r.to(case.td)) for k, (r, _) in ref.items()}
    return ref, got


def operands(case, bh):
    B, N, H, dh = case.B, case.N, case.H, case.dh
    q, k, v = (O.heads(case.qkv, B, N, H, dh, i, 3)[bh:bh + 1].double() for i in range(3))
    return q, k, v, O.heads(case.d_o, B, N, H, dh)[bh:bh + 1].double()


def rejects(case, ref, got, **kw):
    with pytest.raises(AssertionError):
        O.check(case, ref, got, **kw)


@pytest.fixture(scope='module', params=[(BF, 3, 51, 1, 64), (BF, 2, 100, 1, 32), (F32, 1, 70, 2, 16)],
            ids=['tc-packed', 'flash', 'simt-f32'])
def planted(request):
    dt, B, N, H, dh = request.param
    case = O.Case(B, N, H, dh, dt, p=0.5, site=3, seed=11, device='cpu', amp=1.5)
    ref, got = faithful(case)
    O.check(case, ref, got, what='faithful')
    O.check_guards(case)
    return case, ref, got


def test_faithful_rounding_passes_and_p_is_quantised(planted):
    case, ref, got = planted
    assert O.quantised_p(case.p) == 32768
    assert case.keep([0]).unique().tolist() == [0.0, 2.0]


def test_rejects_padded_key_in_one_row_sum(planted):
    case, ref, got = planted
    q, k, v, _ = operands(case, 0)
    z = torch.zeros(1, 1, case.dh, dtype=torch.float64)
    keep = torch.cat([case.keep([0]), torch.ones(1, case.N, 1, dtype=torch.float64)], -1)
    _, _, _, _, Ob, lseb = O.forward64(q, torch.cat([k, z], 1), torch.cat([v, z], 1), case.scale, keep)
    bad = {k_: t.clone() for k_, t in got.items()}
    bad['o'][0, 5] = Ob[0, 5].to(bad['o'].dtype)
    bad['lse'][0, 5] = lseb[0, 5].float()
    rejects(case, ref, bad, names=('o', 'lse'))


def test_rejects_tail_of_last_key_block_unmasked(planted):
    case, ref, got = planted
    Np = O.padded(case.N)
    q, k, v, _ = operands(case, 0)
    z = torch.zeros(1, Np - case.N, case.dh, dtype=torch.float64)
    keep = case.keep([0], cols=torch.arange(Np))
    _, _, _, _, Ob, lseb = O.forward64(q, torch.cat([k, z], 1), torch.cat([v, z], 1), case.scale, keep)
    bad = {k_: t.clone() for k_, t in got.items()}
    bad['lse'][0] = lseb[0].float()
    rejects(case, ref, bad, names=('lse',))


@pytest.mark.parametrize('fault', ['shift', 'pitch-N'])
def test_rejects_misindexed_mask(planted, fault):
    case, ref, got = planted
    q, k, v, do = operands(case, 0)
    keep = case.keep([0], shift=1) if fault == 'shift' else case.keep([0], pitch=case.N)
    _, _, _, _, Ob, _ = O.forward64(q, k, v, case.scale, keep)
    bad = {k_: t.clone() for k_, t in got.items()}
    bad['o'][0] = Ob[0].to(bad['o'].dtype)
    rejects(case, ref, bad, names=('o',))
    lse = case.lse.reshape(-1, case.N)[0:1].double()
    D = (do * O.heads(case.o, case.B, case.N, case.H, case.dh)[0:1].double()).sum(-1)
    dq, dk, dv, *_ = O.backward64(q, k, v, do, case.scale, keep, lse, D)
    for name, t in (('dq', dq), ('dk', dk), ('dv', dv)):
        bad = {k_: x.clone() for k_, x in got.items()}
        bad[name][0] = t[0].to(bad[name].dtype)
        rejects(case, ref, bad, names=(name,))


def test_rejects_missing_keep_scale_on_one_row(planted):
    case, ref, got = planted
    bad = {k: t.clone() for k, t in got.items()}
    bad['o'][0, 7] *= 0.5
    rejects(case, ref, bad, names=('o',))


def test_rejects_swapped_problems(planted):
    case, ref, got = planted
    if case.B * case.H < 2:
        pytest.skip('one problem')
    bad = {k: t.clone() for k, t in got.items()}
    for name in ('o', 'dq'):
        bad = {k: t.clone() for k, t in got.items()}
        bad[name][[0, 1]] = bad[name][[1, 0]]
        rejects(case, ref, bad, names=(name,))


def test_rejects_lse_off_by_log2(planted):
    case, ref, got = planted
    bad = {k: t.clone() for k, t in got.items()}
    bad['lse'][0, 3] += math.log(2.0)
    rejects(case, ref, bad, names=('lse',))


@pytest.mark.parametrize('fault', ['no-scale', 'doubled'])
def test_rejects_bad_dq(planted, fault):
    case, ref, got = planted
    bad = {k: t.clone() for k, t in got.items()}
    bad['dq'] = (bad['dq'].double() / case.scale if fault == 'no-scale' else bad['dq'].double() * 2).to(case.td)
    rejects(case, ref, bad, names=('dq',))


def test_rejects_dk_dv_swapped_for_one_head(planted):
    case, ref, got = planted
    bad = {k: t.clone() for k, t in got.items()}
    bad['dk'][0], bad['dv'][0] = got['dv'][0].clone(), got['dk'][0].clone()
    rejects(case, ref, bad, names=('dk',))
    rejects(case, ref, bad, names=('dv',))


def test_rejects_d_from_undropped_p(planted):
    case, ref, got = planted
    q, k, v, do = operands(case, 0)
    lse = case.lse.reshape(-1, case.N)[0:1].double()
    P = torch.exp(case.scale * (q @ k.transpose(-1, -2)) - lse.unsqueeze(-1))
    D = (P * (do @ v.transpose(-1, -2))).sum(-1)
    dq, dk, _, *_ = O.backward64(q, k, v, do, case.scale, case.keep([0]), lse, D)
    for name, t in (('dq', dq), ('dk', dk)):
        bad = {k_: x.clone() for k_, x in got.items()}
        bad[name][0] = t[0].to(bad[name].dtype)
        rejects(case, ref, bad, names=(name,))


def test_rejects_write_past_the_end(planted):
    case, _, _ = planted
    for buf in (case.o_buf, case.lse_buf, case.dqkv_buf):
        n = buf.numel() - O.GUARD
        old = buf[n].clone()
        buf[n] = 0
        with pytest.raises(AssertionError):
            O.check_guards(case)
        buf[n] = old
    O.check_guards(case)


def test_rejects_unwritten_element(planted):
    case, ref, got = planted
    bad = {k: t.clone() for k, t in got.items()}
    bad['dv'][0, case.N - 1, 0] = float('nan')
    rejects(case, ref, bad, names=('dv',))
