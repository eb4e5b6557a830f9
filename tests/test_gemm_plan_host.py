"""CPU tier of the GEMM conformance suite: the host replica of the tile-width / split-K plan (tests/gemm_oracle.py) pinned
against values worked out by hand from csrc/gemm_tc.cu at 148 SMs, the shape search of the sweep, and the element-wise
checker shown to reject the mistakes it exists to catch."""
import pytest

from ecg_b200 import _lib as L
import gemm_oracle as O

SMS = 148   # B200: 74 CTA-pair clusters

# cfg2: M = 256 records x 51 tokens = 13056 rows = 51 pair tiles.  Scores (waves x BN / efficiency, 74 clusters):
#   N = 2304 (QKV):     256: 9 tiles  -> 459 units, 7 waves -> 1792;  192: 12 -> 612, 9 -> 1963.6;  128: 18 -> 918, 13 -> 2483.6
#   N = 768 (out-proj, FF2), K-major B:  256: 153 units, 3 waves -> 768;  192: 204, 3 -> 654.5;  128: 306, 5 -> 955.2
#   N = 768, MN-major B (dgrad):          192: 3 x 192 / 0.82 = 702.4 < 768
#   N = 3072 (FF1, FF1 dgrad):  256: 612 units, 9 waves -> 2304;  192: 816, 12 -> 2618 (2809 MN-major);  128: 1224, 17
# wgrad (contraction over the 13056 rows: 204 k blocks), auto split = the first split whose units fill >= 90 % of their
# last wave, on 256 x 256 tiles:
#   2304 x 768: 27 tiles: 1 -> 0.36, 2 -> 0.73, 3 -> 0.55, 4 -> 0.73 (not better), 5 -> 135 / 148 = 0.91: split 5;
#               then 256: 135 units, 2 waves -> 512;  192: 180, 3 -> 702;  128: 270, 4 -> 764
#   768 x 768:  9 tiles: 9 s / 74 first >= 0.9 at s = 8 (72 / 74); 256: 72 units, 1 wave
#   3072 x 768 and 768 x 3072: 36 tiles: s = 2 -> 72 / 74 = 0.97; 256: 72 units, 1 wave
PINNED = [
    # name, M, N, K, a_kmajor, b_kmajor, epilogue, split_k, (BN, split)
    ('qkv', 13056, 2304, 768, 1, 1, L.EPI_STORE, 1, (256, 1)),
    ('out-proj', 13056, 768, 768, 1, 1, L.EPI_BIAS_RES, 1, (192, 1)),
    ('out-proj-res32', 13056, 768, 768, 1, 1, L.EPI_BIAS_RES_F32, 1, (192, 1)),
    ('ff1', 13056, 3072, 768, 1, 1, L.EPI_BIAS_GELU, 1, (256, 1)),
    ('ff2', 13056, 768, 3072, 1, 1, L.EPI_BIAS_RES, 1, (192, 1)),
    ('ff1-dgrad', 13056, 3072, 768, 1, 0, L.EPI_DGELU, 1, (256, 1)),
    ('ff2-dgrad', 13056, 768, 3072, 1, 0, L.EPI_STORE, 1, (192, 1)),
    ('qkv-wgrad', 2304, 768, 13056, 0, 0, L.EPI_ATOMIC_F32, 0, (256, 5)),
    ('out-proj-wgrad', 768, 768, 13056, 0, 0, L.EPI_ATOMIC_F32, 0, (256, 8)),
    ('ff1-wgrad', 3072, 768, 13056, 0, 0, L.EPI_ATOMIC_F32, 0, (256, 2)),
    ('ff2-wgrad', 768, 3072, 13056, 0, 0, L.EPI_ATOMIC_F32, 0, (256, 2)),
    # the clamps: 7 k blocks cannot feed 9 splits; 6 k blocks in 4 splits would leave the last one empty (2 + 2 + 2).
    # All of them fit one wave (at most 2 x 4 x 7 = 56 units on 128-wide tiles), where 128 / 0.67 is the best score.
    ('split-clamped-to-k-blocks', 512, 512, 420, 0, 0, L.EPI_ATOMIC_F32, 9, (128, 7)),
    ('split-every-split-a-block', 512, 512, 328, 0, 0, L.EPI_ATOMIC_F32, 4, (128, 3)),
    ('split-3-of-7', 512, 512, 420, 0, 0, L.EPI_ATOMIC_F32, 3, (128, 3)),
    # N <= 128 takes 128 whatever the scores; a single wave prefers the narrow tile (128 / 0.67 < 192 / 0.88 < 256)
    ('narrow-n', 13056, 128, 768, 1, 1, L.EPI_STORE, 1, (128, 1)),
    ('one-wave', 300, 1000, 64, 1, 1, L.EPI_STORE, 1, (128, 1)),
]


@pytest.mark.parametrize('name,M,N,K,a_k,b_k,epi,split,want', PINNED, ids=[p[0] for p in PINNED])
def test_plan_matches_hand_worked_values(name, M, N, K, a_k, b_k, epi, split, want):
    assert O.plan(M, N, K, a_k, b_k, epi, split, SMS) == want


def test_plan_never_picks_256_for_the_fp32_residual():
    for M in (256, 4096, 13056, 30000):
        for N in (768, 1024, 2304, 8192):
            assert O.plan(M, N, 768, 1, 1, L.EPI_BIAS_RES_F32, 1, SMS)[0] < 256


def test_instantiation_lists():
    tc = O.tc_instantiations()
    assert len(tc) == len(set(tc)) == 34
    assert [sum(k[0] == bn for k in tc) for bn in O.WIDTHS] == [12, 12, 10]
    assert len(O.ffma_instantiations()) == 7


def test_model_cases_hit_the_widths_the_models_run():
    got = {name: O.plan(M, N, K, a_k, b_k, epi, O.model_case_options(o)['split_k'], SMS)[0]
           for name, M, N, K, a_k, b_k, epi, o in O.MODEL_CASES}
    assert got['cfg2-qkv'] == got['cfg2-ff1'] == got['cfg2-ff1-dgrad'] == 256
    assert got['cfg2-out-proj'] == got['cfg2-ff2'] == got['cfg2-out-proj-res32'] == got['cfg2-ff2-dgrad'] == 192
    assert {got[n] for n in got if n.endswith('wgrad')} == {256}


@pytest.mark.parametrize('regime', list(O.REGIMES))
def test_search_finds_a_shape_for_every_instantiation(regime):
    clusters = SMS // 2
    for key in O.tc_instantiations():
        bn, a_mn, b_mn, mode, path = key
        specs = O.sweep_specs(key, regime, SMS)
        assert len(specs) == len(O.REGIMES[regime])
        for (M, N, K, opts), v in zip(specs, O.REGIMES[regime]):
            pbn, split = O.plan(M, N, K, not a_mn, not b_mn, mode, opts['split_k'], SMS)
            assert pbn == bn, (O.key_name(key), M, N, K)
            assert N % 8 == 0 and N % 32 != 0 and N % 64 != 0 and K % 64 != 0
            if regime == 'small':
                assert M % 256 != 0
            else:
                assert O.units(M, N, bn, split) >= 2 * clusters and N % bn != 0
        if regime == 'small':
            assert specs[0][0] < 256 and specs[0][2] < 64     # below one pair tile, K below one k block
    # deterministic
    assert O.sweep_specs(O.tc_instantiations()[5], regime, SMS) == O.sweep_specs(O.tc_instantiations()[5], regime, SMS)


# ---- the checker rejects what it is meant to catch ------------------------------------------------------------------
def synthesize(case, r, keep=None, s=None, bias=None):
    """a correct kernel's outputs (fp64 reference rounded to the output types) written into the case's buffers, from
    the reference parts `r` with the dropout multipliers / drop-path factors / bias replaced when given"""
    M, N = case.M, case.N
    keep = r['keep'] if keep is None else keep
    s = r['s'] if s is None else s
    bias = r['bias'] if bias is None else bias
    u = r['acc'] + bias
    if case.mode == L.EPI_BIAS_GELU:
        case.out[:M, :N] = u.to(case.out_td)
        case.out2[:M, :N] = (keep * O.gelu64(u)).to(case.td)
    elif case.mode in (L.EPI_BIAS_RES, L.EPI_BIAS_RES_F32):
        case.out[:M, :N] = (s * keep * u + r['aux']).to(case.out_td)
    elif case.mode == L.EPI_DGELU:
        case.out[:M, :N] = (keep * r['acc'] * O.gelu_grad64(r['aux'])).to(case.out_td)
    else:
        case.out[:M, :N] = u.to(case.out_td)


PERTURBATIONS = ['mask-shift', 'mask-ld-n', 'bias-chunk', 'block-swap', 'path-flip']


@pytest.mark.parametrize('mode', [L.EPI_BIAS_RES, L.EPI_BIAS_GELU, L.EPI_DGELU, L.EPI_BIAS_RES_F32, L.EPI_STORE],
                         ids=lambda m: O.MODE_NAMES[m])
@pytest.mark.parametrize('what', ['correct'] + PERTURBATIONS)
def test_checker_rejects_perturbed_results(mode, what):
    if what == 'path-flip' and mode not in (L.EPI_BIAS_RES, L.EPI_BIAS_RES_F32):
        pytest.skip('drop path belongs to the residual epilogues')
    if what in ('mask-shift', 'mask-ld-n') and mode not in O.DROPOUT_MODES:
        pytest.skip('no dropout in this epilogue')
    if what == 'bias-chunk' and mode == L.EPI_DGELU:
        pytest.skip('no bias in this epilogue')
    M, N, K = 96, 104, 40
    path = mode in (L.EPI_BIAS_RES, L.EPI_BIAS_RES_F32)
    case = O.Case(M, N, K, 1, mode != L.EPI_DGELU, mode, L.BF16, bias=True, ldo_pad=64, p=0.1, site=3,
                  path_rate=0.3 if path else 0.0, rpr=5, path_site=O.PATH_SITE, seed=4, device='cpu')
    r = case.reference()
    if what == 'correct':
        synthesize(case, r)
    elif what == 'mask-shift':
        synthesize(case, r, keep=case.keep(shift=1))
    elif what == 'mask-ld-n':
        synthesize(case, r, keep=case.keep(ld=N))
    elif what == 'bias-chunk':
        b = r['bias'].clone()
        b[40:48] = 0
        synthesize(case, r, bias=b)
    elif what == 'block-swap':
        synthesize(case, r)
        case.out[32:64, 32:64] = case.out[32:64, 64:96].clone()
    elif what == 'path-flip':
        s = r['s'].clone()
        row = int((s[:, 0] == 0).nonzero()[0][0]) if bool((s == 0).any()) else 7
        s[row] = 1.0 / (1.0 - case.path_rate) if float(s[row]) == 0 else 0.0
        synthesize(case, r, s=s)
    if what == 'correct':
        O.check(case, r=r)
    else:
        with pytest.raises(AssertionError):
            O.check(case, r=r)


def test_checker_rejects_writes_outside_the_output():
    case = O.Case(40, 72, 24, 1, 1, L.EPI_BIAS_GELU, L.BF16, ldo_pad=64, p=0.1, site=2, seed=5, device='cpu')
    r = case.reference()
    synthesize(case, r)
    O.check(case, r=r)
    for buf, idx in ((case.out, (3, 72)), (case.out2, (3, 100)), (case.out, (40, 0))):
        saved = buf[idx].clone()
        buf[idx] = 0.0
        with pytest.raises(AssertionError):
            O.check(case, r=r)
        buf[idx] = saved
