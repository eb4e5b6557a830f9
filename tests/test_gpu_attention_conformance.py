"""GPU tier of the attention conformance suite: every attention kernel (tcgen05 packed / long, mma.sync, flash, SIMT,
the Recorder's probabilities) against the fp64 reference of tests/attention_oracle.py, element by element, forward
and backward, with attention-probability dropout, at the head dims and lengths the models run and at the tails where
tiles go wrong.  Also: one-hot probes that pin every kernel's dropout index to the host replica, exact cases, the
persistent tcgen05 grid over several rounds, a dropout counter above 2^31, B*H past 65535 on flash, the profiler's
record of which kernel ran, bit-identical relaunches, CUDA-graph replay, chained and concurrent launches, and
refusals that write nothing."""
import math
import re

import pytest
import torch

pytestmark = pytest.mark.gpu

from ecg_b200 import _lib as L
import attention_oracle as O

BF, F32 = L.BF16, L.F32
P_MIN = 1.0 / 65536          # quantises to threshold 1


@pytest.fixture(scope='module')
def lib():
    assert torch.cuda.is_available()
    lib = L.load()
    assert lib.ecgvit_device_ok() == 1, 'these kernels are sm_100a only'
    return lib


@pytest.fixture(scope='module')
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def stream():
    return torch.cuda.current_stream().cuda_stream


def run_fwd(lib, case, st=None):
    L.check(case.fwd(lib, stream() if st is None else st), 'attention_fwd')


def run_bwd(lib, case, st=None):
    L.check(case.bwd(lib, stream() if st is None else st), 'attention_bwd')


def full_check(lib, case, what='', determinism=True):
    """forward and backward against the reference, sentinels after every output, inputs unchanged, and (optionally)
    a second launch of both bit-identical (tc long dQ: against the bound, its fp32 reduce-adds land in any order)"""
    snap = O.snapshot(case)
    run_fwd(lib, case)
    o0, lse0 = case.o_buf.clone(), case.lse_buf.clone()
    run_bwd(lib, case)
    torch.cuda.synchronize()
    O.check_guards(case, what=what)
    O.check_inputs(case, snap, o=o0, lse=lse0, what=what)
    ref = O.reference(case)
    got = case.outputs()
    O.check(case, ref, got, what=what)
    if determinism:
        first = {k: v.clone() for k, v in got.items()}
        case.reset()
        run_fwd(lib, case)
        run_bwd(lib, case)
        torch.cuda.synchronize()
        again = case.outputs()
        for k in first:
            if k == 'dq' and case.family == 'tc_long':
                O.check(case, ref, again, names=('dq',), what=what + ' relaunch')
                continue
            assert torch.equal(O.bits(first[k]), O.bits(again[k])), f'{O.tag(case, what)}: relaunch {k} differs'
    return ref


# ---- every instantiation on its own shapes --------------------------------------------------------------------------
SCALES = (None, 1.0, 0.05)
PS = (0.0, 0.1, 0.5, P_MIN)


def sweep():
    """(id, B, N, H, dh, dtype, scale, p): tails of N on every family, odd B*H, each (dh, NT) of the mma kernels"""
    S = []
    for N in (1, 2, 63, 64):                                    # tc packed; B*H odd: the last tile's 2nd problem is absent
        S.append((3, N, 1, 64, BF))
    for N in (65, 127, 128, 129, 191, 300, 2401):               # tc long
        S.append((1 if N == 2401 else 3, N, 1 if N == 2401 else 1, 64, BF))
    for dh in (16, 32):                                         # mma<dh, NT>
        for N in (1, 16, 17, 31, 33, 41, 49, 64):
            S.append((5, N, 3, dh, BF))
    for N in (65, 127, 128, 129, 191, 300, 2401):               # flash<32>
        S.append((1 if N == 2401 else 3, N, 1 if N == 2401 else 1, 32, BF))
    S += [(2, 65, 3, 16, BF), (2, 129, 1, 8, BF), (1, 100, 2, 24, BF), (3, 30, 1, 8, BF),
          (2, 51, 3, 64, F32), (3, 1, 1, 16, F32), (1, 2, 3, 8, F32), (2, 129, 1, 32, F32)]
    out = []
    for i, (B, N, H, dh, dt) in enumerate(S):
        out.append((f'{"bf16" if dt == BF else "f32"}-dh{dh}-N{N}-B{B}H{H}', B, N, H, dh, dt, SCALES[i % 3], PS[i % 4]))
    return out


SWEEP = sweep()


def make(B, N, H, dh, dt, scale, p, seed, **kw):
    return O.Case(B, N, H, dh, dt, scale=scale, p=p, site=seed % 7, seed=seed, **kw)


@pytest.mark.parametrize('spec', SWEEP, ids=[s[0] for s in SWEEP])
def test_instantiation_matches_fp64(lib, spec):
    name, B, N, H, dh, dt, scale, p = spec
    for pi, pp in enumerate((p, 0.5 if p != 0.5 else 0.1)):
        case = make(B, N, H, dh, dt, scale, pp, seed=len(name) + pi)
        full_check(lib, case, what=name)


# ---- one-hot probes: the dropout index of every kernel against the host replica ---------------------------------------
PROBES = [(3, 63, 1, 64, BF), (1, 300, 1, 64, BF), (2, 41, 2, 16, BF), (2, 64, 1, 32, BF), (1, 300, 1, 32, BF),
          (1, 100, 2, 16, BF), (1, 100, 1, 32, F32)]


def probe(lib, B, N, H, dh, dt):
    case = make(B, N, H, dh, dt, None, 0.5, seed=N + dh)
    bhs = torch.arange(B * H)
    q, k = (O.heads(case.qkv, B, N, H, dh, i, 3).double() for i in range(2))
    keep = case.keep(bhs)
    S = case.scale * (q @ k.transpose(-1, -2))
    P = torch.exp(S - S.amax(-1, keepdim=True))
    Pl = P * keep / P.sum(-1, keepdim=True)                     # the dropped, normalised probabilities
    tol = 2.0 ** -6
    # forward: V[j] = e_{j - w0} on a dh-key window -> O[i, d] = Pd[i, w0 + d] / l_i; a dropped one reads exactly 0
    for w0 in range(0, N, dh):
        n = min(dh, N - w0)
        O.onehot_window(case, w0, 2)
        case.reset()
        run_fwd(lib, case)
        torch.cuda.synchronize()
        full = O.heads(case.o, B, N, H, dh).double()
        got = full[:, :, :n]
        want = Pl[:, :, w0:w0 + n]
        drop = keep[:, :, w0:w0 + n] == 0
        assert bool((got[drop] == 0).all()), f'{O.tag(case)} fwd window {w0}: a dropped probability is not 0'
        assert bool(((got - want).abs() <= tol * want).all()), f'{O.tag(case)} fwd window {w0}: kept probabilities'
        assert bool((full[:, :, n:] == 0).all())
    # backward: dO[i] = e_{i - w0} on a dh-query window -> dV[j, d] = Pd[w0 + d, j] with P from the stored lse
    lse = case.lse.reshape(B * H, N).double()
    Pb = torch.exp(S - lse.unsqueeze(-1)) * keep
    for w0 in range(0, N, dh):
        n = min(dh, N - w0)
        O.onehot_window(case, w0, None)
        case.reset(fwd=False)
        run_bwd(lib, case)
        torch.cuda.synchronize()
        got = O.heads(case.dqkv, B, N, H, dh, 2, 3)[:, :, :n].double()
        want = Pb[:, w0:w0 + n, :].transpose(-1, -2)
        drop = keep[:, w0:w0 + n, :].transpose(-1, -2) == 0
        assert bool((got[drop] == 0).all()), f'{O.tag(case)} bwd window {w0}: dV of a dropped probability is not 0'
        assert bool(((got - want).abs() <= tol * want).all()), f'{O.tag(case)} bwd window {w0}: dV of kept ones'


@pytest.mark.parametrize('spec', PROBES, ids=[f'{"bf16" if s[4] == BF else "f32"}-dh{s[3]}-N{s[1]}' for s in PROBES])
def test_onehot_probe_pins_the_dropout_index(lib, spec):
    probe(lib, *spec)


# ---- persistent tcgen05 grid ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('which', ['below', 'equal', 'above', 'rounds'])
def test_persistent_tc_grid(lib, sms, which):
    """packed tiles and long items below, at, one above and at 2 SMs + 1 (CTAs take several rounds and slot 1 runs dry
    before slot 0); the long geometry with an odd number of query tiles (N = 300: 3)"""
    items = {'below': sms - 1, 'equal': sms, 'above': sms + 1, 'rounds': 2 * sms + 1}[which]
    full_check(lib, make(2 * items - 1, 51, 1, 64, BF, None, 0.1, seed=items), what=f'packed {items} tiles')
    full_check(lib, make(items, 129, 1, 64, BF, None, 0.1, seed=items + 1), what=f'long {items} items')
    if which == 'rounds':
        full_check(lib, make(1, 300, items, 64, BF, None, 0.1, seed=3), what='long, odd query tiles')


# ---- model shapes -------------------------------------------------------------------------------------------------------
def model_shapes():
    from test_attention_plan_host import mae_visible_tokens
    lead32 = O.simt_max_len(32, True)
    return [('cfg2', 256, 51, 12, 64, BF), ('cfg3-per-lead', 2, 2401, 12, 64, BF),
            ('mae-encoder-visible', 256, mae_visible_tokens(), 12, 64, BF), ('mae-decoder-256', 256, 51, 4, 64, BF),
            ('cfg1-dh32', 32, 51, 8, 32, BF), ('debug-dh16', 32, 41, 4, 16, BF), ('per-lead-dh32-flash', 2, 2401, 8, 32, BF),
            ('fp32-cfg1', 8, 51, 8, 32, F32), ('fp32-debug', 8, 41, 4, 16, F32), (f'fp32-N{lead32}', 2, lead32, 2, 32, F32)]


@pytest.mark.parametrize('spec', model_shapes(), ids=lambda s: s[0])
def test_model_shapes_match_fp64(lib, spec):
    name, B, N, H, dh, dt = spec
    full_check(lib, make(B, N, H, dh, dt, None, 0.1, seed=B + N), what=name, determinism=False)


# ---- exact cases --------------------------------------------------------------------------------------------------------
EXACT = [(3, 51, 1, 64, BF), (1, 300, 1, 64, BF), (1, 2401, 1, 64, BF), (2, 41, 2, 16, BF), (2, 17, 1, 32, BF),
         (1, 129, 2, 32, BF), (1, 65, 1, 16, BF), (1, 64, 2, 32, F32), (1, 100, 1, 32, F32)]


@pytest.mark.parametrize('spec', EXACT, ids=[f'{"bf16" if s[4] == BF else "f32"}-dh{s[3]}-N{s[1]}' for s in EXACT])
def test_uniform_probabilities_are_exact(lib, spec):
    """Q = 0, V = 1: every probability is exactly 1 before normalisation, so O = 1.0 (a padded key in the row sum
    would give N / (N + 1)) and lse = log N.  fp32 O is a sum of N copies of fl(1/N): exact when N is a power of 2."""
    B, N, H, dh, dt = spec
    case = make(B, N, H, dh, dt, None, 0.0, seed=1)
    v = case.qkv.view(B, N, 3, H, dh)
    v[:, :, 0] = 0
    v[:, :, 2] = 1
    run_fwd(lib, case)
    torch.cuda.synchronize()
    o = case.o.double()
    if dt == BF or N & (N - 1) == 0:
        assert torch.equal(O.bits(case.o), O.bits(torch.ones_like(case.o))), f'{O.tag(case)}: O != 1: {o.min()} {o.max()}'
    else:
        assert float((o - 1).abs().max()) <= N * 2.0 ** -24
    lse = case.lse.double()
    assert float((lse - math.log(N)).abs().max()) <= 2.0 ** -22 * max(1.0, math.log(N)), f'{O.tag(case)}: lse != log N'


@pytest.mark.parametrize('dh,dt', [(64, BF), (16, BF), (32, BF), (8, BF), (64, F32)])
def test_single_token_output_is_v(lib, dh, dt):
    case = make(7, 1, 3, dh, dt, None, 0.0, seed=dh)
    run_fwd(lib, case)
    torch.cuda.synchronize()
    v = case.qkv[:, 2 * case.inner:]
    assert torch.equal(O.bits(case.o), O.bits(v.contiguous())), O.tag(case)
    assert bool(torch.isfinite(case.lse).all())


# ---- large problem counts ------------------------------------------------------------------------------------------------
def check_problems(lib, case, bhs, what):
    snap = O.snapshot(case)
    run_fwd(lib, case)
    run_bwd(lib, case)
    torch.cuda.synchronize()
    O.check_guards(case, what=what)
    O.check_inputs(case, snap, what=what)
    ref = O.reference(case, bhs=torch.tensor(bhs))
    O.check(case, ref, case.outputs(torch.tensor(bhs, device='cuda')), what=what)


def test_dropout_counter_above_2_31(lib):
    """N = 2401, H = 1, B = 400 on tc long: B H Np^2 = 2.37e9; the problems whose counter range crosses 2^31 and the
    last one (counters just below 2^32 - 2^31 ... 2.37e9)"""
    B, N = 400, 2401
    Np2 = O.padded(N) ** 2
    cross = (1 << 31) // Np2
    assert cross * Np2 < (1 << 31) <= (cross + 1) * Np2 and B * Np2 > (1 << 31)
    case = make(B, N, 1, 64, BF, None, 0.1, seed=5)
    check_problems(lib, case, [cross, B - 1], 'counter above 2^31')


def test_flash_more_than_65535_problems(lib):
    """B * H = 65536 on flash (dh 32, N = 100): the grid must not put B * H in grid.y (65535 at most)"""
    case = make(65536, 100, 1, 32, BF, None, 0.1, seed=8)
    assert case.family == 'flash'
    check_problems(lib, case, [0, 1, 65534, 65535], 'B*H = 65536')


# ---- the Recorder's probabilities -----------------------------------------------------------------------------------
@pytest.mark.parametrize('dt', [BF, F32], ids=['bf16', 'f32'])
@pytest.mark.parametrize('B,N,H,dh,gap', [(3, 51, 4, 64, 0), (2, 129, 2, 16, 37), (1, 1, 3, 8, 5)])
def test_attention_probs_match_fp64(lib, dt, B, N, H, dh, gap):
    case = make(B, N, H, dh, dt, None, 0.0, seed=N)
    stride = H * N * N + gap
    buf, probs = O.guarded(B * stride, torch.float32, 'cuda')
    L.check(lib.ecgvit_attention_probs(case.qkv.data_ptr(), probs.data_ptr(), B, N, H, dh, case.scale, stride, dt,
                                          stream()), 'attention_probs')
    run_fwd(lib, case)
    torch.cuda.synchronize()
    got = probs.view(B, stride)[:, :H * N * N].reshape(B * H, N, N).double()
    q, k, v = (O.heads(case.qkv, B, N, H, dh, i, 3).double() for i in range(3))
    S, P, l, m, Oe, _ = O.forward64(q, k, v, case.scale, torch.ones_like(q[..., :1]))
    eS, eps, _, blse = O._fwd_bounds(case, q, k, v, torch.ones_like(P), S, P, l, m, Oe)
    want = P / l
    bound = ((3 * eps + 2 * O.C_ACC * N).unsqueeze(-1)) * want
    assert bool(((got - want).abs() <= bound).all()), f'probs off the fp64 softmax: {float((got - want).abs().max())}'
    assert float((got.sum(-1) - 1).abs().max()) <= (2 * N + 4) * 2.0 ** -24
    # consistent with the forward's lse: probs = exp(S - lse)
    lse = case.lse.reshape(B * H, N).double()
    alt = torch.exp(S - lse.unsqueeze(-1))
    assert bool(((got - alt).abs() <= (blse + 3 * eps).unsqueeze(-1) * alt).all())
    gaps = probs.view(B, stride)[:, H * N * N:]
    assert torch.equal(O.bits(gaps), O.bits(torch.full_like(gaps, float('nan'))))
    assert torch.equal(O.bits(buf[-O.GUARD:]), O.bits(torch.full((O.GUARD,), float('nan'), device='cuda')))


# ---- pinned behaviour ---------------------------------------------------------------------------------------------------
def test_tc_packed_backward_never_reads_o(lib):
    case = make(5, 51, 3, 64, BF, None, 0.1, seed=2)
    run_fwd(lib, case)
    run_bwd(lib, case)
    torch.cuda.synchronize()
    want = case.dqkv.clone()
    case.o.fill_(float('nan'))
    case.reset(fwd=False)
    run_bwd(lib, case)
    torch.cuda.synchronize()
    assert torch.equal(O.bits(case.dqkv), O.bits(want))
    O.check(case, O.reference(case, o_in='exact'), case.outputs(), names=('dq', 'dk', 'dv'), what='NaN o')


@pytest.mark.parametrize('B,N,H,dh', [(3, 51, 2, 64), (2, 300, 1, 64), (3, 41, 2, 16), (2, 129, 1, 32), (2, 65, 1, 16)])
def test_null_seed_means_no_dropout(lib, B, N, H, dh):
    """p > 0 with a NULL seed runs without dropout (make_dropout), silently"""
    plain = make(B, N, H, dh, BF, None, 0.0, seed=4)
    run_fwd(lib, plain)
    run_bwd(lib, plain)
    nul = make(B, N, H, dh, BF, None, 0.5, seed=4, null_seed=True)
    run_fwd(lib, nul)
    run_bwd(lib, nul)
    torch.cuda.synchronize()
    for a, b in ((plain.o, nul.o), (plain.lse, nul.lse)) + ((() if plain.family == 'tc_long' else ((plain.dqkv, nul.dqkv),))):
        assert torch.equal(O.bits(a), O.bits(b))
    O.check(nul, O.reference(nul), nul.outputs())


# ---- which kernel ran ---------------------------------------------------------------------------------------------------
KERNEL_RE = re.compile(r'\b(attn_tc_\w+_kernel|attention_\w+_kernel|flash_\w+_kernel)\s*(<[^()]*?>)?\s*\(')


def kernel_name(name):
    m = KERNEL_RE.search(name)
    if not m:
        return None
    args = re.sub(r'\s+', '', m.group(2) or '')
    args = re.sub(r'(__)?nv_bfloat16', 'bf16', args)
    return m.group(1) + args


def profile_calls(lib, calls):
    """run `calls` [(expected kernel names, thunk)] under the profiler; the attention kernels that ran, in order"""
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _, fn in calls:
            fn()
            torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if kernel_name(e.name)), key=lambda e: e.time_range.start)
    return [kernel_name(e.name) for e in ev]


def coverage_calls(lib):
    calls = []
    for name, B, N, H, dh, dt, scale, p in SWEEP:
        case = make(B, N, H, dh, dt, scale, p, seed=1)
        calls.append((case.plan.fwd + case.plan.bwd, lambda c=case: (run_fwd(lib, c), run_bwd(lib, c))))
    for dt, t in ((BF, 'bf16'), (F32, 'float')):
        case = make(2, 30, 2, 16, dt, None, 0.0, seed=1)
        probs = torch.empty(2 * 2 * 30 * 30, device='cuda')
        calls.append(([f'attention_probs_kernel<{t}>'], lambda c=case, pr=probs, dt=dt: L.check(
            lib.ecgvit_attention_probs(c.qkv.data_ptr(), pr.data_ptr(), 2, 30, 2, 16, c.scale, 2 * 30 * 30, dt,
                                       stream()), 'attention_probs')))
    return calls


def test_every_call_runs_the_planned_kernels(lib):
    """every sweep case runs the kernels `plan` predicts, and together they run all 32 attention kernels the library
    compiles"""
    calls = coverage_calls(lib)
    ran = profile_calls(lib, calls)
    want = [k for ks, _ in calls for k in ks]
    assert ran == want, f'kernels differ from the plan: first difference at ' \
                        f'{next((i, a, b) for i, (a, b) in enumerate(zip(ran + [None] * 9, want + [None] * 9)) if a != b)}'
    every = set(O.all_kernels())
    assert set(ran) == every, f'not run: {sorted(every - set(ran))}; unknown: {sorted(set(ran) - every)}'
    print(f'{len(calls)} calls, {len(set(ran))} attention kernels seen')


# ---- graphs, chaining, streams --------------------------------------------------------------------------------------------
GRAPH_SPECS = [(3, 51, 2, 64, BF), (2, 300, 1, 64, BF), (3, 41, 2, 16, BF), (2, 51, 2, 32, BF), (1, 129, 2, 32, BF),
               (1, 100, 1, 16, BF), (1, 40, 2, 32, F32)]


def results(case):
    return [case.o_buf.clone(), case.lse_buf.clone(), case.dqkv_buf.clone()]


def same(case, a, b, what):
    for i, (x, y) in enumerate(zip(a, b)):
        if i == 2 and case.family == 'tc_long':               # dQ: fp32 reduce-adds in any order; dK, dV exact
            n = case.dqkv.numel()
            for part in (1, 2):
                hx, hy = (O.heads(t[:n].view_as(case.dqkv), case.B, case.N, case.H, case.dh, part, 3) for t in (x, y))
                assert torch.equal(O.bits(hx), O.bits(hy)), f'{O.tag(case, what)}: d{"qkv"[part]} differs'
            assert torch.equal(O.bits(x[n:]), O.bits(y[n:]))
            continue
        assert torch.equal(O.bits(x), O.bits(y)), f'{O.tag(case, what)}: output {i} differs'


def test_graph_replay_with_new_seeds_matches_eager(lib):
    cases = [make(*s[:4], s[4], None, 0.3, seed=i) for i, s in enumerate(GRAPH_SPECS)]
    for c in cases:                                             # warm up outside capture
        run_fwd(lib, c)
        run_bwd(lib, c)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            for c in cases:
                run_fwd(lib, c, side.cuda_stream)
                run_bwd(lib, c, side.cuda_stream)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    for rep, seed in enumerate((11, 222, 3333)):
        eager = []
        for c in cases:
            c.seed_dev.fill_(seed)
            c.seed_value = seed
            c.o_buf[:-O.GUARD].fill_(float('nan'))
            run_fwd(lib, c)
            run_bwd(lib, c)
            eager.append(results(c))
        torch.cuda.synchronize()
        for c in cases:
            c.o_buf[:-O.GUARD].fill_(float('nan'))
            c.dqkv_buf[:-O.GUARD].fill_(float('nan'))
        graph.replay()
        torch.cuda.synchronize()
        for c, want in zip(cases, eager):
            same(c, results(c), want, f'replay {rep}')
        ref = O.reference(cases[1])
        O.check(cases[1], ref, cases[1].outputs(), what=f'replay {rep}')


def gemm_qkv(lib, x, w, qkv, st):
    M, K = x.shape
    n = w.shape[0]
    g = L.GemmArgs(M=M, N=n, K=K, A=x.data_ptr(), lda=K, a_kmajor=1, B=w.data_ptr(), ldb=K, b_kmajor=1,
                   epilogue=L.EPI_STORE, out=qkv.data_ptr(), ldo=n, out2=None, aux=None, bias=None, dtype=BF,
                   split_k=1, dropout_stream=0, dropout_p=0.0, dropout_seed=None)
    import ctypes
    L.check(lib.ecgvit_gemm(ctypes.byref(g), st), 'gemm')


@pytest.mark.parametrize('B,N,H,dh', [(16, 51, 12, 64), (2, 300, 4, 64), (16, 51, 8, 32), (2, 129, 4, 32)])
def test_gemm_then_attention_chained_without_sync(lib, B, N, H, dh):
    """QKV projection -> attention forward -> backward back to back on one stream (PDL-launched kernels wait on their
    producers) equals the same calls synchronised one by one"""
    d = H * dh
    g = torch.Generator(device='cuda').manual_seed(N)
    x = (torch.randn(B * N, d, device='cuda', generator=g)).bfloat16()
    w = (torch.randn(3 * d, d, device='cuda', generator=g) * d ** -0.5).bfloat16()
    case = make(B, N, H, dh, BF, None, 0.1, seed=N)
    st = stream()
    outs = []
    for sync in (True, False):
        case.qkv.fill_(float('nan'))
        case.reset()
        torch.cuda.synchronize()
        gemm_qkv(lib, x, w, case.qkv, st)
        if sync:
            torch.cuda.synchronize()
        run_fwd(lib, case)
        if sync:
            torch.cuda.synchronize()
        run_bwd(lib, case)
        torch.cuda.synchronize()
        outs.append(results(case))
    same(case, outs[1], outs[0], 'chained')
    O.check(case, O.reference(case), case.outputs(), what='chained')


def test_two_families_on_two_streams(lib):
    cases = [make(4, 300, 4, 64, BF, None, 0.1, seed=1), make(64, 51, 8, 32, BF, None, 0.1, seed=2),
             make(2, 2401, 2, 32, BF, None, 0.1, seed=3)]
    solo = []
    for c in cases:
        run_fwd(lib, c)
        run_bwd(lib, c)
        torch.cuda.synchronize()
        solo.append(results(c))
        c.reset()
    streams = [torch.cuda.Stream() for _ in cases]
    for s in streams:
        s.wait_stream(torch.cuda.current_stream())
    for c, s in zip(cases, streams):
        run_fwd(lib, c, s.cuda_stream)
        run_bwd(lib, c, s.cuda_stream)
    torch.cuda.synchronize()
    for c, want in zip(cases, solo):
        same(c, results(c), want, 'two streams')


# ---- refusals ----------------------------------------------------------------------------------------------------------
def refusals():
    R = []
    small = (3, 51, 2, 64, BF)
    for k in ('qkv', 'o', 'lse'):
        R.append((f'fwd-null-{k}', small, 'fwd', {k: None}))
    for k in ('qkv', 'o', 'd_o', 'lse', 'dqkv'):
        R.append((f'bwd-null-{k}', small, 'bwd', {k: None}))
    for k, v in (('B', 0), ('N', 0), ('H', 0), ('B', -1), ('N', -5), ('H', -2)):
        for w in ('fwd', 'bwd'):
            R.append((f'{w}-{k}{v}', small, w, {k: v}))
    for w in ('fwd', 'bwd'):
        R.append((f'{w}-dh12', (3, 51, 2, 16, BF), w, {'dh': 12}))
        R.append((f'{w}-dtype-bf16-res32', small, w, {'dtype': L.BF16_RES32}))
        R.append((f'{w}-dtype-7', small, w, {'dtype': 7}))
        R.append((f'{w}-counter-over-2^32', small, w, {'B': 727, 'N': 2401, 'H': 1}))
        R.append((f'{w}-tc-misaligned-qkv', small, w, {'qkv': '+8'}))
    R.append(('fwd-tc-misaligned-o', small, 'fwd', {'o': '+8'}))
    R.append(('bwd-tc-misaligned-d_o', small, 'bwd', {'d_o': '+8'}))
    R.append(('bwd-tc-misaligned-dqkv', small, 'bwd', {'dqkv': '+8'}))
    for spec in ((2, 300, 1, 64, BF), (2, 300, 1, 32, BF)):
        R.append((f'bwd-{spec[3]}-no-scratch', spec, 'bwd', {'scratch': None}))
        R.append((f'bwd-{spec[3]}-misaligned-scratch', spec, 'bwd', {'scratch': '+4'}))
    for dt, t in ((BF, 'bf16'), (F32, 'f32')):
        for w in ('fwd', 'bwd'):
            n = O.simt_max_len(16, w == 'bwd') + 1
            R.append((f'{w}-simt-{t}-N{n}', (1, n, 1, 16, dt), w, {}))
    return R


@pytest.mark.parametrize('spec', refusals(), ids=[r[0] for r in refusals()])
def test_refusals_write_nothing(lib, spec):
    name, (B, N, H, dh, dt), which, ov = spec
    case = make(B, N, H, dh, dt, None, 0.1, seed=1)
    if which == 'bwd':
        run_fwd(lib, case)
    torch.cuda.synchronize()
    args = {}
    for k, v in ov.items():
        if isinstance(v, str):
            base = {'qkv': case.qkv, 'o': case.o, 'd_o': case.d_o, 'dqkv': case.dqkv, 'scratch': case.scratch}[k]
            args[k] = base.data_ptr() + int(v)
        else:
            args[k] = v
    before = [case.o_buf.clone(), case.lse_buf.clone(), case.dqkv_buf.clone()]
    rc = (case.fwd if which == 'fwd' else case.bwd)(lib, stream(), **args)
    torch.cuda.synchronize()
    assert rc != 0, f'{name}: accepted'
    assert L.last_error(), f'{name}: refused without a message'
    for got, want in zip((case.o_buf, case.lse_buf, case.dqkv_buf), before):
        assert torch.equal(O.bits(got), O.bits(want)), f'{name}: a refused call wrote an output'
    ok = make(1, 17, 1, 16, BF, None, 0.0, seed=2)            # no sticky error: the next call runs
    run_fwd(lib, ok)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(ok.o.float()).all())


def test_probs_refuses_short_batch_stride(lib):
    case = make(2, 30, 2, 16, BF, None, 0.0, seed=1)
    buf, probs = O.guarded(2 * 2 * 30 * 30, torch.float32, 'cuda')
    rc = lib.ecgvit_attention_probs(case.qkv.data_ptr(), probs.data_ptr(), 2, 30, 2, 16, case.scale, 2 * 30 * 30 - 1,
                                       BF, stream())
    torch.cuda.synchronize()
    assert rc != 0 and L.last_error()
    assert bool(torch.isnan(buf).all())


def test_counter_limit_is_inclusive(lib):
    """B H Np^2 = 2^32 exactly is accepted with dropout (mma<16, 1>: N = 1, B = 2^20); one problem more is accepted
    without dropout only"""
    B = 1 << 20
    case = make(B, 1, 1, 16, BF, None, 0.1, seed=6)
    run_fwd(lib, case)
    run_bwd(lib, case)
    torch.cuda.synchronize()
    last = torch.tensor([0, B - 1])
    O.check(case, O.reference(case, bhs=last), case.outputs(last.cuda()), what='2^32')
    big = make(B + 1, 1, 1, 16, BF, None, 0.1, seed=6)
    assert big.fwd(lib, stream()) != 0
    torch.cuda.synchronize()
    big.p = 0.0
    run_fwd(lib, big)
    torch.cuda.synchronize()
    v = big.qkv[:, 2 * big.inner:]
    assert torch.equal(O.bits(big.o), O.bits(v.contiguous()))
