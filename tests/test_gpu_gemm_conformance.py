"""GPU tier of the GEMM conformance suite: every tcgen05 instantiation gemm_tc2_kernel<BN, A_MN, B_MN, MODE, kPath> and
every FFMA kernel against an fp64 reference, element by element (tests/gemm_oracle.py), at shapes the host replica of
the width choice (`plan`) sends to each width: small problems with tails in M, N and K, persistent grids where every
cluster walks several tiles, and the contractions the models run.  Dropout, drop path, NULL bias, ldo > N and split-K
vary across the cases; the profiler confirms which kernel ran; persistent launches must be bit-identical from launch to
launch and under CUDA-graph replay; unsupported combinations must be refused without writing anything."""
import re

import pytest
import torch

pytestmark = pytest.mark.gpu

from ecg_b200 import _lib as L
import gemm_oracle as O

REGIME_NAMES = list(O.REGIMES)


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


def tc_case(key, M, N, K, opts, seed):
    bn, a_mn, b_mn, mode, path = key
    return O.Case(M, N, K, not a_mn, not b_mn, mode, L.BF16, seed=seed, **opts)


def run(lib, case):
    L.check(case.launch(lib, stream()), 'gemm')


def sweep_cases(sms):
    """(name, predicted kernel key, Case factory) of every tcgen05 sweep case, model case and FFMA case"""
    out = []
    for ki, key in enumerate(O.tc_instantiations()):
        for regime in REGIME_NAMES:
            for vi, (M, N, K, opts) in enumerate(O.sweep_specs(key, regime, sms)):
                out.append((f'{O.key_name(key)}-{regime}{vi}', ('tc',) + key,
                            lambda key=key, M=M, N=N, K=K, opts=opts, s=ki * 8 + vi: tc_case(key, M, N, K, opts, s)))
    for name, M, N, K, a_k, b_k, mode, o in O.MODEL_CASES:
        opts = O.model_case_options(o)
        bn, _ = O.plan(M, N, K, a_k, b_k, mode, opts['split_k'], sms)
        key = ('tc', bn, not a_k, not b_k, mode, bool(opts.get('path_rate')))
        out.append((name, key, lambda M=M, N=N, K=K, a_k=a_k, b_k=b_k, mode=mode, opts=opts:
                    O.Case(M, N, K, a_k, b_k, mode, L.BF16, seed=5, **opts)))
    for mode, path in O.ffma_instantiations():
        for a_k, b_k in O.LAYOUTS:
            for si, (M, N, K, opts) in enumerate(O.FFMA_SHAPES):
                out.append((f'ffma-{O.MODE_NAMES[mode]}{"-path" if path else ""}-{a_k}{b_k}-{si}', ('ffma', mode, path),
                            lambda mode=mode, path=path, a_k=a_k, b_k=b_k, M=M, N=N, K=K, opts=opts:
                            O.Case(M, N, K, a_k, b_k, mode, L.F32, seed=3, **ffma_opts(opts, path, M))))
    return out


def ffma_opts(opts, path, M):
    o = dict(opts)
    rpr = o.pop('rpr')
    if path:
        o.update(path_rate=O.PATH_RATE, path_site=O.PATH_SITE, rpr=M if rpr == 'M' else rpr)
    return o


# ---- the sweeps ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('regime', REGIME_NAMES)
@pytest.mark.parametrize('key', O.tc_instantiations(), ids=O.key_name)
def test_tcgen05_instantiation_matches_fp64(lib, sms, key, regime):
    """each instantiation on the smallest shapes where the host plan picks its width; in the persistent regime a second
    launch of a non-atomic epilogue must reproduce the first bit for bit"""
    for vi, (M, N, K, opts) in enumerate(O.sweep_specs(key, regime, sms)):
        case = tc_case(key, M, N, K, opts, seed=vi)
        run(lib, case)
        O.check(case, what=f'{O.key_name(key)} {regime}{vi}')
        if regime == 'persistent' and case.mode != L.EPI_ATOMIC_F32:
            first = [t.clone() for t in (case.out, case.out2) if t is not None]
            case.reset()
            run(lib, case)
            again = [t for t in (case.out, case.out2) if t is not None]
            for a, b in zip(first, again):
                assert torch.equal(O.bits(a), O.bits(b)), f'{O.key_name(key)}: a second launch differs'


@pytest.mark.parametrize('case_def', O.MODEL_CASES, ids=[c[0] for c in O.MODEL_CASES])
def test_model_shapes_match_fp64(lib, case_def):
    name, M, N, K, a_k, b_k, mode, o = case_def
    case = O.Case(M, N, K, a_k, b_k, mode, L.BF16, seed=5, **O.model_case_options(o))
    run(lib, case)
    O.check(case, what=name)


@pytest.mark.parametrize('layout', O.LAYOUTS, ids=lambda l: f'a{l[0]}b{l[1]}')
@pytest.mark.parametrize('inst', O.ffma_instantiations(), ids=lambda i: O.MODE_NAMES[i[0]] + ('-path' if i[1] else ''))
def test_ffma_matches_fp64(lib, inst, layout):
    mode, path = inst
    for si, (M, N, K, opts) in enumerate(O.FFMA_SHAPES):
        case = O.Case(M, N, K, layout[0], layout[1], mode, L.F32, seed=3 + si, **ffma_opts(opts, path, M))
        run(lib, case)
        O.check(case, what=f'ffma shape {si}')


# ---- which kernel ran ---------------------------------------------------------------------------------------------
TC_RE = re.compile(r'gemm_tc2_kernel<\s*(\d+)\s*,\s*(true|false)\s*,\s*(true|false)\s*,\s*(\d+)\s*,\s*(true|false)\s*>')
FFMA_RE = re.compile(r'gemm_ffma_kernel<\s*(\d+)\s*(?:,\s*([^>]*))?>')


def kernel_key(name):
    m = TC_RE.search(name)
    if m:
        return ('tc', int(m.group(1)), m.group(2) == 'true', m.group(3) == 'true', int(m.group(4)), m.group(5) == 'true')
    m = FFMA_RE.search(name)
    if m:
        return ('ffma', int(m.group(1)), 'EpiPathParams' in (m.group(2) or ''))
    return None


def test_every_case_runs_the_predicted_kernel_and_every_kernel_runs(lib, sms):
    """one call per sweep case under the profiler: each ran the instantiation `plan` predicted, and together they ran
    all 34 tcgen05 instantiations and all seven FFMA kernels (a new instantiation shows up here as untested)"""
    from torch.profiler import profile, ProfilerActivity
    cases = sweep_cases(sms)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for name, want, make in cases:
            case = make()
            run(lib, case)
            torch.cuda.synchronize()
            del case
    events = sorted((e for e in prof.events() if kernel_key(e.name) is not None), key=lambda e: e.time_range.start)
    names = [e.name for e in events]
    assert len(events) == len(cases), f'{len(events)} GEMM kernels for {len(cases)} calls: {sorted(set(names))[:6]}'
    wrong = [(name, want, kernel_key(e.name)) for (name, want, _), e in zip(cases, events) if kernel_key(e.name) != want]
    assert not wrong, f'{len(wrong)} cases ran another kernel than planned, e.g. {wrong[:4]}'
    ran = {kernel_key(n) for n in names}
    every = {('tc',) + k for k in O.tc_instantiations()} | {('ffma',) + k for k in O.ffma_instantiations()}
    assert ran == every, f'not run: {sorted(every - ran)}; unknown: {sorted(ran - every)}'
    print(f'{len(cases)} cases, {len(ran)} kernels, e.g. {names[0]}')


# ---- graphs and streams -------------------------------------------------------------------------------------------
GRAPH_FAMILIES = [(False, False, L.EPI_STORE, False), (False, False, L.EPI_BIAS_RES, False),
                  (False, False, L.EPI_BIAS_GELU, False), (False, False, L.EPI_BIAS_SUB_ROWSQ, False),
                  (False, True, L.EPI_DGELU, False), (False, False, L.EPI_BIAS_RES_F32, False),
                  (False, False, L.EPI_BIAS_RES, True)]


def persistent_cases(sms):
    """one persistent GEMM per width and epilogue family, with dropout on (the split-K epilogue is left out: its fp32
    partial sums land in whatever order the splits finish, so it is not bit-reproducible by design)"""
    cases = []
    for bn in O.WIDTHS:
        for a_mn, b_mn, mode, path in GRAPH_FAMILIES:
            key = (bn, a_mn, b_mn, mode, path)
            if key not in O.tc_instantiations():
                continue
            M, N, K, opts = O.sweep_specs(key, 'persistent', sms)[1]
            cases.append(tc_case(key, M, N, K, opts, seed=bn + mode))
    return cases


def outputs(case):
    return [t for t in (case.out, case.out2) if t is not None]


def test_graph_replay_matches_eager_bit_for_bit(lib, sms):
    """the scheduler counters re-arm at the end of every launch: three replays of one captured graph holding a
    persistent GEMM of each width and epilogue family give the eager results bit for bit"""
    cases = persistent_cases(sms)
    eager = []
    for c in cases:
        run(lib, c)
        eager.append([t.clone() for t in outputs(c)])
    for c, want in zip(cases, eager):
        O.check(c, out=want[0], out2=want[1] if len(want) > 1 else None, what='eager')
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        for c in cases:
            for t in outputs(c):
                t.fill_(float('nan'))
        with torch.cuda.graph(graph, stream=side):
            for c in cases:
                L.check(c.launch(lib, side.cuda_stream), 'gemm')
    torch.cuda.current_stream().wait_stream(side)
    for rep in range(3):
        for c in cases:
            for t in outputs(c):
                t.fill_(float('nan'))
        graph.replay()
        torch.cuda.synchronize()
        for c, want in zip(cases, eager):
            for got, w in zip(outputs(c), want):
                assert torch.equal(O.bits(got), O.bits(w)), f'replay {rep}: {O.MODE_NAMES[c.mode]} M={c.M} N={c.N}'


def test_two_streams_at_once_match_eager(lib, sms):
    """two persistent GEMMs running at the same time on two streams (each takes its own scheduler counters)"""
    keys = [(128, False, False, L.EPI_BIAS_GELU, False), (256, False, False, L.EPI_BIAS_RES, False)]
    cases = [tc_case(k, *O.sweep_specs(k, 'persistent', sms)[1], seed=i) for i, k in enumerate(keys)]
    eager = []
    for c in cases:
        run(lib, c)
        eager.append([t.clone() for t in outputs(c)])
        for t in outputs(c):
            t.fill_(float('nan'))
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    for s in streams:
        s.wait_stream(torch.cuda.current_stream())
    for c, s in zip(cases, streams):
        L.check(c.launch(lib, s.cuda_stream), 'gemm')
    torch.cuda.synchronize()
    for c, want in zip(cases, eager):
        for got, w in zip(outputs(c), want):
            assert torch.equal(O.bits(got), O.bits(w)), f'two streams: {O.MODE_NAMES[c.mode]} M={c.M} N={c.N}'


# ---- rejections ---------------------------------------------------------------------------------------------------
def rejections():
    bf, f32 = L.BF16, L.F32
    R = []
    for mode in (L.EPI_BIAS_RES, L.EPI_BIAS_GELU, L.EPI_BIAS_SUB_ROWSQ, L.EPI_BIAS_RES_F32):
        for a_k, b_k in ((0, 1), (1, 0), (0, 0)):
            R.append((f'{O.MODE_NAMES[mode]}-a{a_k}b{b_k}', dict(M=300, N=200, K=72, a_k=a_k, b_k=b_k, mode=mode, dtype=bf),
                      {}))
    R += [
        ('res_f32-fp32-mode', dict(M=100, N=64, K=40, a_k=1, b_k=1, mode=L.EPI_BIAS_RES, dtype=f32),
         dict(epilogue=L.EPI_BIAS_RES_F32)),
        ('split-k-without-atomic', dict(M=300, N=200, K=640, a_k=1, b_k=1, mode=L.EPI_STORE, dtype=bf), dict(split_k=2)),
        ('split-k-without-atomic-res', dict(M=300, N=200, K=640, a_k=1, b_k=1, mode=L.EPI_BIAS_RES, dtype=bf),
         dict(split_k=3)),
        ('drop-path-store', dict(M=300, N=200, K=72, a_k=1, b_k=1, mode=L.EPI_STORE, dtype=bf, path_rate=0.3), {}),
        ('drop-path-gelu', dict(M=300, N=200, K=72, a_k=1, b_k=1, mode=L.EPI_BIAS_GELU, dtype=bf, path_rate=0.3), {}),
        ('drop-path-dgelu-fp32', dict(M=100, N=64, K=40, a_k=1, b_k=0, mode=L.EPI_DGELU, dtype=f32, path_rate=0.3), {}),
        ('drop-path-mn-major', dict(M=300, N=200, K=72, a_k=0, b_k=1, mode=L.EPI_BIAS_RES, dtype=bf, path_rate=0.3), {}),
        ('n-not-multiple-of-8', dict(M=300, N=200, K=72, a_k=1, b_k=1, mode=L.EPI_STORE, dtype=bf), dict(N=196)),
        ('lda-not-multiple-of-8', dict(M=300, N=200, K=72, a_k=1, b_k=1, mode=L.EPI_STORE, dtype=bf), dict(K=68, lda=76)),
        ('misaligned-a', dict(M=300, N=200, K=72, a_k=1, b_k=1, mode=L.EPI_STORE, dtype=bf), dict(A='+2')),
        ('misaligned-b', dict(M=300, N=200, K=72, a_k=1, b_k=1, mode=L.EPI_STORE, dtype=bf), dict(B='+8')),
        ('misaligned-out', dict(M=300, N=200, K=72, a_k=1, b_k=1, mode=L.EPI_STORE, dtype=bf), dict(out='+2')),
        ('fp32-n-not-multiple-of-4', dict(M=100, N=64, K=40, a_k=1, b_k=1, mode=L.EPI_STORE, dtype=f32), dict(N=62)),
    ]
    return R


@pytest.mark.parametrize('name,spec,override', rejections(), ids=[r[0] for r in rejections()])
def test_unsupported_combinations_are_refused_without_writing(lib, name, spec, override):
    spec = dict(spec)
    M, N, K, a_k, b_k, mode, dtype = (spec.pop(k) for k in ('M', 'N', 'K', 'a_k', 'b_k', 'mode', 'dtype'))
    path = spec.pop('path_rate', 0.0)
    # the residual epilogues need aux, GELU out2: build the case with them so that only the tested argument is wrong
    build_mode = L.EPI_BIAS_RES if mode == L.EPI_BIAS_RES_F32 and dtype == L.F32 else mode
    case = O.Case(M, N, K, a_k, b_k, build_mode, dtype, p=0.1, site=1, path_rate=path, rpr=51, path_site=O.PATH_SITE)
    ov = {}
    for k, v in override.items():
        if isinstance(v, str):
            base = {'A': case.A, 'B': case.B, 'out': case.out}[k]
            ov[k] = base.data_ptr() + int(v)
        else:
            ov[k] = v
    torch.cuda.synchronize()
    before = [t.clone() for t in outputs(case)]
    rc = case.launch(lib, stream(), **ov)
    torch.cuda.synchronize()
    assert rc < 0, f'{name}: accepted (rc {rc})'
    assert L.last_error(), f'{name}: refused without a message'
    for got, w in zip(outputs(case), before):
        assert torch.equal(O.bits(got), O.bits(w)), f'{name}: refused call wrote its output'
