"""The GEMM's launch plan, an fp64 reference of its epilogues and an element-wise checker.

Shared by tests/test_gemm_plan_host.py (CPU) and tests/test_gpu_gemm_conformance.py (B200):

* `plan` is a host replica of the tile-width and split-K choice of `gemm_bf16_tc` (csrc/gemm_tc.cu), so a test can
  pick shapes that land on a given `gemm_tc2_kernel<BN, A_MN, B_MN, MODE, kPath>` instantiation without forcing one;
* `reference` evaluates every epilogue in float64 from the operands as stored, with the kernels' dropout and drop-path
  draws (`_lib.dropout_keep_mask`, the host replica of the counter hash);
* `check` compares every element against |out - ref| <= c_out |ref| + c_acc K (|A| |B|)_ij (+ the small terms
  documented there), checks the elements that dropout or drop path zeroed exactly, and requires every element outside
  [M, N] of the output buffers to still hold its sentinel.
"""
import ctypes
import math

import torch

from ecg_b200 import _lib as L

BM, BK = 128, 64           # rows per CTA and k block of the tcgen05 kernel: work units are 256-row pair tiles
WIDTHS = (128, 192, 256)
MODE_NAMES = {L.EPI_STORE: 'store', L.EPI_BIAS_RES: 'res', L.EPI_BIAS_GELU: 'gelu', L.EPI_DGELU: 'dgelu',
              L.EPI_ATOMIC_F32: 'atomic', L.EPI_BIAS_RES_F32: 'res_f32', L.EPI_BIAS_SUB_ROWSQ: 'rowsq'}
DROPOUT_MODES = (L.EPI_BIAS_RES, L.EPI_BIAS_GELU, L.EPI_DGELU, L.EPI_BIAS_RES_F32)   # epilogues that apply nn.Dropout
BIAS_MODES = (L.EPI_STORE, L.EPI_BIAS_RES, L.EPI_BIAS_GELU, L.EPI_BIAS_RES_F32, L.EPI_BIAS_SUB_ROWSQ)
AUX_MODES = (L.EPI_BIAS_RES, L.EPI_DGELU, L.EPI_BIAS_RES_F32, L.EPI_BIAS_SUB_ROWSQ)

C_OUT = {L.BF16: 2.0 ** -8, L.F32: 2.0 ** -22}   # rounding of the stored result, relative to |ref|
C_ACC = 2.0 ** -22        # fp32 accumulation over K (4 x the unit roundoff of a round-to-nearest add per term)
C_FP32 = 2.0 ** -22       # fp32 epilogue arithmetic (bias / residual adds, dropout scale) relative to its operands
C_FN = 2.0 ** -21         # erf of the GELU epilogues: Abramowitz-Stegun 7.1.26 is within 1.5e-7 of erf (tcgen05)
GELU_MAX_SLOPE = 1.13     # max |gelu'(u)| (at u = sqrt(2)): how far an accumulation error moves gelu(u)


def cdiv(a, b):
    return -(-a // b)


def plan(M, N, K, a_kmajor, b_kmajor, epilogue, split_k, sms):
    """(BN, split_k) that `gemm_bf16_tc` launches for this problem on a device with `sms` SMs (clusters = sms // 2):
    the auto split-K search of the atomic epilogue, the clamp that leaves every split at least one k block, then the
    tile width with the fewest (waves x BN / staging efficiency); 256 is never chosen for the fp32-residual epilogue
    (`wide_ok`), and N <= 128 always takes 128."""
    clusters = sms // 2
    kb_total = cdiv(K, BK)
    split = split_k if split_k > 1 else 1
    if epilogue == L.EPI_ATOMIC_F32 and split_k <= 0:
        tiles = cdiv(M, 2 * BM) * cdiv(N, 256)
        best, best_eff = 1, 0.0
        s = 1
        while s <= 32 and s * 8 <= kb_total:
            units = tiles * s
            eff = units / (cdiv(units, clusters) * clusters)
            if eff > best_eff + 1e-9:
                best_eff, best = eff, s
            if eff >= 0.9:
                best = s
                break
            s += 1
        split = best
    split = min(split, kb_total)
    while split > 1 and cdiv(kb_total, split) * (split - 1) >= kb_total:
        split -= 1
    tiles_m2 = cdiv(M, 2 * BM)

    def score(bn, eff):
        units = tiles_m2 * cdiv(N, bn) * split
        return cdiv(units, clusters) * bn / eff

    s256 = score(256, 1.0) if epilogue != L.EPI_BIAS_RES_F32 else 1e30
    s192 = score(192, 0.88 if b_kmajor else 0.82)
    s128 = score(128, 0.67)
    if N <= 128 or (s128 < s256 and s128 < s192):
        return 128, split
    return (192 if s192 < s256 else 256), split


def units(M, N, bn, split):
    return cdiv(M, 2 * BM) * cdiv(N, bn) * split


# ---- the instantiations -------------------------------------------------------------------------------------------
# (A_MN, B_MN, MODE) of dispatch_pair's plain cases; every width compiles these, and the drop-path BIAS_RES kernel
TC_LAYOUT_MODES = [(False, False, L.EPI_STORE), (False, False, L.EPI_BIAS_RES), (False, False, L.EPI_BIAS_GELU),
                   (False, False, L.EPI_BIAS_SUB_ROWSQ), (False, True, L.EPI_STORE), (False, True, L.EPI_DGELU),
                   (True, True, L.EPI_ATOMIC_F32), (True, True, L.EPI_STORE), (True, False, L.EPI_STORE)]


def tc_instantiations():
    """(BN, A_MN, B_MN, MODE, kPath) of every gemm_tc2_kernel csrc/gemm_tc.cu compiles: 12 at BN = 128 and 192, 10 at
    BN = 256 (no fp32-residual epilogue there, with or without drop path)"""
    keys = []
    for bn in WIDTHS:
        keys += [(bn, a, b, m, False) for a, b, m in TC_LAYOUT_MODES]
        keys.append((bn, False, False, L.EPI_BIAS_RES, True))
        if bn < 256:
            keys += [(bn, False, False, L.EPI_BIAS_RES_F32, False), (bn, False, False, L.EPI_BIAS_RES_F32, True)]
    return keys


def ffma_instantiations():
    """(MODE, kPath) of every gemm_ffma_kernel csrc/gemm_simt.cu compiles: six epilogues and the drop-path BIAS_RES"""
    return [(m, False) for m in (L.EPI_STORE, L.EPI_BIAS_RES, L.EPI_BIAS_GELU, L.EPI_DGELU, L.EPI_ATOMIC_F32,
                                 L.EPI_BIAS_SUB_ROWSQ)] + [(L.EPI_BIAS_RES, True)]


def key_name(key):
    bn, a_mn, b_mn, mode, path = key
    lay = ('m' if a_mn else 'k') + ('m' if b_mn else 'k')
    return f'bn{bn}-{lay}-{MODE_NAMES[mode]}' + ('-path' if path else '')


# ---- shape search -------------------------------------------------------------------------------------------------
# N = 64 j + 40: a partial last 32-column unit (8 columns) and a partial last 64-column group in every candidate
TAIL_NS = tuple(64 * j + 40 for j in range(300))
SMALL_MS = (1, 129, 255)                  # below one 256-row pair tile
SMALL_MS_2 = (129, 255, 383, 700)         # one or a few pair tiles, the last partial
# 128-wide tiles win over two or more waves only when those are exactly two full waves: 148 tiles of 256 x 128 at
# 74 clusters (e.g. 4 row tiles x 37 column tiles, or 148 row tiles of N <= 128)
PERSISTENT_MS = (300, 700, 1000, 2100, 4200, 8300, 37800)
PERSISTENT_MS_2 = (255, 1000, 2100, 4200, 8300)


def find_shape(key, Ms, Ns, K, sms, split_k=1, min_units=0):
    """the smallest (M * N, then M, then N) shape of the candidate grid on which `plan` picks the width of `key`;
    with min_units, only shapes with at least that many work units and a partial last column tile.  None if none."""
    bn, a_mn, b_mn, mode, _ = key
    best = None
    for M in Ms:
        for N in Ns:
            if best is not None and M * N > best[0]:
                break                       # Ns ascend
            pbn, split = plan(M, N, K, not a_mn, not b_mn, mode, split_k, sms)
            if pbn != bn:
                continue
            if min_units and (units(M, N, bn, split) < min_units or N % bn == 0):
                continue
            cand = (M * N, M, N)
            if best is None or cand < best:
                best = cand
    return None if best is None else (best[1], best[2], K)


PATH_RATE, PATH_SITE = 0.3, 9
# two option sets per regime: bias on / NULL, ldo = N or N + 64, dropout off / 0.1 / 0.5 at a site > 0, drop-path records
# of 51 rows, 1 row or all M rows, and for the split-K epilogue split_k = 0 (auto), 3 (K = 420: 7 k blocks, not a
# multiple), 1 and 6 (7 k blocks: the clamp that leaves every split a k block reduces it to 4)
REGIMES = {
    'small': [dict(Ms=SMALL_MS, K=37, bias=True, ldo_pad=64, p=0.5, site=3, rpr=51, split_k=0, atomic_K=37),
              dict(Ms=SMALL_MS_2, K=200, bias=False, ldo_pad=0, p=0.0, site=0, rpr=1, split_k=3, atomic_K=420)],
    'persistent': [dict(Ms=PERSISTENT_MS, K=136, bias=False, ldo_pad=0, p=0.1, site=2, rpr='M', split_k=1,
                        atomic_K=1000),
                   dict(Ms=PERSISTENT_MS_2, K=328, bias=True, ldo_pad=64, p=0.1, site=5, rpr=51, split_k=6,
                        atomic_K=420)],
}


def sweep_specs(key, regime, sms):
    """[(M, N, K, Case options)] of one instantiation in one regime: the smallest candidate shape on which `plan` picks
    the instantiation's width.  'persistent' shapes have at least two work units per cluster and a partial last column
    tile, so every cluster walks several tiles."""
    bn, a_mn, b_mn, mode, path = key
    specs = []
    for v in REGIMES[regime]:
        atomic = mode == L.EPI_ATOMIC_F32
        K = v['atomic_K'] if atomic else v['K']
        split = v['split_k'] if atomic else 1
        min_units = 2 * (sms // 2) if regime == 'persistent' else 0
        shape = find_shape(key, v['Ms'], TAIL_NS, K, sms, split_k=split, min_units=min_units)
        if shape is None:
            raise AssertionError(f'no {regime} shape for {key_name(key)} at {sms} SMs')
        M, N, K = shape
        opts = dict(bias=v['bias'], ldo_pad=v['ldo_pad'], p=v['p'], site=v['site'], split_k=split)
        if path:
            opts.update(path_rate=PATH_RATE, path_site=PATH_SITE, rpr=M if v['rpr'] == 'M' else v['rpr'])
        specs.append((M, N, K, opts))
    return specs


# The contractions the models run, with dropout p = 0.1 where the epilogue applies it.  cfg2: 256 records x 51 tokens
# (M = 13056), d 768, FF 3072; per-lead tokens: 4 records x 2401 tokens; MAE decoder: width 256, FF 1024, predicting
# 600-value patches.  (name, M, N, K, a_kmajor, b_kmajor, epilogue, options)
M_CFG2, M_LEAD = 256 * 51, 4 * 2401
MODEL_CASES = [
    ('cfg2-qkv', M_CFG2, 2304, 768, 1, 1, L.EPI_STORE, {}),
    ('cfg2-out-proj', M_CFG2, 768, 768, 1, 1, L.EPI_BIAS_RES, {}),
    ('cfg2-out-proj-res32', M_CFG2, 768, 768, 1, 1, L.EPI_BIAS_RES_F32, {}),
    ('cfg2-out-proj-path', M_CFG2, 768, 768, 1, 1, L.EPI_BIAS_RES, dict(path_rate=PATH_RATE, rpr=51)),
    ('cfg2-ff1', M_CFG2, 3072, 768, 1, 1, L.EPI_BIAS_GELU, {}),
    ('cfg2-ff2', M_CFG2, 768, 3072, 1, 1, L.EPI_BIAS_RES, {}),
    ('cfg2-ff2-res32-path', M_CFG2, 768, 3072, 1, 1, L.EPI_BIAS_RES_F32, dict(path_rate=PATH_RATE, rpr=51)),
    ('cfg2-ff1-dgrad', M_CFG2, 3072, 768, 1, 0, L.EPI_DGELU, {}),
    ('cfg2-ff2-dgrad', M_CFG2, 768, 3072, 1, 0, L.EPI_STORE, {}),
    ('cfg2-qkv-wgrad', 2304, 768, M_CFG2, 0, 0, L.EPI_ATOMIC_F32, dict(split_k=0)),
    ('cfg2-out-proj-wgrad', 768, 768, M_CFG2, 0, 0, L.EPI_ATOMIC_F32, dict(split_k=0)),
    ('cfg2-ff1-wgrad', 3072, 768, M_CFG2, 0, 0, L.EPI_ATOMIC_F32, dict(split_k=0)),
    ('cfg2-ff2-wgrad', 768, 3072, M_CFG2, 0, 0, L.EPI_ATOMIC_F32, dict(split_k=0)),
    ('lead-qkv', M_LEAD, 2304, 768, 1, 1, L.EPI_STORE, {}),
    ('lead-out-proj-path', M_LEAD, 768, 768, 1, 1, L.EPI_BIAS_RES, dict(path_rate=PATH_RATE, rpr=2401)),
    ('lead-ff1', M_LEAD, 3072, 768, 1, 1, L.EPI_BIAS_GELU, {}),
    ('mae-dec-qkv', M_CFG2, 768, 256, 1, 1, L.EPI_STORE, {}),
    ('mae-dec-out-proj', M_CFG2, 256, 256, 1, 1, L.EPI_BIAS_RES, {}),
    ('mae-dec-ff1', M_CFG2, 1024, 256, 1, 1, L.EPI_BIAS_GELU, {}),
    ('mae-dec-ff2', M_CFG2, 256, 1024, 1, 1, L.EPI_BIAS_RES, {}),
    ('mae-dec-ff1-dgrad', M_CFG2, 1024, 256, 1, 0, L.EPI_DGELU, {}),
    ('mae-pred-rowsq', M_CFG2, 600, 256, 1, 1, L.EPI_BIAS_SUB_ROWSQ, {}),
]


def model_case_options(opts):
    o = dict(bias=True, ldo_pad=0, p=0.1, site=1, split_k=1)
    o.update(opts)
    if o.get('path_rate'):
        o['path_site'] = PATH_SITE
    return o


# FFMA (fp32) sweep: tails of M, N and K against the 64 x 64 x 16 tile, ldo = N + 64, dropout
FFMA_SHAPES = [(65, 68, 17, dict(bias=True, ldo_pad=64, p=0.5, site=3, rpr=51)),
               (130, 132, 40, dict(bias=False, ldo_pad=0, p=0.0, site=0, rpr=1)),
               (1, 4, 1, dict(bias=True, ldo_pad=0, p=0.1, site=6, rpr='M'))]
LAYOUTS = [(1, 1), (1, 0), (0, 0), (0, 1)]


# ---- operands -----------------------------------------------------------------------------------------------------
def round8(n):
    return cdiv(n, 8) * 8


def bits(t):
    """integer view of a tensor's bits (NaN payloads and signed zeros compare exactly)"""
    return t.view({torch.bfloat16: torch.int16, torch.float32: torch.int32, torch.float64: torch.int64}[t.dtype])


class Case:
    """one GEMM call: shape, layout, epilogue and epilogue options, plus the device buffers it reads and writes.

    Operands are stored with padded leading dimensions where the layout allows (the padding is NaN, so a read past
    K or past M / N of an MN-major operand poisons the result); out / out2 are [M + 1, ldo] buffers (a guard row)
    filled with a NaN sentinel, except the split-K accumulator, which starts at random values with a guard of 0.5."""

    def __init__(self, M, N, K, a_kmajor, b_kmajor, mode, dtype, bias=True, ldo_pad=0, p=0.0, site=0, path_rate=0.0,
                 rpr=1, path_site=0, split_k=1, seed=0, device='cuda'):
        self.M, self.N, self.K = M, N, K
        self.a_kmajor, self.b_kmajor, self.mode, self.dtype = a_kmajor, b_kmajor, mode, dtype
        self.has_bias = bias and mode in BIAS_MODES
        self.p = p if mode in DROPOUT_MODES else 0.0
        self.site, self.path_rate, self.rpr, self.path_site = site, path_rate, rpr, path_site
        self.split_k = split_k
        self.ldo = N + ldo_pad
        self.seed_value = 0x1234567 + 7919 * seed
        self.device = device
        td = torch.bfloat16 if dtype == L.BF16 else torch.float32
        self.td = td
        g = torch.Generator(device=device).manual_seed(1000 + seed)
        # stored operands with a NaN-padded leading dimension (a multiple of 8 elements: 16 bytes of bf16)
        if a_kmajor:
            self.lda = round8(K + 1)
            self.A = torch.full((M, self.lda), float('nan'), device=device, dtype=td)
            self.A[:, :K] = torch.randn(M, K, device=device, generator=g).to(td)
        else:
            self.lda = round8(M + 1)
            self.A = torch.full((K, self.lda), float('nan'), device=device, dtype=td)
            self.A[:, :M] = torch.randn(K, M, device=device, generator=g).to(td)
        if b_kmajor:
            self.ldb = round8(K + 1)
            self.B = torch.full((N, self.ldb), float('nan'), device=device, dtype=td)
            self.B[:, :K] = torch.randn(N, K, device=device, generator=g).to(td)
        else:
            self.ldb = round8(N + 1)
            self.B = torch.full((K, self.ldb), float('nan'), device=device, dtype=td)
            self.B[:, :N] = torch.randn(K, N, device=device, generator=g).to(td)
        self.bias = torch.randn(N, device=device, generator=g) if self.has_bias else None
        out_td = torch.float32 if mode in (L.EPI_ATOMIC_F32, L.EPI_BIAS_RES_F32) else td
        self.out_td = out_td
        self.aux = None
        if mode in AUX_MODES:
            aux_td = torch.float32 if mode == L.EPI_BIAS_RES_F32 else td
            # padding columns of aux hold NaN: an epilogue that read them into a stored column would show it
            self.aux = torch.full((M + 1, self.ldo), float('nan'), device=device, dtype=aux_td)
            scale = 4.0 if mode == L.EPI_BIAS_RES_F32 else 1.0
            self.aux[:M, :N] = (torch.randn(M, N, device=device, generator=g) * scale).to(aux_td)
        self.out0 = None
        if mode == L.EPI_ATOMIC_F32:
            self.out0 = torch.full((M + 1, self.ldo), 0.5, device=device)
            self.out0[:M, :N] = torch.randn(M, N, device=device, generator=g)
        self.seed_dev = torch.tensor([self.seed_value], dtype=torch.int32, device=device)
        self.reset()

    def reset(self):
        M, N = self.M, self.N
        if self.mode == L.EPI_ATOMIC_F32:
            self.out = self.out0.clone()
        else:
            self.out = torch.full((M + 1, self.ldo), float('nan'), device=self.device, dtype=self.out_td)
        self.out2 = None
        if self.mode == L.EPI_BIAS_GELU:
            self.out2 = torch.full((M + 1, self.ldo), float('nan'), device=self.device, dtype=self.td)
        elif self.mode == L.EPI_BIAS_SUB_ROWSQ:
            self.out2 = torch.full((cdiv(N, 64) * M + 64,), float('nan'), device=self.device)

    def args(self, **override):
        kw = dict(M=self.M, N=self.N, K=self.K, A=self.A.data_ptr(), lda=self.lda, a_kmajor=int(self.a_kmajor),
                  B=self.B.data_ptr(), ldb=self.ldb, b_kmajor=int(self.b_kmajor), epilogue=self.mode,
                  out=self.out.data_ptr(), ldo=self.ldo, out2=L.ptr(self.out2), aux=L.ptr(self.aux),
                  bias=L.ptr(self.bias), dtype=self.dtype, split_k=self.split_k, dropout_stream=self.site,
                  dropout_p=self.p, dropout_seed=self.seed_dev.data_ptr() if self.p > 0 or self.path_rate > 0 else None)
        kw.update(override)
        return L.GemmArgs(**kw)

    def launch(self, lib, stream, **override):
        """the return code of ecgvit_gemm (or ecgvit_gemm_drop_path when the case has a drop-path rate)"""
        g = self.args(**override)
        if self.path_rate > 0:
            return lib.ecgvit_gemm_drop_path(ctypes.byref(g), self.path_rate, self.path_site, self.rpr, stream)
        return lib.ecgvit_gemm(ctypes.byref(g), stream)

    # ---- the fp64 reference -----------------------------------------------------------------------------------------
    def operands64(self):
        M, N, K = self.M, self.N, self.K
        A = self.A[:, :K].double() if self.a_kmajor else self.A[:, :M].double().t()
        B = self.B[:, :K].double() if self.b_kmajor else self.B[:, :N].double().t()
        return A, B

    def keep(self, ld=None, shift=0):
        """fp64 [M, N] dropout multipliers (0 or 1/(1-p)) of element index row * ld + col (ld = ldo)"""
        M, N = self.M, self.N
        if self.p <= 0:
            return torch.ones(M, N, dtype=torch.float64, device=self.device)
        ld = self.ldo if ld is None else ld
        idx = (torch.arange(M, device=self.device).view(-1, 1) * ld + torch.arange(N, device=self.device)) + shift
        return L.dropout_keep_mask(self.seed_value, self.site, self.p, idx).double()

    def path_factors(self):
        """fp64 [M, 1] drop-path factors of the rows (1 without drop path)"""
        if self.path_rate <= 0:
            return torch.ones(self.M, 1, dtype=torch.float64, device=self.device)
        rec = torch.arange(self.M, device=self.device) // self.rpr
        return L.dropout_keep_mask(self.seed_value, self.path_site, self.path_rate, rec).double().view(-1, 1)

    def reference(self):
        """dict of fp64 expectations and error scales for `check`"""
        M, N, K = self.M, self.N, self.K
        A, B = self.operands64()
        acc = A @ B.t()
        absab = A.abs() @ B.abs().t()
        bias = self.bias.double() if self.bias is not None else torch.zeros(N, dtype=torch.float64, device=self.device)
        aux = self.aux[:M, :N].double() if self.aux is not None else None
        keep, s = self.keep(), self.path_factors()
        return dict(acc=acc, absab=absab, bias=bias, aux=aux, keep=keep, s=s)


def gelu64(u):
    return 0.5 * u * (1.0 + torch.special.erf(u / math.sqrt(2.0)))


def gelu_grad64(u):
    return 0.5 * (1.0 + torch.special.erf(u / math.sqrt(2.0))) + u * torch.exp(-0.5 * u * u) / math.sqrt(2.0 * math.pi)


def expected(case, r):
    """fp64 expectations {name: (ref [.., ..], bound [.., ..])} of the case's outputs from reference() parts `r`.

    bound = c_out |ref| + c_acc K gain (|A||B|) + c_fp32 gain (|acc| + |bias| + |aux|) (+ c_fn for the erf of the GELU
    epilogues), where gain is how much the epilogue scales an error of the accumulator (dropout and drop-path scales,
    the slope of GELU)."""
    mode, K = case.mode, case.K
    c_out = C_OUT[L.F32 if case.out_td == torch.float32 else case.dtype]
    acc, absab, bias, aux, keep, s = r['acc'], r['absab'], r['bias'], r['aux'], r['keep'], r['s']
    scale = (1.0 / (1.0 - case.p) if case.p > 0 else 1.0) * (1.0 / (1.0 - case.path_rate) if case.path_rate > 0 else 1.0)
    acc_err = C_ACC * K * absab
    res = {}
    if mode == L.EPI_STORE:
        ref = acc + bias
        res['out'] = (ref, c_out * ref.abs() + acc_err + C_FP32 * (acc.abs() + bias.abs()))
    elif mode in (L.EPI_BIAS_RES, L.EPI_BIAS_RES_F32):
        u = acc + bias
        ref = s * keep * u + aux
        res['out'] = (ref, c_out * ref.abs() + scale * (acc_err + C_FP32 * (acc.abs() + bias.abs())) + C_FP32 * aux.abs())
    elif mode == L.EPI_BIAS_GELU:
        u = acc + bias
        e_u = acc_err + C_FP32 * (acc.abs() + bias.abs())
        res['out'] = (u, c_out * u.abs() + e_u)
        h = keep * gelu64(u)
        c2 = C_OUT[case.dtype]
        res['out2'] = (h, c2 * h.abs() + scale * (GELU_MAX_SLOPE * e_u + C_FN * (1.0 + u.abs())))
    elif mode == L.EPI_DGELU:
        gp = gelu_grad64(aux)
        ref = keep * acc * gp
        res['out'] = (ref, c_out * ref.abs() + scale * (GELU_MAX_SLOPE * acc_err + C_FN * acc.abs() * (1.0 + aux.abs())))
    elif mode == L.EPI_ATOMIC_F32:
        o0 = case.out0[:case.M, :case.N].double()
        ref = o0 + acc
        res['out'] = (ref, c_out * (ref.abs() + o0.abs()) + acc_err + C_FP32 * acc.abs())
    elif mode == L.EPI_BIAS_SUB_ROWSQ:
        ref = acc + bias - aux
        e = acc_err + C_FP32 * (acc.abs() + bias.abs() + aux.abs())
        res['out'] = (ref, c_out * ref.abs() + e)
        # fp32 squares of the fp32 residual, summed over 64-column groups: |v^2 - r^2| <= (2|r| + e) e per column, plus
        # the fp32 rounding of up to 64 squares and their sum
        G = cdiv(case.N, 64)
        pad = G * 64 - case.N
        sq = torch.nn.functional.pad(ref * ref, (0, pad)).view(case.M, G, 64).sum(-1).t()
        esq = torch.nn.functional.pad((2 * ref.abs() + e) * e, (0, pad)).view(case.M, G, 64).sum(-1).t()
        res['out2'] = (sq, esq + 2.0 ** -17 * sq + 1e-30)
    return res


def check(case, out=None, out2=None, r=None, what=''):
    """assert that the case's outputs (default: its device buffers) meet the fp64 reference element by element, that
    the elements dropout / drop path zeroed are exact, and that nothing outside [M, N] was written"""
    M, N = case.M, case.N
    out = case.out if out is None else out
    out2 = case.out2 if out2 is None else out2
    r = case.reference() if r is None else r
    exp = expected(case, r)
    tag = f'{what} M={M} N={N} K={case.K} ldo={case.ldo} mode={MODE_NAMES[case.mode]} p={case.p} path={case.path_rate}'

    def within(name, got, ref, bound):
        got = got.double()
        assert bool(torch.isfinite(got).all()), f'{tag}: {name} has non-finite elements in [M, N]'
        err = (got - ref).abs()
        bad = err > bound
        if bool(bad.any()):
            i = int(bad.nonzero()[0][0]), int(bad.nonzero()[0][1])
            raise AssertionError(f'{tag}: {name} {int(bad.sum())} elements out of bound, first at {i}: got '
                                 f'{float(got[i]):.6g} want {float(ref[i]):.6g} bound {float(bound[i]):.3g}')

    ref, bound = exp['out']
    within('out', out[:M, :N], ref, bound)
    # nothing written outside [M, N]: padding columns and the guard row keep their sentinel
    sentinel = case.out0 if case.mode == L.EPI_ATOMIC_F32 else torch.full_like(out, float('nan'))
    assert torch.equal(bits(out[:, N:]), bits(sentinel[:, N:])) and torch.equal(bits(out[M:]), bits(sentinel[M:])), \
        f'{tag}: out written outside [M, N]'
    if case.mode == L.EPI_BIAS_GELU:
        ref2, bound2 = exp['out2']
        within('out2', out2[:M, :N], ref2, bound2)
        assert bool(torch.isnan(out2[:, N:]).all()) and bool(torch.isnan(out2[M:]).all()), \
            f'{tag}: out2 written outside [M, N]'
    if case.mode == L.EPI_BIAS_SUB_ROWSQ:
        G = cdiv(N, 64)
        ref2, bound2 = exp['out2']
        within('rowsq', out2[:G * M].view(G, M), ref2, bound2)
        assert bool(torch.isnan(out2[G * M:]).all()), f'{tag}: row partials written past [ceil(N/64), M]'
    # exact checks where dropout / drop path zeroed the branch
    zero = (r['keep'] * r['s']) == 0
    if bool(zero.any()):
        if case.mode in (L.EPI_BIAS_RES, L.EPI_BIAS_RES_F32):
            got, aux = out[:M, :N], case.aux[:M, :N]
            assert torch.equal(bits(got)[zero], bits(aux)[zero]), f'{tag}: a dropped element is not exactly aux'
        elif case.mode == L.EPI_DGELU:
            assert bool((out[:M, :N][zero] == 0).all()), f'{tag}: a dropped element of dgelu is not 0'
        elif case.mode == L.EPI_BIAS_GELU:
            assert bool((out2[:M, :N][zero] == 0).all()), f'{tag}: a dropped element of gelu(out) is not 0'
    return exp
