"""The attention front door's launch plan, an fp64 reference of forward and backward and an element-wise checker.

Shared by tests/test_attention_plan_host.py (CPU) and tests/test_gpu_attention_conformance.py (B200):

* `plan` is a host replica of the dispatch in `ecgvit_attention_fwd / _bwd` (csrc/attention.cu): which family serves
  (dtype, N, dh), its template arguments, the kernels each call launches and the scratch floats backward needs;
* `reference` evaluates S, P, lse, O and dQ, dK, dV in float64 from the operands as stored (the bf16 or fp32 `qkv`,
  `d_o`, and for backward the stored `o` and `lse`), with the kernels' attention-probability dropout: the keep draw of
  element ((b H + h) Np + i) Np + j, Np = N rounded up to 64, from `_lib.dropout_keep_mask` (the host replica of the
  counter hash), kept probabilities scaled by the quantised 1 / (1 - thr / 65536).  It runs one block of (b, h)
  problems at a time on whatever device the case lives on, so N = 2401 fits;
* `check` compares every element against a bound built from the rounding steps the kernels take; `check_guards` and
  `check_inputs` require the NaN sentinels past every output to keep their bits and the inputs to be unchanged.

The bounds.  All are evaluated in fp64 from magnitudes, per element; u = 2^-8 is the unit roundoff of bf16.

* eS_i, the absolute error of any score S_ij = scale q_i . k_j of query row i: C_ACC dh scale max_j (|q_i| . |k_j|)
  for the fp32 dot product over dh terms, plus C_SCORE max_j |S_ij| for the fp32 products with scale and log2(e) and
  the FMA that subtracts the row maximum before the exponential.
* eps_i, the relative error of every probability of row i: 2 eS_i (the score and the row maximum it is taken
  against) + C_EXP (ex2.approx / expf) per rescale of a running maximum, and there are ceil(N / 64) key blocks at most.
* O:  |O - ref| <= c_out |ref| + (c_p + 3 eps_i + 2 C_ACC N) (|Pd| |V|)_i / l_i, where Pd is the dropped P and l its
  undropped row sum.  c_p = u on the tensor-core paths, which round P to bf16 before P V (the row sum is taken in
  fp32 before that rounding); the SIMT path keeps P in fp32, c_p = 0, and its fp32 accumulation over N keys is the
  C_ACC N term.  c_out = u for a bf16 output, C_F32_OUT for fp32.  3 eps_i: P, and l formed from the same P.
* lse: |lse - ref| <= eS_i + eps_i + C_ACC N + C_SCORE (|m_i| + |log l_i|): the score error moves the maximum, the
  relative error of l moves log l, and the final fp32 multiply-add and logf round.
* dV: c_out |ref| + ((c_p + eps_i + C_ACC N) |Pd_ij|)^T |dO|.
* dQ / dK: an error bound E on dS_ij = P_ij (dP_ij keep_ij - D_i) (the backward recomputes P from the stored lse):
  c_p |dS_ij| for its bf16 rounding (0 on the SIMT path) + eps_i P_ij (|keep dP_ij| + |D_i|) for the error of P +
  P_ij (E_dP_ij + E_D_i) for the dot products dP = dO . V (C_ACC dh (|dO_i| . |V_j|) keep_ij) and D.  Then
  dQ: c_out |ref| + scale (E |K|) + scale C_ACC N ((P (|keep dP| + |D|)) |K|), and dK the same with E^T and |Q|.
  D = rowsum(dO o O_stored).  Every path but tc packed reads the stored O, so E_D = C_ACC dh (|dO_i| . |O_i|).  tc
  packed forms D = sum_j Pd_ij dP_ij in the kernel from its own P and never reads O, so its E_D adds the distance of
  the stored O from the exact one (sum_d |dO_id| times the forward bound of O_id, with c_p = u: this is how far the
  stored O may be from what the kernel's own P gives) and (c_p + eps_i + C_ACC N + lse bound_i) sum_j P_ij |keep dP_ij|.

Constants:
  C_ACC = 2^-22      fp32 accumulation per term (4 x the unit roundoff; covers the tensor core's truncating alignment
                     and an FMA chain alike; as in gemm_oracle)
  C_SCORE = 2^-21    fp32 products and the FMA of the exponent argument, relative to the largest score of the row
  C_EXP = 2^-21      ex2.approx.f32 (max relative error 2^-22.5 by the PTX ISA) and CUDA's expf (2 ulp), with the
                     rounding of its fp32 argument
  C_F32_OUT = 2^-21  the fp32 normalisation (x 1 / l) and store of an fp32 output
"""
import math
from collections import namedtuple

import torch

from ecg_b200 import _lib as L

NMAX = 64                  # Np granularity of the dropout counter, and the longest sequence of the mma kernels
TC_DH = 64                 # the tcgen05 kernels serve head dim 64 only
FLASH_DHS = (32,)
MMA_DHS = (16, 32)
SIMT_SMEM_MAX = 227 * 1024

U_BF16 = 2.0 ** -8
C_ACC = 2.0 ** -22
C_SCORE = 2.0 ** -21
C_EXP = 2.0 ** -21
C_F32_OUT = 2.0 ** -21
GUARD = 64                 # sentinel elements after every output buffer (128 / 256 bytes: keeps 16-byte alignment)


def cdiv(a, b):
    return -(-a // b)


def padded(N):
    return cdiv(N, NMAX) * NMAX


# ---- the launch plan ----------------------------------------------------------------------------------------------
Plan = namedtuple('Plan', 'family targs fwd bwd scratch_floats')


def simt_smem(N, dh, bwd):
    """bytes of dynamic shared memory of the whole-sequence kernels (csrc/attention_simt.cu fwd_smem / bwd_smem)"""
    if bwd:
        return 4 * (4 * N * (dh + 1) + N * (N + 1) + N)
    return 4 * (3 * N * (dh + 1) + N * (N + 1))


def simt_max_len(dh, bwd):
    """the longest N the whole-sequence kernels accept"""
    N = 1
    while simt_smem(N + 1, dh, bwd) <= SIMT_SMEM_MAX:
        N += 1
    return N


def plan(dtype, N, dh, B=1, H=1):
    """which kernels `ecgvit_attention_fwd` / `_bwd` launch for (dtype, N, dh) and how many scratch floats backward
    needs at (B, H) (`ecgvit_attention_bwd_scratch_floats`).  Kernel names are 'base<args>' with the template arguments
    written as in the source (bf16 / float, true / false, no spaces)."""
    if dtype == L.BF16 and dh == TC_DH and N >= 1:
        if N <= NMAX:
            return Plan('tc_packed', ('true',), ['attn_tc_fwd_kernel<true>'], ['attn_tc_bwd_kernel<true>'], 0)
        d_floats = cdiv(B * H * N, 64) * 64
        return Plan('tc_long', ('false',), ['attn_tc_fwd_kernel<false>'],
                    ['attn_tc_dot_kernel', 'attn_tc_bwd_kernel<false>', 'attn_tc_dq_convert_kernel'],
                    d_floats + B * N * H * TC_DH)
    if dtype == L.BF16 and N <= NMAX and dh in MMA_DHS:
        nt = cdiv(N, 16)
        return Plan('mma', (dh, nt), [f'attention_fwd_mma_kernel<{dh},{nt}>'], [f'attention_bwd_mma_kernel<{dh},{nt}>'], 0)
    if dtype == L.BF16 and N > NMAX and dh in FLASH_DHS:
        return Plan('flash', (dh,), [f'flash_fwd_kernel<{dh}>'],
                    [f'flash_bwd_dot_kernel<{dh}>', f'flash_bwd_dq_kernel<{dh}>', f'flash_bwd_dkv_kernel<{dh}>'], B * H * N)
    t = 'bf16' if dtype == L.BF16 else 'float'
    return Plan('simt', (t,), [f'attention_fwd_simt_kernel<{t}>'], [f'attention_bwd_simt_kernel<{t}>'], 0)


def all_kernels():
    """the 32 attention kernels the library compiles"""
    ks = ['attn_tc_fwd_kernel<true>', 'attn_tc_fwd_kernel<false>', 'attn_tc_bwd_kernel<true>', 'attn_tc_bwd_kernel<false>',
          'attn_tc_dot_kernel', 'attn_tc_dq_convert_kernel']
    for dh in MMA_DHS:
        for nt in range(1, 5):
            ks += [f'attention_fwd_mma_kernel<{dh},{nt}>', f'attention_bwd_mma_kernel<{dh},{nt}>']
    for dh in FLASH_DHS:
        ks += [f'{k}<{dh}>' for k in ('flash_fwd_kernel', 'flash_bwd_dot_kernel', 'flash_bwd_dq_kernel',
                                      'flash_bwd_dkv_kernel')]
    for t in ('bf16', 'float'):
        ks += [f'attention_fwd_simt_kernel<{t}>', f'attention_bwd_simt_kernel<{t}>', f'attention_probs_kernel<{t}>']
    return ks


# ---- operands -----------------------------------------------------------------------------------------------------
def bits(t):
    """integer view of a tensor's bits (NaN payloads and signed zeros compare exactly)"""
    return t.view({torch.bfloat16: torch.int16, torch.float32: torch.int32, torch.float64: torch.int64}[t.dtype])


def guarded(n, dtype, device, fill=float('nan')):
    """(flat buffer of n + GUARD elements filled with `fill`, view of its first n)"""
    buf = torch.full((n + GUARD,), fill, dtype=dtype, device=device)
    return buf, buf[:n]


def heads(t, B, N, H, dh, part=0, parts=1):
    """[B*H, N, dh] view-copy of head part `part` of a [B*N, parts*H*dh] tensor (q | k | v, head-major)"""
    return t.reshape(B, N, parts, H, dh)[:, :, part].permute(0, 2, 1, 3).reshape(B * H, N, dh)


def quantised_p(p):
    thr = min(int(p * 65536.0 + 0.5), 65535)
    return thr


class Case:
    """one attention problem [B, N, H, dh] in one dtype with its device buffers: qkv / d_o inputs (random unless set),
    NaN-filled o / lse / dqkv with GUARD NaN elements after each, and NaN-filled scratch of the planned size."""

    def __init__(self, B, N, H, dh, dtype, scale=None, p=0.0, site=0, seed=0, amp=1.0,
                 device='cuda', null_seed=False):
        self.B, self.N, self.H, self.dh, self.dtype = B, N, H, dh, dtype
        self.inner = H * dh
        self.scale = dh ** -0.5 if scale is None else float(scale)
        self.p, self.site = float(p), site
        self.seed_value = 0x2545F49 + 7919 * seed
        self.null_seed = null_seed
        self.device = device
        self.td = torch.bfloat16 if dtype == L.BF16 else torch.float32
        self.plan = plan(dtype, N, dh, B, H)
        g = torch.Generator(device=device).manual_seed(2000 + seed)
        n_qkv, n_o = B * N * 3 * self.inner, B * N * self.inner
        self.qkv_buf, q = guarded(n_qkv, self.td, device)
        self.qkv = q.view(B * N, 3 * self.inner)
        self.qkv.copy_((torch.randn(B * N, 3 * self.inner, device=device, generator=g) * amp).to(self.td))
        self.do_buf, d = guarded(n_o, self.td, device)
        self.d_o = d.view(B * N, self.inner)
        self.d_o.copy_(torch.randn(B * N, self.inner, device=device, generator=g).to(self.td))
        self.seed_dev = torch.tensor([self.seed_value], dtype=torch.int32, device=device)
        self.reset()

    @property
    def family(self):
        return self.plan.family

    def reset(self, fwd=True, bwd=True):
        B, N, H = self.B, self.N, self.H
        if fwd:
            self.o_buf, o = guarded(B * N * self.inner, self.td, self.device)
            self.o = o.view(B * N, self.inner)
            self.lse_buf, lse = guarded(B * H * N, torch.float32, self.device)
            self.lse = lse.view(B, H, N)
        if bwd:
            self.dqkv_buf, dq = guarded(B * N * 3 * self.inner, self.td, self.device)
            self.dqkv = dq.view(B * N, 3 * self.inner)
            self.scratch = None
            if self.plan.scratch_floats:
                self.scratch = torch.full((self.plan.scratch_floats,), float('nan'), device=self.device)

    def seed_ptr(self):
        return None if self.null_seed or self.p <= 0 else self.seed_dev.data_ptr()

    def fwd(self, lib, stream, **ov):
        a = dict(qkv=self.qkv.data_ptr(), o=self.o.data_ptr(), lse=self.lse.data_ptr(), B=self.B, N=self.N, H=self.H,
                 dh=self.dh, scale=self.scale, p=self.p, site=self.site, seed=self.seed_ptr(), dtype=self.dtype)
        a.update(ov)
        return lib.ecgvit_attention_fwd(a['qkv'], a['o'], a['lse'], a['B'], a['N'], a['H'], a['dh'], a['scale'], a['p'],
                                        a['site'], a['seed'], a['dtype'], stream)

    def bwd(self, lib, stream, **ov):
        a = dict(qkv=self.qkv.data_ptr(), o=self.o.data_ptr(), d_o=self.d_o.data_ptr(), lse=self.lse.data_ptr(),
                 dqkv=self.dqkv.data_ptr(), scratch=L.ptr(self.scratch), B=self.B, N=self.N, H=self.H, dh=self.dh,
                 scale=self.scale, p=self.p, site=self.site, seed=self.seed_ptr(), dtype=self.dtype)
        a.update(ov)
        return lib.ecgvit_attention_bwd(a['qkv'], a['o'], a['d_o'], a['lse'], a['dqkv'], a['scratch'], a['B'], a['N'],
                                        a['H'], a['dh'], a['scale'], a['p'], a['site'], a['seed'], a['dtype'], stream)

    def outputs(self, bhs=None):
        """the kernels' results in reference layout: o / dq / dk / dv [nb, N, dh], lse [nb, N]"""
        B, N, H, dh = self.B, self.N, self.H, self.dh
        sel = (lambda t: t) if bhs is None else (lambda t: t[bhs])
        got = dict(o=sel(heads(self.o, B, N, H, dh)), lse=sel(self.lse.reshape(B * H, N)))
        for i, k in enumerate(('dq', 'dk', 'dv')):
            got[k] = sel(heads(self.dqkv, B, N, H, dh, i, 3))
        return got

    def keep(self, bhs, rows=None, cols=None, shift=0, pitch=None):
        """fp64 [nb, rows, cols] dropout multipliers (0 or the quantised 1 / (1 - p)) of problems bhs; `shift` and
        `pitch` (default Np) let a test build a wrongly indexed mask"""
        N = self.N
        rows = torch.arange(N, device=self.device) if rows is None else rows
        cols = torch.arange(N, device=self.device) if cols is None else cols
        dropping = self.p > 0 and not self.null_seed and quantised_p(self.p) > 0
        if not dropping:
            return torch.ones(len(bhs), len(rows), len(cols), dtype=torch.float64, device=self.device)
        Np = padded(N) if pitch is None else pitch
        bh = torch.as_tensor(bhs, device=self.device).to(torch.int64).view(-1, 1, 1)
        idx = (bh * Np + rows.view(1, -1, 1)) * Np + cols.view(1, 1, -1) + shift
        return L.dropout_keep_mask(self.seed_value, self.site, self.p, idx).double().to(self.device)


# ---- the fp64 reference -------------------------------------------------------------------------------------------
def forward64(q, k, v, scale, keep):
    """exact attention of [c, N, dh] problems: (S, P = exp(S - m), l, m, O, lse) with O = (P keep) V / l"""
    S = scale * (q @ k.transpose(-1, -2))
    m = S.amax(-1, keepdim=True)
    P = torch.exp(S - m)
    l = P.sum(-1, keepdim=True)
    O = (P * keep) @ v / l
    return S, P, l, m, O, (m + l.log()).squeeze(-1)


def backward64(q, k, v, do, scale, keep, lse, D):
    """exact gradients (dq, dk, dv, P, dPm, dS) of [c, N, dh] problems from the lse and D = rowsum(dO o O) given"""
    S = scale * (q @ k.transpose(-1, -2))
    P = torch.exp(S - lse.unsqueeze(-1))
    dPm = keep * (do @ v.transpose(-1, -2))
    dS = P * (dPm - D.unsqueeze(-1))
    return scale * (dS @ k), scale * (dS.transpose(-1, -2) @ q), (P * keep).transpose(-1, -2) @ do, P, dPm, dS


def c_p(case):
    return 0.0 if case.family == 'simt' else U_BF16


def c_out(case):
    return U_BF16 if case.dtype == L.BF16 else C_F32_OUT


def _fwd_bounds(case, q, k, v, keep, S, P, l, m, O):
    N, dh, sc = case.N, case.dh, case.scale
    qk = sc * (q.abs() @ k.abs().transpose(-1, -2))
    eS = C_ACC * dh * qk.amax(-1) + C_SCORE * S.abs().amax(-1)                       # [c, N]
    eps = 2 * eS + C_EXP * cdiv(N, 64)
    A = ((P * keep) @ v.abs()) / l                                                   # |Pd| |V| / l
    bO = c_out(case) * O.abs() + (c_p(case) + 3 * eps + 2 * C_ACC * N).unsqueeze(-1) * A
    blse = eS + eps + C_ACC * N + C_SCORE * (m.squeeze(-1).abs() + l.squeeze(-1).log().abs())
    return eS, eps, bO, blse


def reference(case, bhs=None, bwd=True, o_in=None, lse_in=None, chunk_elems=2 ** 25):
    """fp64 expectations and bounds {name: (ref, bound)} of problems `bhs` (default all) for `check`.

    Backward takes P from `lse_in` (default: the case's stored lse) and D from `o_in` (default: the case's stored o);
    pass o_in='exact' for a call whose o is not read (tc packed)."""
    B, N, H, dh = case.B, case.N, case.H, case.dh
    bhs = torch.arange(B * H) if bhs is None else torch.as_tensor(bhs)
    c = max(1, chunk_elems // (N * N))
    parts = {}
    for s in range(0, len(bhs), c):
        idx = bhs[s:s + c].to(case.device)
        q, k, v = (heads(case.qkv, B, N, H, dh, i, 3)[idx].double() for i in range(3))
        keep = case.keep(idx)
        S, P, l, m, O, lse = forward64(q, k, v, case.scale, keep)
        eS, eps, bO, blse = _fwd_bounds(case, q, k, v, keep, S, P, l, m, O)
        out = dict(o=(O, bO), lse=(lse, blse))
        if bwd:
            do = heads(case.d_o, B, N, H, dh)[idx].double()
            ls = case.lse.reshape(B * H, N)[idx].double() if lse_in is None else lse_in[s:s + c].double()
            if isinstance(o_in, str):
                Ost = O
            else:
                Ost = (heads(case.o, B, N, H, dh)[idx] if o_in is None else o_in[s:s + c]).double()
            D = (do * Ost).sum(-1)
            dq, dk, dv, Pb, dPm, dS = backward64(q, k, v, do, case.scale, keep, ls, D)
            eps_b = (eps + C_SCORE * ls.abs()).unsqueeze(-1)
            E_dP = keep * (C_ACC * dh) * (do.abs() @ v.abs().transpose(-1, -2))
            E_D = C_ACC * dh * (do.abs() * Ost.abs()).sum(-1)
            if case.family == 'tc_packed':
                absPdP = (Pb * dPm.abs()).sum(-1)
                E_D = E_D + (do.abs() * bO).sum(-1) + (U_BF16 + eps + C_ACC * N + blse) * absPdP
            absD = D.abs().unsqueeze(-1)
            mag = Pb * (dPm.abs() + absD)                                            # |dS| without cancellation
            E = c_p(case) * dS.abs() + eps_b * mag + Pb * (E_dP + E_D.unsqueeze(-1))
            sc = case.scale
            co = c_out(case)
            out['dq'] = (dq, co * dq.abs() + sc * (E @ k.abs()) + sc * C_ACC * N * (mag @ k.abs()))
            out['dk'] = (dk, co * dk.abs() + sc * (E.transpose(-1, -2) @ q.abs())
                         + sc * C_ACC * N * (mag.transpose(-1, -2) @ q.abs()))
            W = (Pb * keep) * (c_p(case) + eps_b + C_ACC * N)
            out['dv'] = (dv, co * dv.abs() + W.transpose(-1, -2) @ do.abs())
        for name, (r, b) in out.items():
            parts.setdefault(name, []).append((r, b))
    return {name: (torch.cat([r for r, _ in v]), torch.cat([b for _, b in v])) for name, v in parts.items()}


# ---- checks -------------------------------------------------------------------------------------------------------
def tag(case, what=''):
    return (f'{what} {case.family}{case.plan.targs} B={case.B} N={case.N} H={case.H} dh={case.dh} '
            f'dtype={"bf16" if case.dtype == L.BF16 else "f32"} scale={case.scale:.4g} p={case.p}')


def check(case, ref, got, names=('o', 'lse', 'dq', 'dk', 'dv'), what=''):
    """every element of got[name] within the bound of ref[name]; every element finite (the outputs start as NaN)"""
    for name in names:
        if name not in ref:
            continue
        r, b = ref[name]
        g = got[name].double()
        assert bool(torch.isfinite(g).all()), f'{tag(case, what)}: {name} has non-finite (unwritten) elements'
        bad = (g - r).abs() > b
        if bool(bad.any()):
            i = tuple(int(x) for x in bad.nonzero()[0])
            raise AssertionError(f'{tag(case, what)}: {name} {int(bad.sum())} elements out of bound, first at {i}: got '
                                 f'{float(g[i]):.6g} want {float(r[i]):.6g} bound {float(b[i]):.3g}')


def check_guards(case, fwd=True, bwd=True, what=''):
    """the GUARD elements after o, lse and dqkv still hold the NaN sentinel bit for bit"""
    bufs = ([('o', case.o_buf), ('lse', case.lse_buf)] if fwd else []) + ([('dqkv', case.dqkv_buf)] if bwd else [])
    for name, buf in bufs:
        g = buf[-GUARD:]
        assert torch.equal(bits(g), bits(torch.full_like(g, float('nan')))), f'{tag(case, what)}: {name} written past its end'


def snapshot(case):
    return [t.clone() for t in (case.qkv_buf, case.do_buf)]


def check_inputs(case, snap, o=None, lse=None, what=''):
    """qkv and d_o (with their guards), and the o / lse given, are bit-unchanged"""
    for name, a, b in [('qkv', case.qkv_buf, snap[0]), ('d_o', case.do_buf, snap[1])] + \
            ([('o', case.o_buf, o)] if o is not None else []) + ([('lse', case.lse_buf, lse)] if lse is not None else []):
        assert torch.equal(bits(a), bits(b)), f'{tag(case, what)}: input {name} was modified'


def onehot_window(case, w0, part):
    """write a one-hot identity block into rows [w0, w0 + dh) of V (part 2 of qkv) or of d_o (part None), zero elsewhere,
    in every head: V[j] = e_{j - w0}, so O[i, d] = Pd[i, w0 + d] / l_i, and dO[i] = e_{i - w0}, so dV[j, d] = Pd[w0 + d, j]"""
    B, N, H, dh = case.B, case.N, case.H, case.dh
    t = case.qkv if part == 2 else case.d_o
    view = t.view(B, N, -1, H, dh)[:, :, 2 if part == 2 else 0]
    view.zero_()
    n = min(dh, N - w0)
    eye = torch.eye(dh, dtype=t.dtype, device=t.device)[:n]
    view[:, w0:w0 + n] = eye.view(1, n, 1, dh)
