"""
ctypes binding of `libecgvit_b200.so` (C ABI declared in include/ecgvit_b200.h).

There is no fallback: if the library is missing the import of any compute entry point raises, and every
non-zero return code raises RuntimeError with the library's own message.
"""
import ctypes
import os
from ctypes import c_int, c_int64, c_float, c_void_p, c_char_p, POINTER, Structure

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, 'libecgvit_b200.so')

F32, BF16, BF16_RES32 = 0, 1, 2  # BF16_RES32: bf16 mode whose residual-stream operand is fp32 (ecgvit_b200.h)
STATS_FLOATS = 2052  # ECGVIT_STATS_FLOATS
SUMSQ_MAX_BLOCKS = 2048  # partial slots of the gradient-norm scratch (stats[4:])
EPI_STORE, EPI_BIAS_RES, EPI_BIAS_GELU, EPI_DGELU, EPI_ATOMIC_F32, EPI_BIAS_RES_F32, EPI_BIAS_SUB_ROWSQ = 0, 1, 2, 3, 4, 5, 6
REDUCTION = {'mean': 0, 'sum': 1, 'none': 2}


class GemmArgs(Structure):
    """mirror of `ecgvit_gemm_args`"""
    _fields_ = [
        ('M', c_int), ('N', c_int), ('K', c_int),
        ('A', c_void_p), ('lda', c_int64), ('a_kmajor', c_int),
        ('B', c_void_p), ('ldb', c_int64), ('b_kmajor', c_int),
        ('epilogue', c_int),
        ('out', c_void_p), ('ldo', c_int64),
        ('out2', c_void_p), ('aux', c_void_p), ('bias', c_void_p),
        ('dtype', c_int), ('split_k', c_int),
        ('dropout_stream', c_int), ('dropout_p', c_float), ('dropout_seed', c_void_p),
    ]


# name -> argtypes; restype is int unless listed in _RESTYPES
SIGNATURES = {
    'ecgvit_abi_version': [],
    'ecgvit_last_error': [],
    'ecgvit_device_ok': [],
    'ecgvit_patchify': [c_void_p, c_void_p, c_int, c_int, c_int64, c_int, c_int, c_int, c_void_p],
    'ecgvit_patchify_leads': [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_int, c_int, c_int,
                              c_int, c_int, c_void_p],
    'ecgvit_pad_cols': [c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_void_p],
    'ecgvit_unpad_add_f32': [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p],
    'ecgvit_patchify_transform': [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_int, c_int,
                                  c_int, c_int, c_void_p],
    'ecgvit_embed_assemble': [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_int, c_void_p,
                              c_int, c_void_p],
    'ecgvit_embed_assemble_bwd': [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_int,
                                  c_void_p, c_int, c_void_p],
    'ecgvit_mpm_mask': [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
    'ecgvit_embed_assemble_masked': [c_void_p] * 6 + [c_int, c_int, c_int, c_float, c_int, c_void_p, c_int, c_void_p],
    'ecgvit_embed_assemble_masked_bwd': [c_void_p] * 7 + [c_int, c_int, c_int, c_float, c_int, c_void_p, c_int,
                                                          c_void_p],
    'ecgvit_layernorm_patch_fwd': [c_void_p] * 6 + [c_int, c_int, c_int, c_float, c_int, c_void_p],
    'ecgvit_layernorm_patch_bwd': [c_void_p] * 10 + [c_int, c_int, c_int, c_int, c_void_p],
    'ecgvit_mpm_loss': [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
    'ecgvit_mpm_dpred': [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_int,
                         c_void_p],
    'ecgvit_mpm_reconstruction': [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    'ecgvit_mae_index': [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
    'ecgvit_row_gather': [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p],
    'ecgvit_embed_assemble_visible': [c_void_p] * 5 + [c_int, c_int, c_int, c_float, c_int, c_void_p, c_int, c_void_p],
    'ecgvit_embed_assemble_visible_bwd': [c_void_p] * 7 + [c_int, c_int, c_int, c_int, c_float, c_int, c_void_p, c_int,
                                                           c_void_p],
    'ecgvit_mae_unshuffle': [c_void_p] * 5 + [c_int, c_int, c_int, c_int, c_int, c_void_p],
    'ecgvit_mae_unshuffle_bwd': [c_void_p] * 6 + [c_int, c_int, c_int, c_int, c_int, c_void_p],
    'ecgvit_dropout_bwd_copy': [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_float, c_int, c_void_p, c_int,
                                c_void_p],
    'ecgvit_layernorm_fwd': [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float,
                             c_int, c_void_p],
    'ecgvit_layernorm_bwd_scratch_floats': [c_int],
    'ecgvit_layernorm_bwd': [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                             c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_int, c_void_p, c_int, c_int, c_int, c_int,
                             c_void_p],
    'ecgvit_layernorm_bwd_finalize': [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p],
    'ecgvit_gemm': [POINTER(GemmArgs), c_void_p],
    # drop path: the plain arguments (without the stream), then path_p, path_stream, rows_per_record, stream
    'ecgvit_gemm_drop_path': [POINTER(GemmArgs), c_float, c_int, c_int, c_void_p],
    'ecgvit_layernorm_bwd_drop_path': [c_void_p] * 12 + [c_float, c_int, c_void_p, c_int, c_int, c_int, c_int, c_float,
                                                         c_int, c_int, c_void_p],
    'ecgvit_dropout_bwd_copy_drop_path': [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_float, c_int, c_void_p,
                                          c_int, c_float, c_int, c_int, c_void_p],
    'ecgvit_attention_probs': [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_int64, c_int, c_void_p],
    'ecgvit_eval_metrics_scratch_bytes': [c_int],
    'ecgvit_eval_metrics': [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p],
    'ecgvit_attention_fwd': [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_float, c_int,
                             c_void_p, c_int, c_void_p],
    'ecgvit_attention_bwd_scratch_floats': [c_int, c_int, c_int, c_int, c_int],
    'ecgvit_attention_bwd': [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                             c_float, c_float, c_int, c_void_p, c_int, c_void_p],
    'ecgvit_head_fwd': [c_void_p] * 7 + [c_int] + [c_void_p] * 5 + [c_int, c_int, c_int, c_int, c_int, c_float, c_int,
                                                                     c_void_p],
    'ecgvit_head_bwd': [c_void_p] * 5 + [c_int] + [c_void_p] * 11 + [c_int, c_int, c_int, c_int, c_int, c_float, c_void_p,
                                                                      c_int, c_void_p],
    'ecgvit_token_mean': [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    'ecgvit_token_mean_bwd': [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    'ecgvit_colsum': [c_void_p, c_void_p, c_int, c_int, c_int64, c_int, c_void_p],
    'ecgvit_grad_sumsq': [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p],
    'ecgvit_grad_sumsq_partial': [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_int, c_int, c_void_p],
    'ecgvit_grad_sumsq_finalize': [c_void_p, c_int, c_void_p],
    'ecgvit_adamw_step': [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int64, c_void_p, c_void_p, c_int,
                          c_void_p],
    'ecgvit_adamw_step_grouped': [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int64, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_int, c_void_p],
    'ecgvit_grad_scale_by_clip': [c_void_p, c_int64, c_void_p, c_void_p, c_void_p],
    'ecgvit_cast_f32_to_bf16': [c_void_p, c_void_p, c_int64, c_void_p],
}
_RESTYPES = {'ecgvit_last_error': c_char_p, 'ecgvit_layernorm_bwd_scratch_floats': c_int64,
             'ecgvit_eval_metrics_scratch_bytes': c_int64, 'ecgvit_attention_bwd_scratch_floats': c_int64}

_lib = None


def load():
    """Load the shared library (once); raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f'{LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                f'(there is no CPU / PyTorch fallback for the ECG-ViT kernels)')
        lib = ctypes.CDLL(LIB_PATH)
        for name, argtypes in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the symbol is not exported
            fn.argtypes = argtypes
            fn.restype = _RESTYPES.get(name, c_int)
        _lib = lib
    return _lib


def last_error():
    msg = load().ecgvit_last_error()
    return msg.decode() if msg else ''


# kernels launched per successful entry-point call (memsets are not kernels); feeds bench.py's `gpu_launches`
KERNELS_PER_CALL = {'layernorm_patch_bwd': 3, 'attention_bwd_flash': 3, 'head_fwd': 2, 'head_bwd': 3, 'layernorm_bwd': 2, 'layernorm_bwd_partial': 1, 'grad_sumsq': 2, 'eval_metrics': 3,
                    'embed_assemble_visible_bwd': 3, 'mae_unshuffle_bwd': 3}
launch_counter = [0]


def check(rc, what=''):
    if rc != 0:
        raise RuntimeError(f'ecgvit_b200 {what} failed (code {rc}): {last_error()}')
    launch_counter[0] += KERNELS_PER_CALL.get(what, 1)
    if profile[0] is not None:
        # one event after every call: on a single stream, consecutive event deltas are per-call device times
        import torch
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        profile[0].append((what, profile_meta[0], e))
        profile_meta[0] = None


profile = [None]       # set to a list to record (name, meta, event) per entry-point call (bench.py roofline leg)
profile_meta = [None]  # optional description of the next call (GEMM shape / epilogue)


def ptr(t):
    """device pointer of a torch tensor (or None)"""
    return None if t is None else t.data_ptr()


def counter_hash(seed, stream, pair):
    """host replica of csrc/common.cuh `dropout_hash` (two multiply-and-fold rounds) over the int64 tensor `pair`"""
    m32 = 0xFFFFFFFF
    key = (seed ^ ((stream * 0x85EBCA77 + 0xC2B2AE3D) & m32)) & m32

    def mulfold(a, k):  # (a * k) as a 64-bit product, xor of its two 32-bit halves
        a_lo, a_hi = a & 0xFFFF, a >> 16  # split so the int64 products cannot overflow
        p0 = a_lo * k
        p1 = a_hi * k
        total_lo = (p0 + ((p1 & 0xFFFF) << 16))
        lo = total_lo & m32
        hi = ((p1 >> 16) + (total_lo >> 32)) & m32
        return lo ^ hi

    h = mulfold((pair ^ key) & m32, 0x9E3779B1)
    return mulfold(h, 0x7FEB352D)


def dropout_keep_mask(seed, stream, p, index):
    """host replica of the kernels' counter-based dropout (csrc/common.cuh `dropout_hash`, two multiply-and-fold rounds): multiplier (0 or
    1/(1-p_q)) for every element index in the int64 tensor `index`; used by the tests to inject the SAME masks into the
    CPU oracle"""
    import torch
    thr = min(int(p * 65536.0 + 0.5), 65535)
    if thr == 0:
        return torch.ones(index.shape, dtype=torch.float32)
    idx = index.to(torch.int64)
    h = counter_hash(seed, stream, idx >> 1)
    bits = torch.where((idx & 1) == 1, h >> 16, h & 0xFFFF)
    scale = 1.0 / (1.0 - thr / 65536.0)
    return torch.where(bits >= thr, torch.tensor(scale, dtype=torch.float32), torch.tensor(0.0, dtype=torch.float32))


def mpm_mask(seed, B, n, k, site):
    """host replica of ecgvit_mpm_mask: bool [B, n], patch w of record b masked iff the rank of its key
    counter_hash(seed, site, b*n + w) within record b is < k (ties broken by the lower index)"""
    import torch
    keys = counter_hash(seed, site, torch.arange(B * n, dtype=torch.int64)).reshape(B, n)
    # stable sort on (key, index): the k first positions of every row are its masked patches
    order = torch.sort(keys, dim=1, stable=True).indices
    mask = torch.zeros(B, n, dtype=torch.bool)
    mask.scatter_(1, order[:, :k], True)
    return mask


ADAMW_SLICE, ADAMW_FIRST_SLICE = 1, 2


def adamw_hyper(lr, beta1, beta2, eps, weight_decay, step, max_norm, grad_scale, skip=False):
    """the 16-float `hyper` block of ecgvit_grad_sumsq / ecgvit_adamw_step (include/ecgvit_b200.h); derived scalars
    are evaluated in double precision here, exactly where torch.optim.AdamW evaluates them"""
    bc1, bc2 = 1.0 - beta1 ** step, 1.0 - beta2 ** step
    vals = [lr, beta1, beta2, eps, weight_decay, bc1, bc2, max_norm, grad_scale,
            1.0 - beta1, 1.0 - beta2, 1.0 - lr * weight_decay, lr / bc1, bc2 ** 0.5, 1.0 if skip else 0.0]
    return vals + [0.0] * (16 - len(vals))


class PinnedRing:
    """Asynchronous upload of a few host scalars per step.  `dst.copy_(torch.tensor(values))` from pageable memory makes
    the host wait for everything queued on the stream (i.e. the previous step), which exposes the whole host-side
    launch cost between two graph replays; a ring of pinned staging slots lets the copy be truly asynchronous, and a
    slot is rewritten only after the copy that read it has completed (its event), so the host can run several steps
    ahead of the device."""

    def __init__(self, numel, dtype, slots=8):
        import torch
        self.bufs = [torch.empty(numel, dtype=dtype).pin_memory() for _ in range(slots)]
        self.events = [None] * slots
        self.i = 0

    def upload(self, dst, values):
        import torch
        i = self.i
        self.i = (i + 1) % len(self.bufs)
        if self.events[i] is not None:
            self.events[i].synchronize()  # normally long complete
        buf = self.bufs[i]
        buf.copy_(torch.tensor(values, dtype=buf.dtype))
        dst.copy_(buf, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self.events[i] = ev
