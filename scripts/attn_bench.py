#!/usr/bin/env python
"""Times the attention kernels alone (CUDA events, rotating over `layers` distinct buffers like the real step so that
consecutive launches do not hit in L2) at the cfg2 (B=256, N=51) and cfg4 (B=32, N=2401) shapes."""
import os
import sys
import json

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from ecg_b200 import _lib as L


def bench(B, N, H, dh=64, p=0.1, layers=12, reps=5, bwd=True):
    lib = L.load()
    inner = H * dh
    st = torch.cuda.current_stream().cuda_stream
    qkv = [torch.randn(B * N, 3 * inner, device='cuda').bfloat16() for _ in range(layers)]
    o = [torch.empty(B * N, inner, device='cuda', dtype=torch.bfloat16) for _ in range(layers)]
    d_o = [torch.randn(B * N, inner, device='cuda').bfloat16() for _ in range(layers)]
    dqkv = torch.empty_like(qkv[0])
    lse = [torch.empty(B, H, N, device='cuda') for _ in range(layers)]
    seed = torch.tensor([1234], dtype=torch.int32, device='cuda')
    n_scr = int(lib.ecgvit_attention_bwd_scratch_floats(B, N, H, dh, L.BF16))
    scr = torch.empty(max(n_scr, 1), device='cuda')
    scale = dh ** -0.5
    sp = seed.data_ptr() if p > 0 else None

    def fwd(i):
        L.check(lib.ecgvit_attention_fwd(qkv[i].data_ptr(), o[i].data_ptr(), lse[i].data_ptr(), B, N, H, dh, scale, p, 1,
                                         sp, L.BF16, st), 'attn')

    def back(i):
        L.check(lib.ecgvit_attention_bwd(qkv[i].data_ptr(), o[i].data_ptr(), d_o[i].data_ptr(), lse[i].data_ptr(),
                                         dqkv.data_ptr(), scr.data_ptr() if n_scr else None, B, N, H, dh, scale, p, 1, sp,
                                         L.BF16, st), 'attn_bwd')

    out = {}
    for name, fn in (('fwd', fwd),) + ((('bwd', back),) if bwd else ()):
        for i in range(layers):
            fn(i)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(layers):
                fn(i)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) / layers)
        flops = 4.0 * B * H * N * N * dh * (1.0 if name == 'fwd' else 2.5)
        byts = B * N * inner * 2 * (4 if name == 'fwd' else 8)
        out[name] = dict(us=round(best * 1e3, 2), tflops=round(flops / best / 1e9, 1), gbs=round(byts / best / 1e6, 1))
    return out


if __name__ == '__main__':
    res = {}
    for name, (B, N, H, layers) in {'cfg2_B256_N51': (256, 51, 12, 12), 'cfg4_B32_N2401': (32, 2401, 12, 3),
                                    'cfg4_B4_N2401': (4, 2401, 12, 6)}.items():
        for p in (0.0, 0.1):
            res[f'{name}_p{p}'] = bench(B, N, H, p=p, layers=layers)
            print(name, p, res[f'{name}_p{p}'], flush=True)
    if len(sys.argv) > 1:
        json.dump(res, open(sys.argv[1], 'w'), indent=1)
