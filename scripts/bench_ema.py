"""The weight moving average (ema_decay) against training without it.
  step     the captured FusedTrainer step at cfg2 (ecg-vit-base, 12 x 2500, patch 50, B = 256, bf16, dropout 0.1) with
           EMA off and with ema_decay=0.9999, ema_warmup=True, measured in alternating rounds in the same process
           (CUDA events around `--steps` replays, device-resident inputs, after `--warmup` steps; median ms per step)
  kernel   the AdamW update alone over the flat buffers of cfg2 (ecg-vit-base) and cfg5 (ecg-vit-large), bf16 shadow, fp32
           gradients: `ecgvit_adamw_step` (no EMA), `ecgvit_adamw_step_ema` (fused EMA), and `ecgvit_adamw_step`
           followed by `torch.lerp_` over the flat buffer (the separate pass a user-side EMA costs); CUDA events around
           `--iters` launches of each arm, arms alternated over `--rounds`; every buffer is larger than the 126 MB L2
Launches per step are our kernels replayed by one graph launch; peak memory per arm is `torch.cuda.max_memory_allocated`
over building the arm and its warm-up (reset before each arm) minus what was allocated before.  The card name and power
limit are read in the same run.  Prints one JSON line (and writes it to --out).
Usage: python scripts/bench_ema.py [--steps 20] [--warmup 5] [--rounds 5] [--iters 50] [--out FILE]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

DECAY = 0.9999


def cfg(size):
    import ecg_b200
    conf = ecg_b200.EcgVitConfig.from_defined(f'ecg-vit-{size}')
    conf.max_signal_length, conf.patch_size = 2500, 50
    conf.compute_dtype = 'bf16'
    conf.hidden_dropout_prob = conf.attention_probs_dropout_prob = 0.1
    return conf


def events_ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def bench_steps(a, x, y):
    import ecg_b200
    trainers, peak = {}, {}
    for name, ema in (('ema_off', None), ('ema_on', DECAY)):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        before = torch.cuda.memory_allocated()
        torch.manual_seed(77)
        model = ecg_b200.EcgVit(config=cfg('base')).cuda().train()
        trainers[name] = ecg_b200.FusedTrainer(model, use_cuda_graph=True, data_parallel=False, ema_decay=ema,
                                               ema_warmup=ema is not None)
        for _ in range(a.warmup):
            trainers[name].step(x, y)
        torch.cuda.synchronize()
        peak[name] = torch.cuda.max_memory_allocated() - before
    times = {k: [] for k in trainers}
    for _ in range(a.rounds):
        for k, tr in trainers.items():
            times[k].append(events_ms(lambda: tr.step(x, y), a.steps))
    out = {}
    for k, tr in trainers.items():
        tr.check_finite()
        med = statistics.median(times[k])
        out[k] = {'ms_per_step': round(med, 3), 'samples_per_s': round(a.batch / med * 1e3, 1),
                  'rounds_ms': [round(t, 3) for t in times[k]], 'launches_per_step': tr.launches_per_step,
                  'peak_memory_gb': round(peak[k] / 1e9, 3)}
    out['ema_on_over_off'] = round(statistics.median(times['ema_on']) / statistics.median(times['ema_off']), 4)
    del trainers
    torch.cuda.empty_cache()
    return out


def bench_kernel(a, size):
    import ecg_b200
    from ecg_b200 import _lib
    lib = _lib.load()
    _, n = ecg_b200.EcgVit(config=cfg(size))._flat_layout()
    dev = 'cuda'
    gen = torch.Generator(device=dev).manual_seed(0)
    p = torch.randn(n, device=dev, generator=gen)
    m, v = torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    g = torch.randn(n, device=dev, generator=gen) * 1e-3
    ema = p.clone()
    shadow = p.bfloat16()
    hyper = torch.tensor(_lib.adamw_hyper(1e-4, 0.9, 0.999, 1e-8, 0.05, 10, 0.0, 1.0, ema_rate=1.0 - DECAY),
                         dtype=torch.float32, device=dev)
    stats = torch.zeros(_lib.STATS_FLOATS, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    args = (p.data_ptr(), m.data_ptr(), v.data_ptr(), g.data_ptr(), _lib.F32, shadow.data_ptr())
    tail = (hyper.data_ptr(), stats.data_ptr(), 0, st)

    def plain():
        _lib.check(lib.ecgvit_adamw_step(*args, n, *tail), 'adamw_step')

    def fused():
        _lib.check(lib.ecgvit_adamw_step_ema(*args, ema.data_ptr(), n, None, None, *tail), 'adamw_step_ema')

    def separate():
        plain()
        ema.lerp_(p, 1.0 - DECAY)

    arms = {'adamw': plain, 'adamw_fused_ema': fused, 'adamw_then_lerp': separate}
    for fn in arms.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(a.rounds):
        for k, fn in arms.items():
            times[k].append(events_ms(fn, a.iters) * 1e3)
    out = {'flat_elements': n}
    bytes_per = {'adamw': 30, 'adamw_fused_ema': 38, 'adamw_then_lerp': 42}   # the lerp reads ema and p, writes ema
    for k in arms:
        us = statistics.median(times[k])
        out[k] = {'us': round(us, 1), 'rounds_us': [round(t, 1) for t in times[k]],
                  'tb_per_s': round(bytes_per[k] * n / us / 1e6, 2), 'launches': 2 if k == 'adamw_then_lerp' else 1}
    out['fused_ema_extra_us'] = round(out['adamw_fused_ema']['us'] - out['adamw']['us'], 1)
    out['separate_lerp_extra_us'] = round(out['adamw_then_lerp']['us'] - out['adamw']['us'], 1)
    out['ema_buffer_gb'] = round(4 * n / 1e9, 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--iters', type=int, default=50)
    ap.add_argument('--batch', type=int, default=256)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    from ecg_b200 import synthetic_batch
    assert torch.cuda.is_available(), 'bench_ema.py measures on the GPU'
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip()
    x, y = synthetic_batch(a.batch, length=2500, seed=77)
    out = {'gpu': q, 'model': f'ecg-vit-base bf16 dropout 0.1, 12 x 2500, patch 50, B = {a.batch}, captured step',
           'ema': f'ema_decay={DECAY}, ema_warmup=True'}
    out['step'] = bench_steps(a, x.cuda(), y.cuda())
    out['kernel_cfg2'] = bench_kernel(a, 'base')
    out['kernel_cfg5'] = bench_kernel(a, 'large')
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
