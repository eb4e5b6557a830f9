"""Cost of the fine-tuning options on ecg-vit-base, bf16, dropout 0.1.  Prints one JSON line (and writes it to --out).

Two comparisons, each measured in alternating rounds in the same process (both arms see the same clocks and neighbours);
the card name and power limit are read in the same run:
  adamw_kernel  ecgvit_adamw_step_grouped (the map of `param_groups_lrd`, 2 * (depth + 2) groups) against
                ecgvit_adamw_step, bf16 shadow on, over the flat buffers of the cfg2 model (base) and the cfg5 model
                (large).  Every buffer is larger than the 126 MB L2.  CUDA events around `--launches` back-to-back
                launches, median of `--rounds`.
  cfg2_step     the captured FusedTrainer step at cfg2 (12 x 2500, patch 50, B = 256): the default (pool='cls', one
                group) against pool='mean' with `param_groups_lrd` groups.  CUDA events around `--steps` replays,
                device-resident inputs, after `--warmup` steps; samples/s and the kernels each replay launches.
Usage: python scripts/bench_finetune.py [--steps 20] [--warmup 5] [--rounds 5] [--out FILE]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def config(ecg_b200, size, pool='cls'):
    conf = ecg_b200.EcgVitConfig.from_defined(f'ecg-vit-{size}')
    conf.max_signal_length, conf.patch_size = 2500, 50
    conf.compute_dtype = 'bf16'
    conf.hidden_dropout_prob = conf.attention_probs_dropout_prob = 0.1
    conf.pool = pool
    return conf


def adamw_kernel(ecg_b200, size, a):
    from ecg_b200 import _lib
    from ecg_b200.optim import group_map, group_names, group_table
    lib = _lib.load()
    model = ecg_b200.EcgVit(config=config(ecg_b200, size))
    groups = ecg_b200.param_groups_lrd(model)
    gmap = group_map(model, group_names(model, groups)).cuda()
    n = gmap.numel() * 64
    dev = 'cuda'
    p, m, v, g = (torch.randn(n, device=dev) * 0.02, torch.zeros(n, device=dev), torch.zeros(n, device=dev),
                  torch.randn(n, device=dev) * 1e-3)
    shadow = p.bfloat16()
    stats = torch.zeros(_lib.STATS_FLOATS, device=dev)
    vals = _lib.adamw_hyper(1e-4, 0.9, 0.999, 1e-8, 0.05, 10, 0.0, 1.0)
    hyper = torch.tensor(vals + group_table([1e-4 * grp['lr_scale'] for grp in groups],
                                            [grp['weight_decay'] for grp in groups], 0.9, 10), device=dev)
    st = torch.cuda.current_stream().cuda_stream

    def plain():
        _lib.check(lib.ecgvit_adamw_step(p.data_ptr(), m.data_ptr(), v.data_ptr(), g.data_ptr(), _lib.F32,
                                         shadow.data_ptr(), n, hyper.data_ptr(), stats.data_ptr(), 0, st))

    def grouped():
        _lib.check(lib.ecgvit_adamw_step_grouped(p.data_ptr(), m.data_ptr(), v.data_ptr(), g.data_ptr(), _lib.F32,
                                                 shadow.data_ptr(), n, gmap.data_ptr(), hyper.data_ptr() + 64,
                                                 hyper.data_ptr(), stats.data_ptr(), 0, st))

    arms = {'plain': plain, 'grouped': grouped}
    for f in arms.values():
        for _ in range(a.warmup):
            f()
    times = {k: [] for k in arms}
    for _ in range(a.rounds):
        for k, f in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.launches):
                f()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / a.launches)
    # algorithmic bytes: p, m, v read + write, fp32 g read, bf16 shadow write; the group map adds n / 64 bytes
    base_bytes = n * (4 * 6 + 4 + 2)
    out = {'flat_elements': n, 'groups': len(groups), 'group_map_bytes': gmap.numel(),
           'group_map_share_of_traffic': round(gmap.numel() / base_bytes, 6)}
    for k in arms:
        med = statistics.median(times[k])
        byts = base_bytes + (gmap.numel() if k == 'grouped' else 0)
        out[k] = {'us_per_call': round(med * 1e3, 2), 'rounds_us': [round(t * 1e3, 2) for t in times[k]],
                  'tb_per_s': round(byts / (med * 1e-3) / 1e12, 2)}
    out['grouped_over_plain'] = round(statistics.median(times['grouped']) / statistics.median(times['plain']), 4)
    del p, m, v, g, shadow
    torch.cuda.empty_cache()
    return out


def step_ms(tr, x, y, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss, _ = tr.step(x, y)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, float(loss)


def cfg2_step(ecg_b200, a, batch=256):
    from ecg_b200 import synthetic_batch
    x, y = synthetic_batch(batch, length=2500, seed=77)
    x, y = x.cuda(), y.cuda()
    trainers = {}
    for name, pool, lrd in (('default', 'cls', False), ('mean_pool_lrd', 'mean', True)):
        torch.manual_seed(77)
        model = ecg_b200.EcgVit(config=config(ecg_b200, 'base', pool)).cuda().train()
        groups = ecg_b200.param_groups_lrd(model) if lrd else None
        trainers[name] = ecg_b200.FusedTrainer(model, use_cuda_graph=True, data_parallel=False, param_groups=groups)
        for _ in range(a.warmup):
            trainers[name].step(x, y)
    torch.cuda.synchronize()
    times, losses = {k: [] for k in trainers}, {}
    for _ in range(a.rounds):
        for k, tr in trainers.items():
            ms, losses[k] = step_ms(tr, x, y, a.steps)
            times[k].append(ms)
    out = {}
    for k, tr in trainers.items():
        med = statistics.median(times[k])
        out[k] = {'samples_per_s': round(batch / med * 1e3, 1), 'ms_per_step': round(med, 3),
                  'rounds_ms': [round(t, 3) for t in times[k]], 'last_loss': round(losses[k], 5),
                  'launches_per_step': tr.launches_per_step}
    out['mean_pool_lrd_over_default'] = round(statistics.median(times['mean_pool_lrd'])
                                              / statistics.median(times['default']), 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--launches', type=int, default=50)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    import ecg_b200
    assert torch.cuda.is_available(), 'bench_finetune.py measures on the GPU'
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip()
    row = {'gpu': q, 'model': 'ecg-vit bf16 dropout 0.1, 12 x 2500, patch 50'}
    row['adamw_kernel'] = {'cfg2_base': adamw_kernel(ecg_b200, 'base', a),
                           'cfg5_large': adamw_kernel(ecg_b200, 'large', a)}
    row['cfg2_step'] = cfg2_step(ecg_b200, a)
    line = json.dumps(row)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
