"""Cost of stochastic depth (`drop_path_rate`) on the captured cfg2 training step (ecg-vit-base, 12 x 2500, patch 50,
B = 256, bf16).  Prints one JSON line (and writes it to --out).

Two comparisons, at dropout 0.1 and at dropout 0: drop_path_rate 0 against 0.1.  The four trainers are built first; each
comparison then alternates its two arms over `--rounds` rounds in the same process (both arms see the same clocks and
neighbours).  CUDA events around `--steps` graph replays, device-resident inputs, after `--warmup` steps; samples/s and
the kernels each replay launches.  The card name and power limit are read in the same run.
Usage: python scripts/bench_drop_path.py [--steps 20] [--warmup 5] [--rounds 5] [--out FILE]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def config(ecg_b200, dropout, rate):
    conf = ecg_b200.EcgVitConfig.from_defined('ecg-vit-base')
    conf.max_signal_length, conf.patch_size = 2500, 50
    conf.compute_dtype = 'bf16'
    conf.hidden_dropout_prob = conf.attention_probs_dropout_prob = dropout
    conf.drop_path_rate = rate
    return conf


def step_ms(tr, x, y, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss, _ = tr.step(x, y)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, float(loss)


def compare(ecg_b200, a, dropout, x, y):
    batch = x.shape[0]
    trainers = {}
    for rate in (0.0, 0.1):
        torch.manual_seed(77)
        model = ecg_b200.EcgVit(config=config(ecg_b200, dropout, rate)).cuda().train()
        trainers[f'drop_path_{rate}'] = ecg_b200.FusedTrainer(model, use_cuda_graph=True, data_parallel=False)
    for tr in trainers.values():
        for _ in range(a.warmup):
            tr.step(x, y)
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
    out['on_over_off'] = round(statistics.median(times['drop_path_0.1']) / statistics.median(times['drop_path_0.0']), 4)
    del trainers
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--batch', type=int, default=256)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    import ecg_b200
    from ecg_b200 import synthetic_batch
    assert torch.cuda.is_available(), 'bench_drop_path.py measures on the GPU'
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip()
    row = {'gpu': q, 'model': f'ecg-vit-base bf16, 12 x 2500, patch 50, B = {a.batch}, captured FusedTrainer step'}
    x, y = synthetic_batch(a.batch, length=2500, seed=77)
    x, y = x.cuda(), y.cuda()
    # the masked copies that drop path adds at dropout 0: two [M, d] bf16 writes per block (M = B * 51 tokens)
    c = config(ecg_b200, 0.0, 0.1)
    row['dxm_bytes_per_step_at_dropout0'] = 2 * a.batch * 51 * c.hidden_size * 2 * c.num_hidden_layers
    row['dropout_0.1'] = compare(ecg_b200, a, 0.1, x, y)
    row['dropout_0.0'] = compare(ecg_b200, a, 0.0, x, y)
    line = json.dumps(row)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
