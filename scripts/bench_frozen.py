"""Linear probing and partial fine-tuning against full fine-tuning: the captured FusedTrainer step at cfg2 (ecg-vit-base,
12 x 2500, patch 50, B = 256, bf16, dropout 0.1) with three sets of `requires_grad` flags:
  full     every parameter trains
  partial  the last 4 encoder blocks and the head train (MAE's partial fine-tuning)
  probe    only the head trains (linear probing)
The arms are measured in alternating rounds in the same process (same clocks and neighbours): CUDA events around
`--steps` replays, device-resident inputs, after `--warmup` steps; median ms per step, samples/s and the kernels each
replay launches.  Peak memory per arm is `torch.cuda.max_memory_allocated` over building the arm and its warm-up steps
(the statistic is reset before each arm), minus what was allocated before.  The card name and power limit are read in
the same run.  Prints one JSON line (and writes it to --out).
Usage: python scripts/bench_frozen.py [--steps 20] [--warmup 5] [--rounds 5] [--out FILE]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

ARMS = {'full': None, 'partial': 4, 'probe': 0}   # arm -> number of trainable top blocks (None: everything trains)


def freeze(model, k):
    depth = model.config.num_hidden_layers
    for name, p in model.named_parameters():
        if k is None or name.startswith('vit.mlp_head.'):
            continue
        parts = name.split('.')
        top_block = name.startswith('vit.transformer.layers.') and int(parts[3]) >= depth - k
        p.requires_grad_(top_block)
    return model


def step_ms(tr, x, y, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss, _ = tr.step(x, y)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, float(loss)


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
    assert torch.cuda.is_available(), 'bench_frozen.py measures on the GPU'
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip()
    x, y = synthetic_batch(a.batch, length=2500, seed=77)
    x, y = x.cuda(), y.cuda()
    trainers, peak = {}, {}
    for name, k in ARMS.items():
        conf = ecg_b200.EcgVitConfig.from_defined('ecg-vit-base')
        conf.max_signal_length, conf.patch_size = 2500, 50
        conf.compute_dtype = 'bf16'
        conf.hidden_dropout_prob = conf.attention_probs_dropout_prob = 0.1
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        before = torch.cuda.memory_allocated()
        torch.manual_seed(77)
        model = freeze(ecg_b200.EcgVit(config=conf), k).cuda().train()
        trainers[name] = ecg_b200.FusedTrainer(model, use_cuda_graph=True, data_parallel=False)
        for _ in range(a.warmup):
            trainers[name].step(x, y)
        torch.cuda.synchronize()
        peak[name] = torch.cuda.max_memory_allocated() - before
    times, losses = {k: [] for k in trainers}, {}
    for _ in range(a.rounds):
        for k, tr in trainers.items():
            ms, losses[k] = step_ms(tr, x, y, a.steps)
            times[k].append(ms)
    out = {'gpu': q, 'model': f'ecg-vit-base bf16 dropout 0.1, 12 x 2500, patch 50, B = {a.batch}, captured step'}
    for k, tr in trainers.items():
        med = statistics.median(times[k])
        out[k] = {'samples_per_s': round(a.batch / med * 1e3, 1), 'ms_per_step': round(med, 3),
                  'rounds_ms': [round(t, 3) for t in times[k]], 'last_loss': round(losses[k], 5),
                  'launches_per_step': tr.launches_per_step, 'peak_memory_gb': round(peak[k] / 1e9, 3),
                  'trainable_parameters': sum(p.numel() for p in tr.model.parameters() if p.requires_grad)}
    for k in ('partial', 'probe'):
        out[f'{k}_speedup_over_full'] = round(statistics.median(times['full']) / statistics.median(times[k]), 3)
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
