"""Throughput of MAE-style pre-training (EcgVitForMaskedAutoencoding) against SimMIM-style pre-training
(EcgVitForMaskedPatchModeling) on ecg-vit-base, bf16, dropout 0.1, default decoder (256 wide x 4 layers, 4 heads,
mlp 1024).  Prints one JSON line.

Groups, each measured in alternating rounds in the same process (every leg sees the same clocks and neighbours):
  cfg2_B256     12 x 2500, patch 50 (n = 50), B = 256: SimMIM 0.5, MAE 0.75, MAE 0.5
  cfg2_B1024    the same at B = 1024: SimMIM 0.5, MAE 0.75 (at B = 256 MAE's encoder GEMMs have only 256 * 13 = 3328 rows)
  per_lead_B32  per-lead tokens, 12 x 5000, patch 25 (n = 2400), B = 32: SimMIM 0.5, MAE 0.75

Step times: CUDA events around `--steps` replays of the captured FusedTrainer step, device-resident inputs, after
`--warmup` steps.  FLOP per record: the forward pass's matrix products computed from the shapes (2 * rows * cols *
inner for every GEMM, 4 * N^2 * d per attention layer); a training step counts 3x that.  Per-call device times of the
MAE entry points: one eager forward + backward on a single stream (ECGVIT_WGRAD_STREAM=0), an event after every call,
median of `--reps` passes.  Usage: python scripts/bench_mae.py [--steps 20] [--warmup 5] [--rounds 3]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

DECODER = dict(decoder_hidden_size=256, decoder_num_hidden_layers=4, decoder_num_attention_heads=4,
               decoder_intermediate_size=1024)
GEOMETRY = {'cfg2': dict(max_signal_length=2500, patch_size=50),
            'per_lead': dict(max_signal_length=5000, patch_size=25, per_lead_tokens=True)}
NEW_CALLS = ('mpm_mask', 'mae_index', 'row_gather', 'embed_assemble_visible', 'mae_unshuffle', 'mae_unshuffle_bwd',
             'embed_assemble_visible_bwd')


def config(ecg_b200, geometry):
    conf = ecg_b200.EcgVitConfig.from_defined('ecg-vit-base')
    for k, v in GEOMETRY[geometry].items():
        setattr(conf, k, v)
    conf.compute_dtype = 'bf16'
    conf.hidden_dropout_prob = conf.attention_probs_dropout_prob = 0.1
    return conf


def make(ecg_b200, geometry, kind, ratio):
    torch.manual_seed(77)
    if kind == 'simmim':
        return ecg_b200.EcgVitForMaskedPatchModeling(config=config(ecg_b200, geometry), mask_ratio=ratio)
    return ecg_b200.EcgVitForMaskedAutoencoding(config=config(ecg_b200, geometry), mask_ratio=ratio, **DECODER)


def stack_flop(N, d, mlp, depth):
    return depth * (2 * N * (4 * d * d + 2 * d * mlp) + 4 * N * N * d)


def forward_flop(c, kind, ratio):
    """algorithmic forward FLOP of one record"""
    per_lead = bool(getattr(c, 'per_lead_tokens', False))
    n = c.max_signal_length // c.patch_size * (c.num_channels if per_lead else 1)
    K = c.patch_size * (1 if per_lead else c.num_channels)
    d, mlp, L = c.hidden_size, c.intermediate_size, c.num_hidden_layers
    if kind == 'simmim':
        return 2 * n * K * d + stack_flop(n + 1, d, mlp, L) + 2 * n * d * K
    nv = n - int(round(ratio * n))
    dd = DECODER['decoder_hidden_size']
    return (2 * nv * K * d + stack_flop(nv + 1, d, mlp, L) + 2 * (nv + 1) * d * dd
            + stack_flop(n + 1, dd, DECODER['decoder_intermediate_size'], DECODER['decoder_num_hidden_layers'])
            + 2 * n * dd * K)


def step_ms(tr, x, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss, _ = tr.step(x)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, float(loss)


def run_group(ecg_b200, geometry, batch, legs, a):
    from ecg_b200 import synthetic_batch
    c = config(ecg_b200, geometry)
    x, _ = synthetic_batch(batch, length=c.max_signal_length, seed=77)
    x = x.cuda()
    trainers = {}
    for name, (kind, ratio) in legs.items():
        model = make(ecg_b200, geometry, kind, ratio).cuda().train()
        trainers[name] = ecg_b200.FusedTrainer(model, use_cuda_graph=True, data_parallel=False)
        for _ in range(a.warmup):
            trainers[name].step(x)
    torch.cuda.synchronize()
    times = {k: [] for k in legs}
    losses = {}
    for _ in range(a.rounds):
        for k, tr in trainers.items():
            ms, losses[k] = step_ms(tr, x, a.steps)
            times[k].append(ms)
    out = {}
    for k, (kind, ratio) in legs.items():
        med = statistics.median(times[k])
        fwd = forward_flop(c, kind, ratio)
        out[k] = {'samples_per_s': round(batch / med * 1e3, 1), 'ms_per_step': round(med, 3),
                  'rounds_ms': [round(t, 3) for t in times[k]], 'last_loss': round(losses[k], 5),
                  'launches_per_step': trainers[k].launches_per_step,
                  'forward_gflop_per_record': round(fwd / 1e9, 3),
                  'train_tflop_per_s': round(3 * fwd * batch / (med * 1e-3) / 1e12, 1)}
    del trainers
    torch.cuda.empty_cache()
    return out


def per_call_times(ecg_b200, geometry, batch, reps):
    """{name: median ms} of the MAE step's new calls"""
    from ecg_b200 import _lib, synthetic_batch
    model = make(ecg_b200, geometry, 'mae', 0.75).cuda().train()
    x, _ = synthetic_batch(batch, length=model.config.max_signal_length, seed=77)
    x = x.cuda()
    model._prepare(x.device)
    eng = model._engine
    assert eng.side_stream is None
    samples = {}
    for r in range(reps + 1):
        model._flat_g.zero_()
        eng.new_dropout_seed()
        torch.cuda.synchronize()
        _lib.profile[0] = []
        start = torch.cuda.Event(enable_timing=True)
        start.record()
        eng.forward(x)
        eng.backward()
        torch.cuda.synchronize()
        recs, _lib.profile[0] = _lib.profile[0], None
        prev = start
        for name, _, ev in recs:
            ms = prev.elapsed_time(ev)
            prev = ev
            if r > 0 and name in NEW_CALLS:
                samples.setdefault(name, []).append(ms)
    return {k: round(statistics.median(v), 4) for k, v in samples.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--calls-only', nargs=2, metavar=('GEOMETRY', 'BATCH'), help=argparse.SUPPRESS)
    a = ap.parse_args()
    import ecg_b200
    if a.calls_only:
        print(json.dumps(per_call_times(ecg_b200, a.calls_only[0], int(a.calls_only[1]), a.reps)))
        return
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip()
    row = {'gpu': q, 'model': 'ecg-vit-base bf16 dropout 0.1', 'decoder': DECODER}
    row['cfg2_B256'] = run_group(ecg_b200, 'cfg2', 256, {'simmim_0.5': ('simmim', 0.5), 'mae_0.75': ('mae', 0.75),
                                                          'mae_0.5': ('mae', 0.5)}, a)
    row['cfg2_B1024'] = run_group(ecg_b200, 'cfg2', 1024, {'simmim_0.5': ('simmim', 0.5), 'mae_0.75': ('mae', 0.75)}, a)
    row['per_lead_B32'] = run_group(ecg_b200, 'per_lead', 32, {'simmim_0.5': ('simmim', 0.5),
                                                               'mae_0.75': ('mae', 0.75)}, a)
    env = dict(os.environ, ECGVIT_WGRAD_STREAM='0')
    row['new_call_ms'] = {}
    for geometry, batch in (('cfg2', 256), ('per_lead', 32)):
        out = subprocess.run([sys.executable, __file__, '--calls-only', geometry, str(batch), '--reps', str(a.reps)],
                             env=env, capture_output=True, text=True, check=True)
        row['new_call_ms'][f'{geometry}_B{batch}_mae_0.75'] = json.loads(out.stdout.strip().splitlines()[-1])
    print(json.dumps(row))


if __name__ == '__main__':
    main()
