"""Cost of masked-patch pre-training next to classification at cfg2 (ecg-vit-base, bf16, 12 x 2500 records, patch 50,
B = 256, dropout 0.1, mask ratio 0.5): samples/s of the captured FusedTrainer step of EcgVitForMaskedPatchModeling and
of EcgVit, measured in the same process in alternating rounds, plus per-call device times of the entry points the
pre-training step adds.  Prints one JSON line.

Step times: CUDA events around `--steps` graph replays, device-resident inputs, after `--warmup` steps.
Per-call times: one eager forward + backward on a single stream (ECGVIT_WGRAD_STREAM=0) with an event after every
entry-point call; the delta to the previous event is the call's device time when the device is the bottleneck (median
of `--reps` passes).  Usage: python scripts/bench_pretrain.py [--steps 30] [--warmup 5] [--rounds 3] [--batch 256]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def config(ecg_b200):
    conf = ecg_b200.EcgVitConfig.from_defined('ecg-vit-base')
    conf.max_signal_length, conf.patch_size, conf.compute_dtype = 2500, 50, 'bf16'
    conf.hidden_dropout_prob = conf.attention_probs_dropout_prob = 0.1
    return conf


def step_ms(tr, x, y, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss, _ = tr.step(x, y)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, float(loss)


NEW_CALLS = ('mpm_mask', 'embed_assemble_masked', 'layernorm_patch_fwd', 'mpm_loss', 'mpm_dpred', 'layernorm_patch_bwd',
             'embed_assemble_masked_bwd')


def per_call_times(ecg_b200, x, reps):
    """{name: median ms} of the pre-training step's new calls (recon GEMMs named by their epilogue / shape)"""
    from ecg_b200 import _lib
    torch.manual_seed(77)
    model = ecg_b200.EcgVitForMaskedPatchModeling(config=config(ecg_b200)).cuda().train()
    model._prepare(x.device)
    eng = model._engine
    assert eng.side_stream is None
    d = model.config.hidden_size
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
        if r == 0:
            continue   # warm-up pass
        prev = start
        for name, meta, ev in recs:
            ms = prev.elapsed_time(ev)
            prev = ev
            if name == 'gemm' and meta is not None:
                M, N, K, epi = meta[:4]
                if epi == _lib.EPI_BIAS_SUB_ROWSQ:
                    name = f'gemm_recon_fwd_rowsq[{M}x{N}x{K}]'
                elif (M, N) == (eng._cur.Kp, d):
                    name = f'gemm_recon_wgrad[{M}x{N}x{K}]'
                elif N == d and K == eng._cur.Kp:
                    name = f'gemm_recon_dgrad[{M}x{N}x{K}]'
                else:
                    continue
            elif name not in NEW_CALLS:
                continue
            samples.setdefault(name, []).append(ms)
    return {k: round(statistics.median(v), 4) for k, v in samples.items()}


def mask_draw_ms(ecg_b200, n, batch, reps=20):
    """device time of one ecgvit_mpm_mask launch (CUDA events around `reps` launches): n patches per record, k = n / 2"""
    from ecg_b200 import _lib
    lib = _lib.load()
    seed = torch.tensor([12345, 0], device='cuda', dtype=torch.int32)
    mask = torch.empty(batch * n, device='cuda', dtype=torch.uint8)
    counts = torch.empty(batch, device='cuda', dtype=torch.int32)
    st = torch.cuda.current_stream().cuda_stream
    launch = lambda: _lib.check(lib.ecgvit_mpm_mask(seed.data_ptr(), batch, n, n // 2, 49, mask.data_ptr(),
                                                    counts.data_ptr(), st), 'mpm_mask')
    launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        launch()
    e1.record()
    torch.cuda.synchronize()
    return round(e0.elapsed_time(e1) / reps, 4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--batch', type=int, default=256)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--calls-only', action='store_true', help=argparse.SUPPRESS)
    a = ap.parse_args()
    import ecg_b200
    from ecg_b200 import synthetic_batch
    x, y = synthetic_batch(a.batch, length=2500, seed=77)
    x, y = x.cuda(), y.cuda()
    if a.calls_only:
        print(json.dumps(per_call_times(ecg_b200, x, a.reps)))
        return
    torch.manual_seed(77)
    cls = ecg_b200.EcgVit(config=config(ecg_b200)).cuda().train()
    torch.manual_seed(77)
    pre = ecg_b200.EcgVitForMaskedPatchModeling(config=config(ecg_b200), mask_ratio=0.5).cuda().train()
    legs = {'classification': (ecg_b200.FusedTrainer(cls, use_cuda_graph=True, data_parallel=False), y),
            'pretrain': (ecg_b200.FusedTrainer(pre, use_cuda_graph=True, data_parallel=False), None)}
    for tr, labels in legs.values():
        for _ in range(a.warmup):
            tr.step(x, labels)
    torch.cuda.synchronize()
    times = {k: [] for k in legs}
    losses = {}
    for _ in range(a.rounds):   # alternating rounds: both legs see the same clocks and neighbours
        for k, (tr, labels) in legs.items():
            ms, losses[k] = step_ms(tr, x, labels, a.steps)
            times[k].append(ms)
    med = {k: statistics.median(v) for k, v in times.items()}
    del legs, cls, pre
    torch.cuda.empty_cache()
    # per-call times in a process of its own: the single-stream engine is chosen when the engine is created
    env = dict(os.environ, ECGVIT_WGRAD_STREAM='0')
    out = subprocess.run([sys.executable, __file__, '--calls-only', '--batch', str(a.batch), '--reps', str(a.reps)],
                         env=env, capture_output=True, text=True, check=True)
    calls = json.loads(out.stdout.strip().splitlines()[-1])
    # the mask draw compares every pair of keys of a record: its cost at the per-lead geometry (cfg4: 12 x 5000, patch 25,
    # n = 2400) as well as at cfg2's n = 50
    mask_ms = {f'n{n}_B{b}': mask_draw_ms(ecg_b200, n, b) for n, b in ((50, a.batch), (2400, 32), (2400, 256))}
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip()
    row = {'config': 'cfg2: ecg-vit-base bf16 12x2500 P50 B=%d dropout 0.1 mask_ratio 0.5' % a.batch,
           'gpu': q,
           'pretrain_samples_per_s': round(a.batch / med['pretrain'] * 1e3, 1),
           'classification_samples_per_s': round(a.batch / med['classification'] * 1e3, 1),
           'pretrain_ms_per_step': round(med['pretrain'], 3), 'classification_ms_per_step': round(med['classification'], 3),
           'pretrain_over_classification': round(med['pretrain'] / med['classification'], 4),
           'rounds_ms': {k: [round(t, 3) for t in v] for k, v in times.items()},
           'last_loss': losses, 'new_call_ms': calls, 'mask_draw_ms': mask_ms}
    print(json.dumps(row))


if __name__ == '__main__':
    main()
