#!/usr/bin/env python
"""
bench.py -- ECG-ViT training-step throughput (BASELINE.json metric: train samples/s on synthetic 12x2500, bf16).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cfg2|cfg4|cfg5]
                    [--batch B | --global-batch G] [--no-graph] [--api-loop] [--dump-outputs DIR]

One "step" = zero_grad + forward + backward + (bucketed grad all-reduce) + clip_grad_norm(1.0) + AdamW on one batch of
synthetic signals (seed 77), i.e. /root/reference/ecg_transformer/models/train.py:271-283 without its logging.
Workload at N=1: BASELINE.json configs[1] -- ECG-ViT base (d=768, 12 layers, 12 heads, patch 50), bf16, batch 256.
For N>1 every rank keeps batch 256 (weak scaling; N=8 is configs[2]'s global batch 2048); `--global-batch 2048` runs
configs[2] as written (1024 / 512 / 256 per GPU at N = 2 / 4 / 8, strong scaling).

Prints ONE JSON line (rank 0).  `value` = samples/s with inputs resident in HBM; `e2e` = the same through the public
API from pinned HOST buffers (H2D of the batch + D2H of the loss inside the timed region); `roofline` = the tcgen05
GEMM kernel family against the measured cuBLAS bf16 BURST peak (the kernels are timed alone), `roofline_kernels` = that
plus every memory-bound kernel of the step against the measured copy bandwidth; `cpu_baseline` = the CPU oracle port on this box's cores.
`--impl reference` times the reference's own CPU path (oracle port: the reference is pure Python over an un-vendored
package and /root/reference does not exist on the GPU box) on the same model config, bounded batch.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'ecg_vit_base_bf16_train_samples_per_s'
UNIT = 'samples/s'
BASE_CFG = dict(max_signal_length=2500, patch_size=50, num_channels=12, hidden_size=768, num_hidden_layers=12,
                num_attention_heads=12, intermediate_size=3072, hidden_dropout_prob=0.1,
                attention_probs_dropout_prob=0.1)  # dropout 0.1 = the reference's default (ecg_vit.py:38-39)
NUM_CLASS = 71
# BASELINE.json `configs`: [1] is the metric's workload (default); the others are selectable for scaling / parity runs
WORKLOADS = {
    'cfg2': dict(model=BASE_CFG, per_gpu_batch=256,
                 name='ECG-ViT base (d=768, 12 layers, 12 heads, patch 50) bf16 pre-training step, batch 256 per GPU, '
                      '12x2500 signals (BASELINE.json configs[1]; configs[2] at N=8)'),
    'cfg4': dict(model=dict(BASE_CFG, max_signal_length=5000, patch_size=25, per_lead_tokens=True), per_gpu_batch=32,
                 name='ECG-ViT base long-signal 12x5000, patch 25, per-lead tokens (N = 2401), batch 32 per GPU '
                      '(BASELINE.json configs[3]; the batch is not specified there)'),
    'cfg5': dict(model=dict(BASE_CFG, hidden_size=1024, num_hidden_layers=24, num_attention_heads=16,
                            intermediate_size=4096, activation_checkpointing=True), per_gpu_batch=512,
                 name='ECG-ViT large (d=1024, 24 layers, 16 heads) bf16, activation checkpointing, 512 per GPU = global '
                      '4096 at N=8, 12x2500 signals (BASELINE.json configs[4])'),
}


def train_flops_per_sample(c):
    """SURVEY.md 8d / BASELINE.md 3: 2 FLOP per MAC, contractions only, no input dgrad for the patch embedding
    (activation recomputation is NOT counted: algorithmic FLOPs)"""
    per_lead = bool(c.get('per_lead_tokens', False))
    n_patch = c['max_signal_length'] // c['patch_size'] * (c['num_channels'] if per_lead else 1)
    patch_dim = c['patch_size'] * (1 if per_lead else c['num_channels'])
    N = n_patch + 1
    d, mlp, depth = c['hidden_size'], c['intermediate_size'], c['num_hidden_layers']
    inner = d
    f_embed = 2 * n_patch * patch_dim * d
    f_lin = 2 * N * (3 * d * inner + inner * d + 2 * d * mlp)
    f_attn = 4 * N * N * inner
    f_head = 2 * d * NUM_CLASS
    return 3 * (depth * (f_lin + f_attn) + f_head) + 2 * f_embed


def cpu_model_string():
    try:
        for ln in open('/proc/cpuinfo'):
            if ln.startswith('model name'):
                return ln.split(':', 1)[1].strip()
    except OSError:
        pass
    return 'unknown'


def gemm_traffic():
    """average DRAM bytes per tcgen05-GEMM launch from the committed ncu capture of one step (profiles/)"""
    for name in ('r02_step_launches.json', 'r01_step_final.json'):
        try:
            fam = json.load(open(os.path.join(ROOT, 'profiles', name)))['gemm_family']
            return fam['dram_bytes_per_launch'], ('profiles/%s (ncu dram__bytes_read.sum + dram__bytes_write.sum, avg over '
                                                  'the GEMM launches of one step)' % name)
        except Exception:
            continue
    return None, 'no ncu capture committed'


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(tflops_sustained=p['bf16_tflops_sustained'], tflops_burst=p['bf16_tflops'], hbm_gbs=p['hbm_gbs'],
                    source='MEASURED_PEAKS.json')
    return dict(tflops_sustained=1400.0, tflops_burst=1590.0, hbm_gbs=6650.0, source='B200_PROFILING.md fallback')


class ClockSampler:
    """SM clock / power / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe): NVML from a
    background thread every 20 ms (nvidia-smi -lms as a fallback)."""
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.samples, self.stop_flag, self.thread, self.nvml = [], False, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')  # CUDA ordinal -> NVML index
            idx = int(vis.split(',')[self.index]) if vis and all(t.strip().isdigit() for t in vis.split(',')) else self.index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.FIELDS}', '--format=csv,noheader,nounits',
                                          '-lms', '100', '-i', str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        bits = {'hw_slowdown': n.nvmlClocksEventReasonHwSlowdown if hasattr(n, 'nvmlClocksEventReasonHwSlowdown') else 0x8,
                'hw_thermal_slowdown': 0x40, 'sw_thermal_slowdown': 0x20, 'sw_power_cap': 0x4}
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                try:
                    rs = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    rs = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.samples.append((sm, pw, [k for k, b in bits.items() if rs & b]))
            except Exception:
                pass
            time.sleep(0.02)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            if not self.samples:
                return {'sm_mhz': None, 'sm_max_mhz': self.max_sm, 'reasons': ['no samples'], 'samples': 0}
            power = [p for _, p, _ in self.samples]
            thr = statistics.median(power)
            loaded = [s for s, p, _ in self.samples if p >= thr]
            reasons = sorted({r for _, _, rs in self.samples for r in rs})
            return {'sm_mhz': statistics.median(loaded), 'sm_max_mhz': self.max_sm, 'reasons': reasons,
                    'samples': len(self.samples), 'power_w_max': max(power), 'source': 'nvml, 20 ms period'}
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            f = [t.strip() for t in ln.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[3:7]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        if sm:
            thr = statistics.median(power)
            loaded = [s for s, p in zip(sm, power) if p >= thr] or sm
            return {'sm_mhz': statistics.median(loaded), 'sm_max_mhz': max(mx), 'reasons': sorted(reasons),
                    'samples': len(sm), 'power_w_max': max(power), 'source': 'nvidia-smi -lms 100'}
        return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples'], 'samples': 0}


def cpu_reference_steps(cfg, batch, steps, warmup, threads=None):
    """the reference path on host cores: oracle restatement of EcgVit/ViT + stock torch AdamW / clip_grad_norm_"""
    import torch
    from oracle.ecg_vit_oracle import OracleConfig, OracleEcgVit, OracleTrainer, synthetic_batch
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    torch.manual_seed(77)
    cfg = {k: v for k, v in cfg.items() if k != 'activation_checkpointing'}  # a B200 knob; the reference has none
    model = OracleEcgVit(config=OracleConfig(**cfg)).train()
    tr = OracleTrainer(model, learning_rate=3e-4, weight_decay=1e-2, schedule='constant')
    x, y = synthetic_batch(batch, length=cfg['max_signal_length'])
    for _ in range(warmup):
        tr.step(x, y)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        tr.step(x, y)
        times.append(time.perf_counter() - t0)
    return times, torch.get_num_threads()


CFG1 = dict(max_signal_length=2500, patch_size=50, num_channels=12, hidden_size=256, num_hidden_layers=4,
            num_attention_heads=8, intermediate_size=1024, hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1)


def cpu_cfg1():
    """BASELINE.json configs[0] exactly as SURVEY.md 8(d) / BASELINE.md 4 define its timing: d256 / 4 layers / 8 heads /
    mlp 1024, batch 32, fp32, all host threads, 3 warm-up + 10 timed steps, median"""
    times, threads = cpu_reference_steps(CFG1, 32, steps=10, warmup=3)
    med = statistics.median(times)
    return {'workload': 'BASELINE.json configs[0]: ECG-ViT small (d=256, 4 layers, 8 heads, patch 50) fwd+bwd+clip+AdamW fp32, '
                        '12x2500, batch 32, CPU', 'value': 32 / med, 'unit': UNIT, 'ms_per_step_median': 1e3 * med,
            'steps': 10, 'warmup': 3, 'cores': threads, 'os_cpu_count': os.cpu_count(), 'cpu': cpu_model_string(),
            'kind': 'port', 'dropout': 0.1}


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    wl = WORKLOADS[args.config]
    cfg = wl['model']
    batch = args.ref_batch if args.config != 'cfg4' else 1
    times, threads = cpu_reference_steps(cfg, batch, args.steps, max(1, min(args.warmup, 2)))
    ms = 1e3 * sum(times) / len(times)
    value = batch / (ms / 1e3)
    sample = (f'{args.steps} steps of the same model (fp32, stock torch AdamW + clip_grad_norm_) on a bounded batch of '
              f'{batch} synthetic signals (the GPU arm uses {wl["per_gpu_batch"]} per step and GPU)')
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': wl['name'], 'batch_per_step': batch, 'device': 'cpu', 'dropout': args.dropout,
                   'cpu': cpu_model_string()},
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': threads, 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def dump_outputs(path, model, trainer, loss, logits, n_sample=1 << 20):
    """Writes what the timed step handed its caller, as float32 .npy files under `path`: the loss, the logits, the
    gradient norm and a fixed sample of the updated parameters (seed 0, 2^20 indices into the parameters concatenated
    in state_dict order, which does not depend on the library's internal flat layout).  Two builds run with the same
    arguments start from the same weights and inputs, so their files can be compared one for one."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    params = torch.cat([v.detach().reshape(-1).float() for v in model.state_dict().values()])
    idx = torch.from_numpy(np.random.default_rng(0).integers(0, params.numel(), n_sample)).to(params.device)
    arrays = {'loss': loss, 'logits': logits, 'grad_norm': torch.tensor(trainer.grad_norm()), 'params_sample': params[idx]}
    for name, t in arrays.items():
        np.save(os.path.join(path, name + '.npy'), t.detach().float().cpu().numpy())


def time_graph(torch, launch_all, reps):
    """device time per launch of `launch_all()` (which issues `reps` launches on the current stream): the batch is
    captured into a CUDA graph and the REPLAY is timed with CUDA events (launched one by one from Python, a 10-60 us
    kernel's queue runs dry between calls and the idle gaps would be charged to the kernel)"""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        launch_all()  # warm-up (function attributes, tensor maps) outside capture
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        launch_all()
    g.replay()
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best / reps


def hbm_kernel_rooflines(torch, _lib, cfg, B, p_drop, n_params, peaks, launches):
    """The memory-bound kernels of the step, each timed alone at its cfg shape (graph replay over 12 distinct buffer
    sets, so consecutive launches do not hit in L2) against the measured copy bandwidth.  Algorithmic bytes per launch:
    the operands the op must read and write once (DESIGN.md section 4)."""
    lib = _lib.load()
    dev = torch.device('cuda', torch.cuda.current_device())
    per_lead = bool(cfg.get('per_lead_tokens', False))
    N = cfg['max_signal_length'] // cfg['patch_size'] * (cfg['num_channels'] if per_lead else 1) + 1
    d, mlp, H = cfg['hidden_size'], cfg['intermediate_size'], cfg['num_attention_heads']
    M, dh, reps = B * N, d // H, 12
    bf = torch.bfloat16
    out = []

    def add(name, bytes_per_launch, ms, per_step):
        gbs = bytes_per_launch / (ms * 1e-3) / 1e9
        out.append({'kernel': name, 'bound': 'hbm', 'achieved': gbs, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                    'frac': gbs / peaks['hbm_gbs'], 'bytes_per_launch': bytes_per_launch, 'ms_per_launch': ms,
                    'launches_per_step': per_step, 'timing': 'alone, CUDA-graph replay of 12 launches, CUDA events'})

    def st():
        return torch.cuda.current_stream().cuda_stream

    seed = torch.tensor([1234], dtype=torch.int32, device=dev)
    sp = seed.data_ptr() if p_drop > 0 else None
    # LayerNorm forward / backward
    xs = [torch.randn(M, d, device=dev).to(bf) for _ in range(reps)]
    ys = [torch.empty(M, d, device=dev, dtype=bf) for _ in range(reps)]
    gamma, beta = torch.ones(d, device=dev), torch.zeros(d, device=dev)
    mean, rstd = torch.empty(M, device=dev), torch.empty(M, device=dev)
    ms = time_graph(torch, lambda: [_lib.check(lib.ecgvit_layernorm_fwd(
        xs[i].data_ptr(), gamma.data_ptr(), beta.data_ptr(), ys[i].data_ptr(), mean.data_ptr(), rstd.data_ptr(), M, d,
        1e-5, _lib.BF16, st()), 'layernorm_fwd') for i in range(reps)], reps)
    add('layernorm_fwd_kernel', 4 * M * d, ms, launches.get('layernorm_fwd', 0))
    dres = torch.randn(M, d, device=dev).to(bf)
    dxm = torch.empty(M, d, device=dev, dtype=bf)
    dg, db, dc = (torch.zeros(d, device=dev) for _ in range(3))
    scr = torch.empty(int(lib.ecgvit_layernorm_bwd_scratch_floats(d)), device=dev)
    lib.ecgvit_layernorm_fwd(xs[0].data_ptr(), gamma.data_ptr(), beta.data_ptr(), ys[0].data_ptr(), mean.data_ptr(),
                             rstd.data_ptr(), M, d, 1e-5, _lib.BF16, st())
    ms = time_graph(torch, lambda: [_lib.check(lib.ecgvit_layernorm_bwd(
        ys[i].data_ptr(), xs[i].data_ptr(), gamma.data_ptr(), mean.data_ptr(), rstd.data_ptr(), dres.data_ptr(),
        ys[(i + 1) % reps].data_ptr(), dg.data_ptr(), db.data_ptr(), dc.data_ptr(), scr.data_ptr(),
        dxm.data_ptr() if p_drop > 0 else None, p_drop, 3, sp, M, d, 1, _lib.BF16, st()), 'layernorm_bwd_partial')
        for i in range(reps)], reps)
    add('layernorm_bwd_kernel' + (' (+ dropout-masked copy)' if p_drop > 0 else ''), (10 if p_drop > 0 else 8) * M * d, ms,
        launches.get('layernorm_bwd_partial', 0) + launches.get('layernorm_bwd', 0))
    del xs, ys, dres, dxm
    # attention forward / backward (tcgen05 kernels: HBM-bound at N = 51)
    qkv = [torch.randn(M, 3 * d, device=dev).to(bf) for _ in range(reps)]
    o = [torch.empty(M, d, device=dev, dtype=bf) for _ in range(reps)]
    lse = torch.empty(B, H, N, device=dev)
    n_scr = int(lib.ecgvit_attention_bwd_scratch_floats(B, N, H, dh, _lib.BF16))
    ascr = torch.empty(max(n_scr, 1), device=dev)
    ms = time_graph(torch, lambda: [_lib.check(lib.ecgvit_attention_fwd(
        qkv[i].data_ptr(), o[i].data_ptr(), lse.data_ptr(), B, N, H, dh, dh ** -0.5, p_drop, 1, sp, _lib.BF16, st()),
        'attention_fwd') for i in range(reps)], reps)
    add('attn_tc_fwd_kernel' if dh == 64 else 'attention_fwd', 8 * M * d, ms, launches.get('attention_fwd', 0))
    dqkv = torch.empty(M, 3 * d, device=dev, dtype=bf)
    ms = time_graph(torch, lambda: [_lib.check(lib.ecgvit_attention_bwd(
        qkv[i].data_ptr(), o[i].data_ptr(), o[(i + 1) % reps].data_ptr(), lse.data_ptr(), dqkv.data_ptr(),
        ascr.data_ptr() if n_scr else None, B, N, H, dh, dh ** -0.5, p_drop, 1, sp, _lib.BF16, st()), 'attention_bwd')
        for i in range(reps)], reps)
    add('attn_tc_bwd_kernel' if dh == 64 else 'attention_bwd', 14 * M * d + (0 if N <= 64 else 2 * M * d), ms,
        launches.get('attention_bwd', 0) + launches.get('attention_bwd_flash', 0))
    del qkv, o, dqkv
    # FF1 bias gradient
    du = [torch.randn(M, mlp, device=dev).to(bf) for _ in range(4)]
    col = torch.zeros(mlp, device=dev)
    ms = time_graph(torch, lambda: [_lib.check(lib.ecgvit_colsum(du[i % 4].data_ptr(), col.data_ptr(), M, mlp, mlp,
                                                                  _lib.BF16, st()), 'colsum') for i in range(reps)], reps)
    add('colsum_kernel', 2 * M * mlp, ms, launches.get('colsum', 0))
    del du
    # gradient norm + AdamW over the flat buffers
    n = (n_params + 3) // 4 * 4
    p_, m_, v_, g_ = (torch.zeros(n, device=dev) for _ in range(4))
    g_.normal_()
    shadow = torch.empty(n, device=dev, dtype=bf)
    hyper = torch.tensor(_lib.adamw_hyper(3e-4, 0.9, 0.999, 1e-8, 1e-2, 1, 1.0, 1.0), device=dev, dtype=torch.float32)
    stats = torch.zeros(_lib.STATS_FLOATS, device=dev)
    ms = time_graph(torch, lambda: [_lib.check(lib.ecgvit_grad_sumsq(g_.data_ptr(), _lib.F32, n, hyper.data_ptr(), stats.data_ptr(),
                                                                      st()), 'grad_sumsq') for _ in range(4)], 4)
    add('grad_sumsq_kernel', 4 * n, ms, 1)
    ms = time_graph(torch, lambda: [_lib.check(lib.ecgvit_adamw_step(
        p_.data_ptr(), m_.data_ptr(), v_.data_ptr(), g_.data_ptr(), _lib.F32, shadow.data_ptr(), n, hyper.data_ptr(),
        stats.data_ptr(), 0, st()), 'adamw_step') for _ in range(4)], 4)
    add('adamw_kernel (clip + AdamW + bf16 shadow)', 30 * n, ms, 1)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='cfg2', choices=sorted(WORKLOADS), help='BASELINE.json workload (default: the metric\'s)')
    ap.add_argument('--batch', type=int, default=None, help='per-GPU batch (default: the workload\'s)')
    ap.add_argument('--global-batch', type=int, default=None,
                    help='fixed GLOBAL batch split over the ranks (strong scaling; BASELINE.json configs[2]: 2048)')
    ap.add_argument('--ref-batch', type=int, default=16, help='bounded CPU batch of the reference arm')
    ap.add_argument('--no-graph', action='store_true', help='launch kernels from Python instead of one CUDA graph')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-roofline', action='store_true', help='skip the per-kernel roofline legs')
    ap.add_argument('--api-loop', action='store_true',
                    help='also time the reference-style loop through the nn.Module API (INTEGRATION.md section A)')
    ap.add_argument('--dropout', type=float, default=0.1, help='hidden / attention-probs dropout (reference default 0.1)')
    ap.add_argument('--profile-json', default=None, help='write the per-kernel event breakdown here')
    ap.add_argument('--nccl-max-ctas', type=int, default=None,
                    help='cap the CTAs of NCCL\'s collectives (communicator config): they compete with the persistent GEMMs for SMs')
    ap.add_argument('--bucket-layers', type=int, default=1, help='encoder layers per gradient all-reduce bucket')
    ap.add_argument('--defer', action='store_true',
                    help='run clip + AdamW of step k beside the forward pass of step k + 1 (FusedTrainer(defer_optimizer=True)); '
                         'measured neutral at cfg2: the slices displace CTAs of the persistent forward GEMMs')
    ap.add_argument('--grad-reduce', default='auto', choices=['auto', 'fp32', 'bf16'], help='dtype of the gradient all-reduce')
    ap.add_argument('--dump-outputs', default=None, metavar='DIR',
                    help='after the timed steps, write the outputs of the last one as DIR/<name>.npy (rank 0)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the GPU step (--impl ours)')
    wl = WORKLOADS[args.config]
    MODEL_CFG = dict(wl['model'])
    MODEL_CFG['hidden_dropout_prob'] = MODEL_CFG['attention_probs_dropout_prob'] = args.dropout
    wl = dict(wl, model=MODEL_CFG)
    WORKLOADS[args.config] = wl
    if args.impl == 'reference':
        return run_reference_arm(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    import ecg_b200
    from ecg_b200 import _lib
    from ecg_b200 import synthetic_batch  # seeded input generator (SURVEY.md 8d); nothing of oracle/ on this arm

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        if args.nccl_max_ctas:
            opts = dist.ProcessGroupNCCL.Options()
            opts.config.max_ctas = args.nccl_max_ctas
            opts.config.min_ctas = min(args.nccl_max_ctas, 1)
            dist.init_process_group('nccl', device_id=dev, pg_options=opts)
        else:
            dist.init_process_group('nccl', device_id=dev)
    assert _lib.load().ecgvit_device_ok() == 1, 'bench.py needs an sm_100 (B200) device: there is no fallback path'

    if args.global_batch is not None:
        assert args.global_batch % world == 0, '--global-batch must divide by the number of ranks'
        B, scaling = args.global_batch // world, 'strong'
    else:
        B, scaling = (args.batch or wl['per_gpu_batch']), 'weak'
    torch.manual_seed(77)
    model = ecg_b200.EcgVit(config=ecg_b200.EcgVitConfig(compute_dtype='bf16', **MODEL_CFG)).to(dev).train()
    use_graph = not args.no_graph  # NCCL all-reduces are captured into the step graph as well
    trainer = ecg_b200.FusedTrainer(model, learning_rate=3e-4, weight_decay=1e-2, schedule='constant',
                                    max_grad_norm=1.0, use_cuda_graph=use_graph, bucket_layers=args.bucket_layers,
                                    grad_reduce_dtype=args.grad_reduce, defer_optimizer=args.defer)
    xh, yh = synthetic_batch(B, length=MODEL_CFG['max_signal_length'], seed=77 + rank)
    xh, yh = xh.pin_memory(), yh.pin_memory()
    x, y = xh.to(dev), yh.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    # ---- device-resident arm -------------------------------------------------------------------------------
    for _ in range(args.warmup):
        trainer.step(x, y)
    torch.cuda.synchronize()
    n0 = _lib.launch_counter[0]
    if not use_graph:
        trainer.step(x, y)
        launches_per_step = _lib.launch_counter[0] - n0
    else:
        launches_per_step = trainer.launches_per_step
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    last = [None]

    def train_step():
        last[0] = trainer.step(x, y)

    total_ms = timed(train_step, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    trainer.check_finite()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, trainer, *last[0])  # before later steps overwrite the step's buffers
    ms_per_step = total_ms / args.steps
    value = world * B / (ms_per_step / 1e3)

    # ---- end-to-end arm: pinned host batch -> H2D -> step -> D2H of the loss, every step -------------------
    # The caller reads every step's loss on the host (train.py:278), but one step late: the D2H copy of step i's loss is
    # ordered before step i+1's kernels and is waited for only after step i+1 has been enqueued, and the H2D copy of
    # batch i+1 runs on a side stream during step i.  Nothing is skipped: per step the whole batch goes in and 4 bytes
    # come out.
    loss_host = torch.zeros(2).pin_memory()
    loss_ready = [torch.cuda.Event(), torch.cuda.Event()]
    staged = [trainer.stage(xh, yh)]
    e2e_i = [0]
    losses = []

    def e2e_step():
        i = e2e_i[0]
        xd, yd = staged[0]
        loss, _ = trainer.step(xd, yd)
        staged[0] = trainer.stage(xh, yh)
        loss_host[i & 1:(i & 1) + 1].copy_(loss.reshape(1), non_blocking=True)
        loss_ready[i & 1].record()
        if i > 0:
            loss_ready[(i - 1) & 1].synchronize()
            losses.append(float(loss_host[(i - 1) & 1]))
        e2e_i[0] = i + 1

    for _ in range(2):
        e2e_step()
    e2e_ms = timed(e2e_step, args.steps) / args.steps
    e2e_value = world * B / (e2e_ms / 1e3)
    assert all(l == l for l in losses), 'non-finite loss read back in the end-to-end arm'
    trainer.flush()          # the deferred optimizer's last update (nothing below may see half-updated state)
    trainer.check_finite()

    # ---- optional: the reference-style loop through the nn.Module API (INTEGRATION.md section A) ------------
    api_loop = None
    if args.api_loop and world == 1:
        from ecg_b200 import FusedAdamW, clip_grad_norm_
        m2 = ecg_b200.EcgVit(config=ecg_b200.EcgVitConfig(compute_dtype='bf16', **MODEL_CFG)).to(dev).train()
        opt = FusedAdamW(m2, lr=3e-4, weight_decay=1e-2)

        def api_step():
            opt.zero_grad()
            out = m2(sample_values=x, labels=y)
            out.loss.backward()
            clip_grad_norm_(m2, 1.0)
            opt.step()

        for _ in range(3):
            api_step()
        api_ms = timed(api_step, max(5, args.steps // 2)) / max(5, args.steps // 2)
        api_loop = {'ms_per_step': api_ms, 'value': B / (api_ms / 1e3), 'unit': UNIT,
                    'what': 'zero_grad / model(**inputs) / loss.backward() / clip_grad_norm_ / FusedAdamW.step(), eager launches'}
        del m2, opt

    # ---- roofline legs ------------------------------------------------------------------------------------------
    roofline, kernels, roofline_kernels = None, None, None
    flops_step = B * train_flops_per_sample(MODEL_CFG)
    if rank == 0 and not args.no_roofline:
        peaks = measured_peaks()
        eager = ecg_b200.FusedTrainer(model, use_cuda_graph=False, data_parallel=False)
        model._after_layer_backward = None  # the profiling step runs on rank 0 alone: no collective
        model._engine.side_stream = None    # single stream, so consecutive event deltas are per-call device times
        eager.step(x, y)
        torch.cuda.synchronize()
        _lib.profile[0] = []
        start = torch.cuda.Event(enable_timing=True)
        start.record()
        eager.step(x, y)
        torch.cuda.synchronize()
        rec, _lib.profile[0] = _lib.profile[0], None
        prev, agg = start, {}
        gemm_calls = {}
        for name, meta, ev in rec:
            dt_ms = prev.elapsed_time(ev)
            prev = ev
            a = agg.setdefault(name, [0, 0.0])
            a[0] += 1
            a[1] += dt_ms
            if name == 'gemm':
                gemm_calls.setdefault(tuple(meta[:6]), []).append(meta[6])
        step_ms_eager = sum(v[1] for v in agg.values())
        # eager per-call event deltas include host launch gaps: they give call counts and rough SHARES only
        kernels = {k: {'calls': v[0], 'ms': round(v[1], 4), 'share': round(v[1] / step_ms_eager, 4)} for k, v in agg.items()}
        launches = {k: v[0] for k, v in agg.items()}
        # The dominant kernel family, timed on its own: every distinct GEMM of the step (shape, operand majors, epilogue)
        # is re-launched back to back (a replayed CUDA graph of >= 12 launches), rotating over the step's own instances
        # of that call (different layers -> different weights and activation buffers), weighted by launches per step.
        import ctypes
        lib = _lib.load()
        gemm_rows, gemm_flops, gemm_ms = [], 0.0, 0.0
        for key, instances in gemm_calls.items():
            M_, N_, K_, epi, a_k, b_k = key
            reps = max(12, len(instances))
            ms = time_graph(torch, lambda: [_lib.check(lib.ecgvit_gemm(ctypes.byref(instances[i % len(instances)]),
                                                                        torch.cuda.current_stream().cuda_stream), 'gemm')
                                            for i in range(reps)], reps)
            fl = 2.0 * M_ * N_ * K_
            gemm_rows.append(dict(M=M_, N=N_, K=K_, epi=epi, a_kmajor=a_k, b_kmajor=b_k, launches_per_step=len(instances),
                                  ms=round(ms, 4), tflops=round(fl / (ms * 1e-3) / 1e12, 1)))
            gemm_flops += fl * len(instances)
            gemm_ms += ms * len(instances)
        achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12
        n_gemm = agg['gemm'][0]
        whole = flops_step / (ms_per_step * 1e-3) / 1e12
        roofline = {
            'kernel': 'gemm_tc2_kernel (tcgen05.mma cta_group::2 kind::f16; all fwd / dgrad / wgrad launches of one step)',
            'bound': 'tensor', 'achieved': achieved, 'peak': peaks['tflops_burst'], 'unit': 'TFLOP/s',
            'frac': achieved / peaks['tflops_burst'], 'traffic': gemm_traffic()[0], 'traffic_source': gemm_traffic()[1],
            'peak_source': f"{peaks['source']} bf16_tflops (burst: the kernels are timed alone, as sub-millisecond graph "
                           f"replays), of measured",
            'launches': n_gemm, 'avg_launch_ms': gemm_ms / n_gemm, 'flops_per_launch_avg': gemm_flops / n_gemm,
            'step_share': (gemm_ms / ms_per_step), 'step_share_note': 'sum of GEMM launch times / device-timed step',
            'frac_of_sustained_peak': achieved / peaks['tflops_sustained'],
            'whole_step_tflops': whole, 'whole_step_frac_of_nominal_2250': whole / 2250.0,
            'whole_step_frac_of_measured_sustained': whole / peaks['tflops_sustained'],
            'whole_step_note': 'algorithmic FLOPs of the step / device-timed step (a long step: sustained peak applies)',
        }
        roofline_kernels = [dict(roofline, kernel='gemm_tc2_kernel family', launches_per_step=n_gemm)]
        roofline_kernels = [{k: v for k, v in roofline_kernels[0].items()
                             if k in ('kernel', 'bound', 'achieved', 'peak', 'unit', 'frac', 'launches_per_step')}]
        if not MODEL_CFG.get('per_lead_tokens'):
            n_params = sum(p.numel() for p in model.parameters())
            roofline_kernels += hbm_kernel_rooflines(torch, _lib, MODEL_CFG, B, args.dropout, n_params, peaks, launches)
        if args.profile_json:
            with open(args.profile_json, 'w') as f:
                json.dump({'kernels': kernels, 'roofline': roofline, 'roofline_kernels': roofline_kernels,
                           'gemm_launches': gemm_rows}, f, indent=1)

    # ---- CPU baseline (rank 0, N=1 only): bounded sample of the same workload + BASELINE configs[0] ------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cb = 8 if args.config != 'cfg4' else 1
        times, threads = cpu_reference_steps(MODEL_CFG, cb, steps=2, warmup=1)
        v = cb / (sum(times) / len(times))
        cpu_baseline = {'value': v, 'unit': UNIT, 'cores': threads, 'kind': 'port', 'cpu': cpu_model_string(),
                        'sample': f'2 timed steps (+1 warm-up) of the same model in fp32 on a batch of {cb} synthetic '
                                  f'signals: oracle restatement + stock torch AdamW/clip_grad_norm_',
                        'cfg1': cpu_cfg1()}

    if rank == 0:
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': scaling, 'vs_baseline': None,
            'dtype': 'bf16', 'data': 'synthetic',
            'config': {'workload': wl['name'], 'global_batch': world * B, 'per_gpu_batch': B, 'dropout': args.dropout,
                       'parallelism': f'dp{world}', 'nccl_max_ctas': args.nccl_max_ctas, 'bucket_layers': args.bucket_layers, 'grad_reduce': args.grad_reduce,
                       'l2': 'per-step working set (GBs of activations + optimizer traffic) exceeds the 126 MB L2, no '
                             'explicit flush',
                       'cuda_graph': use_graph, 'optimizer': 'AdamW lr 3e-4 wd 1e-2, clip_grad_norm 1.0',
                       'optimizer_placement': 'each step runs clip + AdamW of the PREVIOUS step beside its forward pass '
                                              '(every timed step contains exactly one full update)' if args.defer
                                              else 'end of step',
                       'residual_stream': 'fp32' if model._res_f32 else 'bf16',
                       'activation_checkpointing': bool(MODEL_CFG.get('activation_checkpointing', False))},
            'clocks': clocks,
            'e2e': {'value': e2e_value, 'unit': UNIT, 'ms_per_step': e2e_ms,
                    'h2d_bytes_per_step': world * (xh.numel() + yh.numel()) * 4, 'd2h_bytes_per_step': world * 4},
            'gpu_launches': launches_per_step * args.steps,
            'tflops': flops_step * world / (ms_per_step * 1e-3) / 1e12,
            'roofline': roofline, 'roofline_kernels': roofline_kernels, 'cpu_baseline': cpu_baseline, 'kernels': kernels,
            'api_loop': api_loop,
        }
        print(json.dumps(line), flush=True)
    sys.stdout.flush()
    if world > 1:
        # NCCL communicators captured in live CUDA graphs do not tear down cleanly: leave without the destructor dance
        torch.cuda.synchronize()
        os._exit(0)


if __name__ == '__main__':
    main()
