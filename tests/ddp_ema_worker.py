"""torchrun worker for tests/test_gpu_ddp_ema.py: data-parallel FusedTrainer with the weight moving average over NCCL:
every rank updates its own copy, the copies stay bit-identical, and they match the single-GPU run on the union batch."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ecg_b200  # noqa: E402
from oracle.ecg_vit_oracle import synthetic_batch  # noqa: E402  (seeded input generator only)

CFG = dict(max_signal_length=2500, patch_size=50, num_channels=12, hidden_size=256, num_hidden_layers=4,
           num_attention_heads=8, intermediate_size=1024, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)


def main():
    use_graph = len(sys.argv) > 1 and sys.argv[1] == 'graph'
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    per_rank = 8
    x, y = synthetic_batch(per_rank * world, seed=3)
    kw = dict(learning_rate=1e-3, max_grad_norm=0.05, ema_decay=0.9, ema_warmup=True)
    for dtype, reduce, tol in (('fp32', 'fp32', 2e-5), ('bf16', 'bf16', 2e-2)):
        # different initial weights per rank: rank 0's weights and average are broadcast at start-up
        torch.manual_seed(11 + 1000 * rank)
        model = ecg_b200.EcgVit(config=ecg_b200.EcgVitConfig(compute_dtype=dtype, **CFG)).to(dev).train()
        tr = ecg_b200.FusedTrainer(model, bucket_layers=3, use_cuda_graph=use_graph, grad_reduce_dtype=reduce, **kw)
        xs, ys = x[rank * per_rank:(rank + 1) * per_rank].to(dev), y[rank * per_rank:(rank + 1) * per_rank].to(dev)
        for _ in range(3):
            tr.step(xs, ys)
        torch.cuda.synchronize()
        tr.check_finite()
        ema = tr.ema.buf.clone()
        gathered = [torch.empty_like(ema) for _ in range(world)]
        dist.all_gather(gathered, ema)
        assert all(torch.equal(g, gathered[0]) for g in gathered), 'the averages diverged across ranks'
        if rank == 0:
            torch.manual_seed(11)
            ref = ecg_b200.EcgVit(config=ecg_b200.EcgVitConfig(compute_dtype=dtype, **CFG)).to(dev).train()
            rt = ecg_b200.FusedTrainer(ref, data_parallel=False, **kw)
            for _ in range(3):
                rt.step(x.to(dev), y.to(dev))
            torch.cuda.synchronize()
            err = float((ema - rt.ema.buf).norm() / rt.ema.buf.norm())
            moved = float((ema - model._flat_p).norm() / model._flat_p.norm())
            print(f'[{dtype} reduce {reduce}] graph={use_graph} ema rel err vs union batch {err:.3e} '
                  f'(ema vs weights {moved:.3e})', flush=True)
            assert err < tol and moved > 0, (err, moved)
    dist.barrier()
    torch.cuda.synchronize()
    if rank == 0:
        print('ddp ema ok', flush=True)
    sys.stdout.flush()
    os._exit(0)


if __name__ == '__main__':
    main()
