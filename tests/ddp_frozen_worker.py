"""torchrun worker for tests/test_gpu_ddp_frozen.py: data-parallel FusedTrainer with frozen parameters over NCCL == the
single-GPU step on the union batch, with the same requires_grad flags."""
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


def freeze(model, pattern):
    depth = model.config.num_hidden_layers
    for name, p in model.named_parameters():
        if pattern == 'head_only':
            frozen = not name.startswith('vit.mlp_head.')
        else:   # the last block and the head train
            frozen = not (name.startswith('vit.mlp_head.') or name.startswith(f'vit.transformer.layers.{depth - 1}.'))
        p.requires_grad_(not frozen)
    return model


def main():
    use_graph = len(sys.argv) > 1 and sys.argv[1] == 'graph'
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    per_rank = 8
    x, y = synthetic_batch(per_rank * world, seed=3)
    for pattern in ('head_only', 'last'):
        for dtype, reduce, tol in (('fp32', 'fp32', 2e-5), ('bf16', 'bf16', 2e-2), ('bf16', 'fp32', 2e-2)):
            torch.manual_seed(11 + 1000 * rank)
            model = freeze(ecg_b200.EcgVit(config=ecg_b200.EcgVitConfig(compute_dtype=dtype, **CFG)), pattern)
            model = model.to(dev).train()
            tr = ecg_b200.FusedTrainer(model, learning_rate=1e-3, max_grad_norm=0.05, bucket_layers=3,
                                       use_cuda_graph=use_graph, grad_reduce_dtype=reduce)
            xs, ys = x[rank * per_rank:(rank + 1) * per_rank].to(dev), y[rank * per_rank:(rank + 1) * per_rank].to(dev)
            lo = None
            for i in range(3):
                tr.step(xs, ys)
                if i == 0:
                    lo = model.trainable_span().lo
                    start = model._flat_p[:lo].clone()   # rank 0's frozen prefix, broadcast at start-up
            torch.cuda.synchronize()
            tr.check_finite()
            flat = model._flat_p.clone()
            assert torch.equal(flat[:lo], start), 'a frozen tensor moved'
            gathered = [torch.empty_like(flat) for _ in range(world)]
            dist.all_gather(gathered, flat)
            assert all(torch.equal(g, gathered[0]) for g in gathered), 'ranks diverged'
            if rank == 0:
                torch.manual_seed(11)
                ref = freeze(ecg_b200.EcgVit(config=ecg_b200.EcgVitConfig(compute_dtype=dtype, **CFG)), pattern)
                ref = ref.to(dev).train()
                rt = ecg_b200.FusedTrainer(ref, learning_rate=1e-3, max_grad_norm=0.05, data_parallel=False)
                for _ in range(3):
                    rt.step(x.to(dev), y.to(dev))
                torch.cuda.synchronize()
                err = float((flat - ref._flat_p).norm() / ref._flat_p.norm())
                gn = (tr.grad_norm(), rt.grad_norm())
                print(f'[{pattern} {dtype} reduce {reduce}] graph={use_graph} rel err vs union batch {err:.3e}  '
                      f'grad norms {gn}', flush=True)
                assert err < tol, err
                assert abs(gn[0] - gn[1]) < 5e-2 * gn[1]
    dist.barrier()
    torch.cuda.synchronize()
    if rank == 0:
        print('ddp frozen ok', flush=True)
    sys.stdout.flush()
    os._exit(0)


if __name__ == '__main__':
    main()
