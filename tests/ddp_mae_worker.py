"""torchrun worker for tests/test_gpu_ddp_mae.py: MAE-style pre-training with a data-parallel FusedTrainer == the CPU
oracle's step on the union batch with every rank's drawn mask."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ecg_b200  # noqa: E402
from oracle.ecg_vit_oracle import OracleConfig, synthetic_batch  # noqa: E402
from oracle.mae_oracle import OracleMaskedAutoencoder  # noqa: E402
from oracle.mpm_oracle import OracleMaskedPatchTrainer  # noqa: E402

CFG = dict(max_signal_length=500, patch_size=50, num_channels=12, hidden_size=64, num_hidden_layers=3,
           num_attention_heads=4, intermediate_size=128, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
DEC = dict(decoder_hidden_size=32, decoder_num_hidden_layers=2, decoder_num_attention_heads=2, decoder_intermediate_size=64)


def main():
    use_graph = len(sys.argv) > 1 and sys.argv[1] == 'graph'
    shared = len(sys.argv) > 2 and sys.argv[2] == 'shared'   # both ranks on GPU 0, gloo collectives (eager only)
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    dev = torch.device('cuda', 0 if shared else local)
    torch.cuda.set_device(dev)
    if shared:
        dist.init_process_group('gloo')
    else:
        dist.init_process_group('nccl', device_id=dev)
    per_rank, steps = 4, 3
    x, _ = synthetic_batch(per_rank * world, length=CFG['max_signal_length'], seed=3)
    torch.manual_seed(11)
    oracle = OracleMaskedAutoencoder(OracleConfig(**CFG), **DEC).train()
    with torch.no_grad():
        oracle.decoder.mask_token.normal_()
    # every rank but 0 starts from different weights: the trainer must broadcast rank 0's replica
    torch.manual_seed(11 + 1000 * rank)
    model = ecg_b200.EcgVitForMaskedAutoencoding(config=ecg_b200.EcgVitConfig(compute_dtype='fp32', **CFG), **DEC)
    if rank == 0:
        model.load_state_dict(oracle.state_dict(), strict=True)
    model.to(dev).train()
    tr = ecg_b200.FusedTrainer(model, learning_rate=1e-3, max_grad_norm=1.0, bucket_layers=1, use_cuda_graph=use_graph)
    xs = x[rank * per_rank:(rank + 1) * per_rank].to(dev)
    masks = []
    for _ in range(steps):
        tr.step(xs)
        mine = model._engine.mask().to(torch.uint8)
        parts = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(parts, mine)
        masks.append(torch.cat(parts).bool().cpu())
    torch.cuda.synchronize()
    tr.check_finite()
    flat = model._flat_p.clone()
    gathered = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(gathered, flat)
    assert all(torch.equal(g, gathered[0]) for g in gathered), 'ranks diverged'
    if rank == 0:
        n = masks[0].shape[1]
        assert not torch.equal(masks[0][:per_rank], masks[0][per_rank:2 * per_rank]), 'ranks drew the same masks'
        ot = OracleMaskedPatchTrainer(oracle, learning_rate=1e-3, max_grad_norm=1.0)
        for m in masks:   # equal counts per record, so the mean of the per-rank losses is the union-batch loss
            assert (m.sum(1) == round(0.75 * n)).all()
            ot.step(x, m)
        sd = model.state_dict()
        worst = max(float((sd[k].cpu().double() - v.double()).norm() / v.double().norm().clamp_min(1e-30))
                    for k, v in oracle.state_dict().items())
        print(f'world={world} graph={use_graph} shared={shared} worst parameter rel err vs union-batch oracle {worst:.3e}', flush=True)
        assert worst < 2e-5, worst
    dist.barrier()
    torch.cuda.synchronize()
    if rank == 0:
        print('ddp mae ok', flush=True)
    sys.stdout.flush()
    os._exit(0)   # communicators captured in live CUDA graphs do not tear down cleanly


if __name__ == '__main__':
    main()
