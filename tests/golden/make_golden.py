"""
Generates tests/golden/ecgvit_small_step.npz THROUGH THE REFERENCE'S OWN WRAPPER.

Run in the build container only (needs /root/reference):   python tests/golden/make_golden.py

What is reference code here: `EcgVit`, `EcgVitConfig` (ecg_transformer/models/ecg_vit.py, imported verbatim via
oracle/ref_shim.py) and the step order of `MyTrainer.train` (models/train.py:271-283) with stock
torch.optim.AdamW / nn.utils.clip_grad_norm_ / transformers' constant schedule.  What is restated: the
un-vendored third-party `vit_pytorch.ViT` (oracle/vit_restated.py) -- the reference repo ships no golden vectors
for this path, so parity stays "unpinned" for that one file (DESIGN.md).
"""
import os
import sys

import numpy as np
import torch
from torch import nn

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from conftest import golden_sample  # noqa: E402
from oracle import ref_shim  # noqa: E402
from oracle.ecg_vit_oracle import synthetic_batch, patch_matrix  # noqa: E402

CFG = dict(max_signal_length=500, patch_size=50, num_channels=12, hidden_size=64, num_hidden_layers=2,
           num_attention_heads=4, intermediate_size=128, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
BATCH, SEED, LR, WD, CLIP, N_STEPS = 4, 77, 3e-4, 1e-2, 1.0, 3


def compact(out):
    """Keeps the file under 1 MB: the initial and step-3 weights stay whole (tests load them as model state), gradients
    and step-1 weights keep the sample `golden_sample` takes.  The key order -- the reference's state_dict order -- is
    kept, and tests check it."""
    return {k: golden_sample(v) if k.startswith(('grad/', 'step1/')) else v for k, v in out.items()}


def main():
    EcgVit, EcgVitConfig, get_train_args, _ = ref_shim.load_reference()
    from transformers import get_constant_schedule_with_warmup
    torch.manual_seed(SEED)
    model = EcgVit(config=EcgVitConfig(**CFG))
    model.train()
    x, y = synthetic_batch(BATCH, length=CFG['max_signal_length'], seed=SEED)
    out = {'x': x.numpy(), 'y': y.numpy()}
    for k, v in model.state_dict().items():
        out['init/' + k] = v.numpy().copy()
    args = get_train_args(dict(schedule='constant', learning_rate=LR, weight_decay=WD, warmup_ratio=0.0), n_train=64)
    optimizer = torch.optim.AdamW(model.parameters(), lr=args['learning_rate'], weight_decay=args['weight_decay'])
    scheduler = get_constant_schedule_with_warmup(optimizer, num_warmup_steps=0)
    for step in range(1, N_STEPS + 1):
        optimizer.zero_grad()
        o = model(sample_values=x, labels=y)
        o.loss.backward()
        if step == 1:
            out['logits'] = o.logits.detach().numpy().copy()
            out['loss'] = np.array(o.loss.item(), dtype=np.float64)
            for k, p in model.named_parameters():
                out['grad/' + k] = p.grad.numpy().copy()
        total_norm = nn.utils.clip_grad_norm_(model.parameters(), max_norm=CLIP, error_if_nonfinite=True)
        out[f'norm{step}'] = np.array(float(total_norm), dtype=np.float64)
        out[f'loss{step}'] = np.array(o.loss.item(), dtype=np.float64)
        optimizer.step()
        scheduler.step()
        if step in (1, N_STEPS):
            for k, v in model.state_dict().items():
                out[f'step{step}/' + k] = v.numpy().copy()
    # eval-mode per-sample loss (loss_reduction='none', train.py:332-333)
    model.eval()
    model.loss_reduction = 'none'
    with torch.no_grad():
        o = model(sample_values=x, labels=y)
    out['eval_loss_none'] = o.loss.numpy().copy()
    out['eval_logits'] = o.logits.numpy().copy()
    # integer-exact patch indexing: feed index values through the reference Rearrange
    idx = torch.arange(2 * 12 * 500, dtype=torch.float32).reshape(2, 12, 500)
    ref_patches = model.vit.to_patch_embedding[0](idx.unsqueeze(-2))  # the einops Rearrange layer
    assert torch.equal(ref_patches.reshape(-1, 600), patch_matrix(idx, 50))
    out['patch_index'] = ref_patches.reshape(-1, 600).numpy().astype(np.int32)
    path = os.path.join(ROOT, 'tests', 'golden', 'ecgvit_small_step.npz')
    np.savez_compressed(path, **compact(out))
    print('wrote', path, f'{os.path.getsize(path) / 1e6:.2f} MB', 'loss', out['loss'], 'norm1', out['norm1'])


if __name__ == '__main__':
    main()
