"""CPU tier: masked-patch pre-training -- parameter layout, the encoder hand-off to `EcgVit`, the host replica of the
device mask draw, the oracle, and `unpatchify`."""
import torch

from conftest import GOLDEN_CFG
from ecg_b200 import EcgVit, EcgVitConfig, EcgVitForMaskedPatchModeling, _lib
from oracle.ecg_vit_oracle import OracleConfig, OracleEcgVit, patch_matrix, synthetic_batch
from oracle.mpm_oracle import OracleMaskedPatchModel

HEAD = ['vit.mlp_head.0.weight', 'vit.mlp_head.0.bias', 'vit.mlp_head.1.weight', 'vit.mlp_head.1.bias']


def test_state_dict_keys_and_order():
    cfg = EcgVitConfig(**GOLDEN_CFG)
    pre = EcgVitForMaskedPatchModeling(config=cfg)
    keys = list(pre.state_dict())
    cls_keys = [k for k in EcgVit(config=cfg).state_dict() if k not in HEAD]
    vit_keys = [k for k in keys if k.startswith('vit.')]
    # EcgVit's encoder keys in EcgVit's order, with the mask token right after the CLS token
    assert vit_keys == cls_keys[:cls_keys.index('vit.cls_token') + 1] + ['vit.mask_token'] + \
        cls_keys[cls_keys.index('vit.cls_token') + 1:]
    assert keys.index('vit.mask_token') < keys.index('vit.transformer.layers.0.0.norm.weight')
    assert keys[len(vit_keys):] == ['recon_head.0.weight', 'recon_head.0.bias', 'recon_head.1.weight',
                                    'recon_head.1.bias']
    sd = pre.state_dict()
    d, K = cfg.hidden_size, cfg.patch_size * cfg.num_channels
    assert tuple(sd['vit.mask_token'].shape) == (1, 1, d) and float(sd['vit.mask_token'].abs().sum()) == 0.0
    assert tuple(sd['recon_head.1.weight'].shape) == (K, d) and tuple(sd['recon_head.0.weight'].shape) == (d,)
    # flat-buffer names: the mask token sits before layer 0 (the last gradient bucket of a data-parallel run)
    short = list(pre._short_names().values())
    assert short.index('mask') < short.index('l0.ln1.w')
    assert short[-4:] == ['recon.ln.w', 'recon.ln.b', 'recon.w', 'recon.b']
    # the keys match the CPU oracle's, so its weights load strictly
    assert list(OracleMaskedPatchModel(OracleConfig(**GOLDEN_CFG)).state_dict()) == keys


def test_per_lead_recon_width():
    cfg = EcgVitConfig(**dict(GOLDEN_CFG, per_lead_tokens=True))
    pre = EcgVitForMaskedPatchModeling(config=cfg)
    assert tuple(pre.state_dict()['recon_head.1.weight'].shape) == (cfg.patch_size, cfg.hidden_size)


def test_encoder_state_dict_transfers_to_ecgvit():
    cfg = EcgVitConfig(**GOLDEN_CFG)
    torch.manual_seed(3)
    pre = EcgVitForMaskedPatchModeling(config=cfg)
    enc = pre.encoder_state_dict()
    assert 'vit.mask_token' not in enc and all(k.startswith('vit.') for k in enc)
    fine = EcgVit(config=cfg)
    res = fine.load_state_dict(enc, strict=False)
    assert sorted(res.missing_keys) == sorted(HEAD) and res.unexpected_keys == []
    for k, v in enc.items():
        assert torch.equal(fine.state_dict()[k], v), k


def test_mask_replica_draws_exactly_k_and_is_seeded():
    B, n, site = 16, 50, 9
    for k in (0, 1, 25, 49, 50):
        m = _lib.mpm_mask(1234, B, n, k, site)
        assert m.dtype == torch.bool and tuple(m.shape) == (B, n)
        assert (m.sum(1) == k).all()
    a = _lib.mpm_mask(1234, B, n, 25, site)
    assert torch.equal(a, _lib.mpm_mask(1234, B, n, 25, site))       # deterministic per seed
    assert not torch.equal(a, _lib.mpm_mask(1235, B, n, 25, site))   # another seed, another mask
    assert not torch.equal(a, _lib.mpm_mask(1234, B, n, 25, site + 1))
    assert len({tuple(r.tolist()) for r in a}) == B                  # records differ
    # nested: the k smallest keys contain the k - 1 smallest
    assert (_lib.mpm_mask(7, B, n, 10, site) >= _lib.mpm_mask(7, B, n, 9, site)).all()


def test_mask_replica_is_the_rank_of_the_counter_hash():
    B, n, k, seed, site = 3, 40, 13, 99, 5
    keys = _lib.counter_hash(seed, site, torch.arange(B * n, dtype=torch.int64)).reshape(B, n)
    idx = torch.arange(n)
    rank = ((keys[:, None, :] < keys[:, :, None]) |
            ((keys[:, None, :] == keys[:, :, None]) & (idx[None, None, :] < idx[None, :, None]))).sum(-1)
    assert torch.equal(_lib.mpm_mask(seed, B, n, k, site), rank < k)


def test_oracle_without_mask_reproduces_the_restated_vit_token_stream():
    ocfg = OracleConfig(**GOLDEN_CFG)
    torch.manual_seed(5)
    pre = OracleMaskedPatchModel(ocfg)
    cls_model = OracleEcgVit(config=ocfg)
    res = cls_model.load_state_dict({k: v for k, v in pre.state_dict().items() if k != 'vit.mask_token'}, strict=False)
    assert sorted(res.missing_keys) == sorted(HEAD)
    x, _ = synthetic_batch(3, length=GOLDEN_CFG['max_signal_length'])
    seen = {}
    cls_model.vit.transformer.register_forward_hook(lambda mod, inp, out: seen.setdefault('z', out))
    cls_model.eval()(x)
    pre.eval()
    mask = torch.zeros(3, 10, dtype=torch.bool)
    a, z = pre.encode(x, mask)
    assert torch.equal(z, seen['z'])
    assert torch.equal(a.reshape(-1, a.shape[-1]), patch_matrix(x, GOLDEN_CFG['patch_size']))
    # a masked patch changes the stream only through the mask token
    mask[0, 3] = True
    _, zm = pre.encode(x, mask)
    assert torch.equal(zm[1:], z[1:]) and not torch.equal(zm[0], z[0])


def test_oracle_loss_is_the_masked_mse():
    torch.manual_seed(6)
    pre = OracleMaskedPatchModel(OracleConfig(**GOLDEN_CFG)).eval()
    x, _ = synthetic_batch(2, length=GOLDEN_CFG['max_signal_length'])
    mask = torch.zeros(2, 10, dtype=torch.bool)
    mask[0, [1, 4]] = True
    mask[1, 7] = True
    loss, pred = pre(x, mask)
    a = pre.patches(x)
    want = torch.cat([(pred[0, [1, 4]] - a[0, [1, 4]]).reshape(-1), (pred[1, 7] - a[1, 7])]).pow(2).mean()
    assert torch.allclose(loss, want, rtol=1e-6, atol=0)


def test_unpatchify_inverts_the_patch_matrix():
    cfg = EcgVitConfig(**GOLDEN_CFG)
    pre = EcgVitForMaskedPatchModeling(config=cfg)
    x = torch.randn(3, cfg.num_channels, cfg.max_signal_length)
    P = cfg.patch_size
    a = patch_matrix(x, P).reshape(3, cfg.max_signal_length // P, P * cfg.num_channels)
    assert torch.equal(pre.unpatchify(a), x)
    # per-lead tokens: token (c, w), features t
    lead = EcgVitForMaskedPatchModeling(config=EcgVitConfig(**dict(GOLDEN_CFG, per_lead_tokens=True)))
    a = x.reshape(3, cfg.num_channels, -1, P).reshape(3, -1, P)
    assert torch.equal(lead.unpatchify(a), x)
    oracle = OracleMaskedPatchModel(OracleConfig(**dict(GOLDEN_CFG, per_lead_tokens=True)))
    assert torch.equal(oracle.patches(x), a)


def test_mask_ratio_is_validated():
    import pytest
    with pytest.raises(ValueError):
        EcgVitForMaskedPatchModeling(config=EcgVitConfig(**GOLDEN_CFG), mask_ratio=1.5)


def test_patch_width_that_the_residual_kernels_cannot_read_is_rejected():
    import pytest
    with pytest.raises(ValueError, match='multiple of 8'):
        EcgVitForMaskedPatchModeling(config=EcgVitConfig(**dict(GOLDEN_CFG, patch_size=25)))   # 25 * 12 = 300
    # per-lead rows are padded instead
    EcgVitForMaskedPatchModeling(config=EcgVitConfig(**dict(GOLDEN_CFG, patch_size=25, per_lead_tokens=True)))


def test_mask_token_gradient_falls_in_the_last_bucket_and_the_recon_head_in_the_first():
    """data-parallel buckets are slices of the flat buffer (forward order): the mask token's gradient, produced last by
    the embedding backward, must sit in the trigger -1 bucket; the recon head's, produced first, in the top bucket"""
    from ecg_b200.model import _ALIGN
    from ecg_b200.parallel import bucket_slices
    cfg = EcgVitConfig(**dict(GOLDEN_CFG, num_hidden_layers=3))
    pre = EcgVitForMaskedPatchModeling(config=cfg)
    params = dict(pre.named_parameters())
    off, layout = 0, {}
    for name, key in pre._short_names().items():   # the offsets `_flatten` assigns
        layout[key] = (off, params[name].numel())
        off += (params[name].numel() + _ALIGN - 1) // _ALIGN * _ALIGN
    depth = cfg.num_hidden_layers
    slices = bucket_slices([layout[f'l{l}.ln1.w'][0] for l in range(depth)], off, depth, 1)

    def trigger_of(key):
        o, n = layout[key]
        (t,) = [t for t, lo, hi in slices if lo <= o and o + n <= hi]
        return t

    assert trigger_of('mask') == -1 and trigger_of('cls') == -1 and trigger_of('embed.w') == -1
    for key in ('recon.ln.w', 'recon.ln.b', 'recon.w', 'recon.b'):
        assert trigger_of(key) == depth - 1
    assert slices[0][0] == depth - 1   # issued first in backward
