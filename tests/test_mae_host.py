"""CPU tier: MAE-style pre-training -- parameter layout, the encoder hand-off to `EcgVit`, gradient-bucket placement, the
oracle's visible gather / unshuffle / loss, and the constructor's rejections."""
import pytest
import torch

from conftest import GOLDEN_CFG
from ecg_b200 import EcgVit, EcgVitConfig, EcgVitForMaskedAutoencoding
from oracle.ecg_vit_oracle import OracleConfig, synthetic_batch
from oracle.mae_oracle import OracleMaskedAutoencoder, gather_visible, unshuffle, visible_positions

HEAD = ['vit.mlp_head.0.weight', 'vit.mlp_head.0.bias', 'vit.mlp_head.1.weight', 'vit.mlp_head.1.bias']
DEC = dict(decoder_hidden_size=32, decoder_num_hidden_layers=2, decoder_num_attention_heads=2,
           decoder_intermediate_size=64)


def test_state_dict_keys_order_and_shapes_load_strictly_into_the_oracle():
    cfg = EcgVitConfig(**GOLDEN_CFG)
    torch.manual_seed(1)
    mae = EcgVitForMaskedAutoencoding(config=cfg, **DEC)
    sd = mae.state_dict()
    keys = list(sd)
    cls_keys = [k for k in EcgVit(config=cfg).state_dict() if k not in HEAD]
    assert keys[:len(cls_keys)] == cls_keys   # EcgVit's encoder keys first, in EcgVit's order, no mask token
    rest = keys[len(cls_keys):]
    assert rest[:6] == ['decoder.mask_token', 'decoder.pos_embedding', 'decoder.norm.weight', 'decoder.norm.bias',
                        'decoder.embed.weight', 'decoder.embed.bias']
    assert rest[-4:] == ['recon_head.0.weight', 'recon_head.0.bias', 'recon_head.1.weight', 'recon_head.1.bias']
    assert all(k.startswith('decoder.transformer.layers.') for k in rest[6:-4])
    d, dd, K = cfg.hidden_size, DEC['decoder_hidden_size'], cfg.patch_size * cfg.num_channels
    assert tuple(sd['decoder.mask_token'].shape) == (1, 1, dd) and float(sd['decoder.mask_token'].abs().sum()) == 0
    assert tuple(sd['decoder.pos_embedding'].shape) == (1, 11, dd) and float(sd['decoder.pos_embedding'].std()) > 0.5
    assert tuple(sd['decoder.embed.weight'].shape) == (dd, d) and tuple(sd['decoder.norm.weight'].shape) == (d,)
    assert tuple(sd['recon_head.1.weight'].shape) == (K, dd)
    assert tuple(sd['decoder.transformer.layers.1.1.fn.net.0.weight'].shape) == (DEC['decoder_intermediate_size'], dd)
    oracle = OracleMaskedAutoencoder(OracleConfig(**GOLDEN_CFG), **DEC)
    assert list(oracle.state_dict()) == keys
    oracle.load_state_dict(sd, strict=True)
    mae.load_state_dict(oracle.state_dict(), strict=True)
    short = list(mae._short_names().values())
    assert short[len(cls_keys):len(cls_keys) + 6] == ['dec.mask', 'dec.pos', 'dec.ln.w', 'dec.ln.b', 'dec.embed.w',
                                                      'dec.embed.b']
    assert 'dec1.ff2.b' in short and 'dec0.qkv.w' in short and short[-4:] == ['recon.ln.w', 'recon.ln.b', 'recon.w',
                                                                                 'recon.b']


def test_encoder_state_dict_transfers_to_ecgvit():
    cfg = EcgVitConfig(**GOLDEN_CFG)
    torch.manual_seed(3)
    mae = EcgVitForMaskedAutoencoding(config=cfg, **DEC)
    enc = mae.encoder_state_dict()
    assert all(k.startswith('vit.') for k in enc)
    fine = EcgVit(config=cfg)
    res = fine.load_state_dict(enc, strict=False)
    assert sorted(res.missing_keys) == sorted(HEAD) and res.unexpected_keys == []
    for k, v in enc.items():
        assert torch.equal(fine.state_dict()[k], v), k


def test_decoder_and_recon_head_sit_in_the_first_bucket():
    """the decoder's and the recon head's gradients are produced first in backward: the first bucket (trigger depth - 1);
    pos / cls / embedding, produced last, stay in the trigger -1 bucket"""
    from ecg_b200.model import _ALIGN
    from ecg_b200.parallel import bucket_slices
    cfg = EcgVitConfig(**dict(GOLDEN_CFG, num_hidden_layers=3))
    mae = EcgVitForMaskedAutoencoding(config=cfg, **DEC)
    params = dict(mae.named_parameters())
    off, layout = 0, {}
    for name, key in mae._short_names().items():   # the offsets `_flatten` assigns
        layout[key] = (off, params[name].numel())
        off += (params[name].numel() + _ALIGN - 1) // _ALIGN * _ALIGN
    depth = cfg.num_hidden_layers
    slices = bucket_slices([layout[f'l{l}.ln1.w'][0] for l in range(depth)], off, depth, 1)

    def trigger_of(key):
        o, n = layout[key]
        (t,) = [t for t, lo, hi in slices if lo <= o and o + n <= hi]
        return t

    for key in ('pos', 'cls', 'embed.w', 'embed.b'):
        assert trigger_of(key) == -1, key
    for key in [k for k in layout if k.startswith('dec') or k.startswith('recon')]:
        assert trigger_of(key) == depth - 1, key
    assert slices[0][0] == depth - 1


def test_oracle_gather_and_unshuffle_equal_a_per_record_loop():
    g = torch.Generator().manual_seed(4)
    B, n, F, k = 5, 12, 3, 7
    mask = torch.zeros(B, n, dtype=torch.bool)
    for b in range(B):
        mask[b, torch.randperm(n, generator=g)[:k]] = True
    mask[0] = torch.arange(n) < k          # first patch masked
    mask[1] = torch.arange(n) >= n - k     # last patch masked
    assert (mask.sum(1) == k).all()
    a = torch.randn(B, n, F, generator=g)
    vis = visible_positions(mask)
    got = gather_visible(a, vis)
    t = torch.randn(B, n - k + 1, F, generator=g)
    tok = torch.randn(1, 1, F, generator=g)
    u = unshuffle(t, mask, tok)
    for b in range(B):
        pos = [p for p in range(n) if not mask[b, p]]
        assert vis[b].tolist() == pos
        assert torch.equal(got[b], a[b, pos])
        assert torch.equal(u[b, 0], t[b, 0])
        j = 0
        for p in range(n):
            if mask[b, p]:
                assert torch.equal(u[b, 1 + p], tok[0, 0])
            else:
                assert torch.equal(u[b, 1 + p], t[b, 1 + j])
                j += 1


def test_oracle_loss_is_the_masked_mse():
    torch.manual_seed(6)
    mae = OracleMaskedAutoencoder(OracleConfig(**GOLDEN_CFG), **DEC).eval()
    x, _ = synthetic_batch(2, length=GOLDEN_CFG['max_signal_length'])
    mask = torch.zeros(2, 10, dtype=torch.bool)
    mask[0, [1, 4]] = True
    mask[1, [0, 9]] = True
    loss, pred = mae(x, mask)
    a = mae.patches(x)
    want = torch.cat([(pred[0, [1, 4]] - a[0, [1, 4]]).reshape(-1), (pred[1, [0, 9]] - a[1, [0, 9]]).reshape(-1)])
    assert torch.allclose(loss, want.pow(2).mean(), rtol=1e-6, atol=0)
    # the encoder never sees a masked patch: changing one leaves the encoder output alone
    x2 = x.clone()
    x2[0, :, 50:100] += 1.0     # patch 1 of record 0 (masked)
    _, z = mae.encode(x, mask)
    _, z2 = mae.encode(x2, mask)
    assert torch.equal(z, z2) and z.shape == (2, 9, GOLDEN_CFG['hidden_size'])


def test_constructor_rejections():
    cfg = EcgVitConfig(**GOLDEN_CFG)   # n = 10
    for ratio in (0.0, 0.04, 0.96, 1.0):   # no masked or no visible patch
        with pytest.raises(ValueError, match='masked'):
            EcgVitForMaskedAutoencoding(config=cfg, mask_ratio=ratio, **DEC)
    EcgVitForMaskedAutoencoding(config=cfg, mask_ratio=0.1, **DEC)
    EcgVitForMaskedAutoencoding(config=cfg, mask_ratio=0.9, **DEC)
    with pytest.raises(ValueError, match='multiple of decoder_num_attention_heads'):
        EcgVitForMaskedAutoencoding(config=cfg, decoder_hidden_size=36, decoder_num_attention_heads=8)
    with pytest.raises(ValueError, match='decoder_intermediate_size'):
        EcgVitForMaskedAutoencoding(config=cfg, **dict(DEC, decoder_intermediate_size=100))
    with pytest.raises(ValueError, match='multiple of 8'):
        EcgVitForMaskedAutoencoding(config=EcgVitConfig(**dict(GOLDEN_CFG, patch_size=25)), **DEC)   # 25 * 12 = 300
    EcgVitForMaskedAutoencoding(config=EcgVitConfig(**dict(GOLDEN_CFG, patch_size=25, per_lead_tokens=True)), **DEC)
