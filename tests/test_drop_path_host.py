"""CPU tier: stochastic depth (`EcgVitConfig.drop_path_rate`): the config field, the per-block rates, the host replica
of the per-record keep draw, and the oracle injection the GPU tests use (tests/drop_path_oracle.py)."""
import pytest
import torch

import ecg_b200
from ecg_b200 import EcgVit, EcgVitConfig, EcgVitForMaskedAutoencoding, EcgVitForMaskedPatchModeling
from ecg_b200.config import drop_path_rates
from conftest import GOLDEN_CFG
from drop_path_oracle import path_keep, path_site, inject_drop_path
from oracle.ecg_vit_oracle import OracleConfig, OracleEcgVit, synthetic_batch


def test_config_default_is_zero_and_bad_rates_raise():
    assert EcgVitConfig().drop_path_rate == 0.0
    assert EcgVitConfig(drop_path_rate=0.1).drop_path_rate == 0.1
    for bad in (-0.1, 1.0, 1.5):
        with pytest.raises(ValueError):
            EcgVitConfig(drop_path_rate=bad)
    c = EcgVitConfig(**GOLDEN_CFG)
    c.drop_path_rate = 1.0     # set after construction: the model rejects it too
    with pytest.raises(ValueError):
        EcgVit(num_class=5, config=c)


def test_state_dict_keys_do_not_change():
    for cls, kw in ((EcgVit, dict(num_class=5)), (EcgVitForMaskedPatchModeling, {}),
                    (EcgVitForMaskedAutoencoding, dict(decoder_hidden_size=32, decoder_num_hidden_layers=1,
                                                       decoder_num_attention_heads=4, decoder_intermediate_size=64))):
        a = cls(config=EcgVitConfig(**GOLDEN_CFG), **kw).state_dict().keys()
        b = cls(config=EcgVitConfig(drop_path_rate=0.2, **GOLDEN_CFG), **kw).state_dict().keys()
        assert list(a) == list(b)


@pytest.mark.parametrize('depth', [1, 2, 5, 12])
def test_per_layer_rates_are_timm_linspace(depth):
    c = EcgVitConfig(**dict(GOLDEN_CFG, num_hidden_layers=depth), drop_path_rate=0.3)
    assert drop_path_rates(c) == [float(v) for v in torch.linspace(0, 0.3, depth)]
    assert drop_path_rates(c)[0] == 0.0
    if depth == 1:
        assert drop_path_rates(c) == [0.0]


def test_replica_is_deterministic_and_keeps_at_rate():
    B = 65536
    for r in (0.1, 0.5):
        a = path_keep(1234, 4 * 8 + 2, r, B)
        b = path_keep(1234, 4 * 8 + 2, r, B)
        assert torch.equal(a, b)
        kept = float((a > 0).float().mean())
        assert abs(kept - (1 - r)) < 0.01, (r, kept)
        q = round(r * 65536) / 65536   # the rate is quantised to 1/65536
        assert torch.allclose(a[a > 0], torch.tensor(1.0 / (1.0 - q)))
    assert not torch.equal(path_keep(1234, 34, 0.5, 64), path_keep(1235, 34, 0.5, 64))
    assert torch.equal(path_keep(1234, 34, 0.0, 8), torch.ones(8))


@pytest.mark.parametrize('depth', [1, 2, 8, 24])
def test_sites_do_not_collide_with_dropout_or_mask_sites(depth):
    dropout_sites = set(range(0, 4 * depth + 1))
    mask_site = 4 * depth + 1
    sites = [path_site(depth, l, j) for l in range(depth) for j in (0, 1)]
    assert len(set(sites)) == len(sites)
    assert not (set(sites) & dropout_sites) and mask_site not in sites
    assert min(sites) == 4 * depth + 2


def test_oracle_injection_matches_hand_composition():
    torch.manual_seed(0)
    cfg = dict(GOLDEN_CFG, num_hidden_layers=3)
    oracle = OracleEcgVit(num_class=5, config=OracleConfig(**dict(cfg, num_class=5))).eval()
    x, _ = synthetic_batch(6, length=500, num_class=5, seed=1)
    seed, rate = 777, 0.5
    handles = inject_drop_path(oracle.vit.transformer, seed, rate)
    try:
        with torch.no_grad():
            got = oracle(sample_values=x).logits
    finally:
        for h in handles:
            h.remove()
    # hand-composed: the same blocks, x + s[b] * branch(x)
    vit = oracle.vit
    D = len(vit.transformer.layers)
    rates = [float(v) for v in torch.linspace(0, rate, D)]
    with torch.no_grad():
        img = x.unsqueeze(2)
        t = vit.to_patch_embedding(img)
        B = t.shape[0]
        t = torch.cat((vit.cls_token.expand(B, -1, -1), t), dim=1) + vit.pos_embedding[:, :t.shape[1] + 1]
        dropped = 0
        for l, (attn, ff) in enumerate(vit.transformer.layers):
            sa = path_keep(seed, path_site(D, l, 0), rates[l], B).view(B, 1, 1)
            sf = path_keep(seed, path_site(D, l, 1), rates[l], B).view(B, 1, 1)
            dropped += int((sa == 0).sum() + (sf == 0).sum())
            t = t + sa * attn(t)
            t = t + sf * ff(t)
        want = vit.mlp_head(t[:, 0])
        plain = oracle(sample_values=x).logits
    assert dropped > 0
    assert torch.allclose(got, want, rtol=0, atol=0)
    assert not torch.allclose(got, plain)
