"""CPU tier: fine-tuning support -- `param_groups_lrd` against a direct restatement of MAE's algorithm, the grouped
AdamW's group map, the mean-pooled oracle head, and the rejections (unknown pool, a parameter in two groups, betas
that differ between groups)."""
import pytest
import torch

from conftest import GOLDEN_CFG
import ecg_b200
from ecg_b200 import (EcgVit, EcgVitConfig, EcgVitForMaskedAutoencoding, EcgVitForMaskedPatchModeling, FusedAdamW,
                      FusedTrainer, param_groups_lrd)
from ecg_b200.optim import UNGROUPED, group_map, group_names
from oracle.ecg_vit_oracle import OracleConfig, OracleEcgVit, synthetic_batch

MAE_DEC = dict(decoder_hidden_size=32, decoder_num_hidden_layers=2, decoder_num_attention_heads=2,
               decoder_intermediate_size=64)


def models():
    cfg = EcgVitConfig(compute_dtype='fp32', **GOLDEN_CFG)
    return [EcgVit(config=cfg), EcgVitForMaskedPatchModeling(cfg), EcgVitForMaskedAutoencoding(cfg, **MAE_DEC)]


def mae_param_groups_lrd(model, weight_decay, no_weight_decay_list, layer_decay):
    """MAE's util/lr_decay.py `param_groups_lrd` + `get_layer_id_for_vit`, with this model's parameter names
    (cls_token / pos_embed / patch_embed / blocks.i -> vit.cls_token / vit.pos_embedding / vit.to_patch_embedding /
    vit.transformer.layers.i; the mask token sits with the embedding as in MAE's fine-tuning of SimMIM encoders)"""
    num_layers = model.config.num_hidden_layers + 1
    layer_scales = [layer_decay ** (num_layers - i) for i in range(num_layers + 1)]

    def get_layer_id_for_vit(name):
        if name in ['vit.cls_token', 'vit.pos_embedding', 'vit.mask_token']:
            return 0
        elif name.startswith('vit.to_patch_embedding'):
            return 0
        elif name.startswith('vit.transformer.layers'):
            return int(name.split('.')[3]) + 1
        else:
            return num_layers

    param_group_names, param_groups = {}, {}
    for n, p in model.named_parameters():
        if not p.requires_grad:
            continue
        if p.ndim == 1 or n in no_weight_decay_list:
            g_decay, this_decay = 'no_decay', 0.
        else:
            g_decay, this_decay = 'decay', weight_decay
        layer_id = get_layer_id_for_vit(n)
        group_name = 'layer_%d_%s' % (layer_id, g_decay)
        if group_name not in param_group_names:
            this_scale = layer_scales[layer_id]
            param_group_names[group_name] = {'lr_scale': this_scale, 'weight_decay': this_decay, 'params': []}
            param_groups[group_name] = {'lr_scale': this_scale, 'weight_decay': this_decay, 'params': []}
        param_group_names[group_name]['params'].append(n)
        param_groups[group_name]['params'].append(p)
    return list(param_group_names.values())


@pytest.mark.parametrize('layer_decay', [0.75, 1.0])
@pytest.mark.parametrize('which', [0, 1, 2])
def test_param_groups_lrd_matches_mae(which, layer_decay):
    model = models()[which]
    names = {id(p): n for n, p in model.named_parameters()}
    got = param_groups_lrd(model, weight_decay=0.05, layer_decay=layer_decay)
    want = mae_param_groups_lrd(model, 0.05, ['vit.pos_embedding', 'vit.cls_token', 'vit.mask_token',
                                              'decoder.mask_token'], layer_decay)
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert set(g) == {'params', 'lr_scale', 'weight_decay'}
        assert [names[id(p)] for p in g['params']] == w['params']
        assert g['lr_scale'] == pytest.approx(w['lr_scale'], rel=1e-15) and g['weight_decay'] == w['weight_decay']
    # every trainable parameter is in exactly one group
    assert sorted(n for w in want for n in w['params']) == sorted(n for n, _ in model.named_parameters())
    depth = model.config.num_hidden_layers
    by_name = {n: g for g in got for n in (names[id(p)] for p in g['params'])}
    assert by_name['vit.transformer.layers.0.0.fn.to_qkv.weight']['lr_scale'] == pytest.approx(layer_decay ** depth)
    assert by_name['vit.to_patch_embedding.1.weight']['lr_scale'] == pytest.approx(layer_decay ** (depth + 1))
    assert by_name['vit.cls_token']['weight_decay'] == 0.0 and by_name['vit.pos_embedding']['weight_decay'] == 0.0
    assert by_name['vit.transformer.layers.1.1.norm.weight']['weight_decay'] == 0.0
    assert by_name['vit.transformer.layers.1.1.fn.net.0.weight']['weight_decay'] == 0.05
    top = 'vit.mlp_head.1.weight' if which == 0 else 'recon_head.1.weight'
    assert by_name[top]['lr_scale'] == 1.0


def test_frozen_parameters_are_left_out_of_the_groups():
    model = models()[0]
    model.vit.cls_token.requires_grad_(False)
    got = param_groups_lrd(model)
    assert all(p is not model.vit.cls_token for g in got for p in g['params'])


@pytest.mark.parametrize('which', [0, 2])
def test_group_map_marks_every_block_of_every_parameter(which):
    model = models()[which]
    groups = param_groups_lrd(model)
    groups = groups[:-1]            # the last group's parameters stay ungrouped
    names = group_names(model, groups)
    gm = group_map(model, names)
    layout, total = model._flat_layout()
    assert gm.dtype == torch.uint8 and gm.numel() * 64 == total
    gid = {n: i for i, ns in enumerate(names) for n in ns}
    for o, n, _, name in layout.values():
        assert o % 64 == 0
        blocks = gm[o // 64:(o + n + 63) // 64]
        assert bool((blocks == gid.get(name, UNGROUPED)).all()), name
    # the slices the deferred optimizer issues start on tensor starts, i.e. on whole map entries
    depth = model.config.num_hidden_layers
    for l in range(depth):
        assert layout[f'l{l}.ln1.w'][0] % 64 == 0


def test_mean_pool_oracle_equals_a_hand_composed_mean():
    cfg = OracleConfig(**GOLDEN_CFG)
    torch.manual_seed(3)
    oracle = OracleEcgVit(config=cfg).eval()
    oracle.vit.pool = 'mean'    # the restated vit_pytorch ViT reads `pool` at forward
    x, y = synthetic_batch(3, length=cfg.max_signal_length)
    v = oracle.vit
    with torch.no_grad():
        t = v.to_patch_embedding(x.unsqueeze(-2))
        t = torch.cat((v.cls_token.expand(t.shape[0], -1, -1), t), dim=1) + v.pos_embedding[:, :t.shape[1] + 1]
        t = v.transformer(t)
        want = v.mlp_head(t.mean(dim=1))
        got = oracle(x).logits
        cls = v.mlp_head(t[:, 0])
    assert torch.allclose(got, want, rtol=0, atol=0)
    assert not torch.allclose(got, cls)


def test_pool_config_and_rejections():
    assert EcgVitConfig().pool == 'cls'
    with pytest.raises(ValueError):
        EcgVitConfig(pool='max')
    cfg = EcgVitConfig(**GOLDEN_CFG)
    cfg.pool = 'token'
    with pytest.raises(ValueError):
        EcgVit(config=cfg)
    m = EcgVit(config=EcgVitConfig(pool='mean', **GOLDEN_CFG))
    assert m._mean_pool and m.vit.pool == 'mean'
    # the pre-training heads read every patch token: pool does not apply there, and the keys do not change
    pre = EcgVitForMaskedAutoencoding(EcgVitConfig(pool='mean', **GOLDEN_CFG), **MAE_DEC)
    assert not pre._mean_pool
    assert list(m.state_dict()) == list(EcgVit(config=EcgVitConfig(**GOLDEN_CFG)).state_dict())
    missing, unexpected = m.load_state_dict(pre.encoder_state_dict(), strict=False)
    assert sorted(missing) == ['vit.mlp_head.0.bias', 'vit.mlp_head.0.weight', 'vit.mlp_head.1.bias',
                               'vit.mlp_head.1.weight'] and not unexpected


def test_group_rejections():
    model = models()[0]
    groups = param_groups_lrd(model)
    twice = groups + [{'params': [model.vit.cls_token], 'lr_scale': 1.0, 'weight_decay': 0.0}]
    with pytest.raises(ValueError):
        FusedAdamW(model, lr=1e-3, param_groups=twice)
    with pytest.raises(ValueError):
        group_names(model, twice)
    other = [dict(g) for g in groups]
    other[1]['betas'] = (0.8, 0.999)
    with pytest.raises(ValueError):
        FusedAdamW(model, lr=1e-3, param_groups=other)
    other = [dict(g) for g in groups]
    other[0]['eps'] = 1e-6
    with pytest.raises(ValueError):
        FusedAdamW(model, lr=1e-3, param_groups=other)
    with pytest.raises(ValueError):
        group_names(model, [{'params': [torch.nn.Parameter(torch.zeros(3))]}])


def test_fused_adamw_groups_default_lr_and_schedule():
    model = models()[0]
    opt = FusedAdamW(model, lr=2e-3, param_groups=param_groups_lrd(model, layer_decay=0.5))
    assert [g['lr'] for g in opt.param_groups] == pytest.approx([2e-3 * g['lr_scale'] for g in opt.param_groups])
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda s: 0.5)
    assert [g['lr'] for g in opt.param_groups] == pytest.approx([1e-3 * g['lr_scale'] for g in opt.param_groups])
    sd = opt.state_dict()
    opt2 = FusedAdamW(model, lr=2e-3, param_groups=param_groups_lrd(model, layer_decay=0.5))
    opt2.load_state_dict(sd)
    assert [(g['lr'], g['lr_scale'], g['weight_decay']) for g in opt2.param_groups] == \
        [(g['lr'], g['lr_scale'], g['weight_decay']) for g in opt.param_groups]
    del sched


def test_trainer_group_state_round_trip_and_mismatch():
    model = models()[0]
    tr = FusedTrainer(model, param_groups=param_groups_lrd(model))
    state = tr._groups_state()
    assert len(state) == len(param_groups_lrd(model)) and all(isinstance(n, tuple) for n, _, _ in state)
    plain = FusedTrainer(model)
    assert plain.param_groups is None
    with pytest.raises(ValueError):   # betas that differ from the trainer's
        FusedTrainer(model, param_groups=[dict(g, betas=(0.8, 0.9)) for g in param_groups_lrd(model)])
