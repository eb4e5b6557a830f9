"""CPU tier: frozen parameters (requires_grad=False) -- the trainable span every module reads, the gradient buckets over
it, the group map with the frozen tensors at 255, the graph key and the rejections (nothing to train, deferred
optimizer)."""
import pytest
import torch

from conftest import GOLDEN_CFG
from ecg_b200 import EcgVit, EcgVitConfig, EcgVitForMaskedAutoencoding, EcgVitForMaskedPatchModeling, FusedTrainer
from ecg_b200.optim import UNGROUPED, group_map
from ecg_b200.parallel import bucket_slices

MAE_DEC = dict(decoder_hidden_size=32, decoder_num_hidden_layers=2, decoder_num_attention_heads=2,
               decoder_intermediate_size=64)
CFG4 = dict(GOLDEN_CFG, num_hidden_layers=4)
EMBEDDING = ('vit.to_patch_embedding.', 'vit.pos_embedding', 'vit.cls_token', 'vit.mask_token')


def models(cfg=CFG4):
    c = EcgVitConfig(compute_dtype='fp32', **cfg)
    return [EcgVit(config=c), EcgVitForMaskedPatchModeling(c), EcgVitForMaskedAutoencoding(c, **MAE_DEC)]


def block_of(name):
    return int(name.split('.')[3]) if name.startswith('vit.transformer.layers.') else None


def freeze(model, pattern, k=2):
    """the freezing patterns of the tests; returns the expected lowest trainable position"""
    depth = model.config.num_hidden_layers
    for name, p in model.named_parameters():
        b = block_of(name)
        if pattern == 'head_only':
            frozen = name.startswith('vit.') and not name.startswith('vit.mlp_head.')
        elif pattern == 'last_k':        # blocks < k and the embedding
            frozen = name.startswith(EMBEDDING) or (b is not None and b < k)
        elif pattern == 'pos':
            frozen = name == 'vit.pos_embedding'
        elif pattern == 'qkv':
            frozen = name == 'vit.transformer.layers.1.0.fn.to_qkv.weight'
        elif pattern == 'all':
            frozen = True
        else:
            frozen = False
        p.requires_grad_(not frozen)
    return {'none': -1, 'head_only': depth, 'last_k': k, 'pos': -1, 'qkv': -1, 'all': None}[pattern]


@pytest.mark.parametrize('which', [0, 1, 2])
@pytest.mark.parametrize('pattern', ['none', 'head_only', 'last_k', 'pos', 'qkv', 'all'])
def test_trainable_span(which, pattern):
    model = models()[which]
    lowest = freeze(model, pattern)
    layout, total = model._flat_layout()
    span = model.trainable_span()
    assert span.lowest == lowest
    names = [(k, v) for k, v in layout.items()]
    trains = {v[3]: p.requires_grad for v, p in zip(layout.values(), model.parameters())}
    first = next((v[0] for k, v in names if trains[v[3]]), total)
    assert span.lo == first
    assert span.frozen == frozenset(k for k, v in names if not trains[v[3]])
    # a frozen tensor inside [lo, n) only where something is frozen above a trainable tensor: `pos` is the first tensor of
    # the flat buffers (a module's own parameters come before its children's), so freezing it leaves a frozen prefix
    assert span.frozen_inside == (pattern == 'qkv')
    if pattern == 'pos':
        assert span.lo == layout['cls'][0] > 0
    if pattern == 'none':
        assert span.lo == 0 and not span.frozen
    if pattern == 'last_k':
        assert span.lo == layout['l2.ln1.w'][0]
    if pattern == 'head_only':
        assert span.lo == min(v[0] for v in layout.values()
                              if not v[3].startswith('vit.') or v[3].startswith('vit.mlp_head.'))
    # the span follows the flags, and its key changes with them
    key = span.key
    next(model.parameters()).requires_grad_(not next(model.parameters()).requires_grad)
    assert model.trainable_span().key != key


@pytest.mark.parametrize('bucket_layers', [1, 3])
@pytest.mark.parametrize('which', [0, 1, 2])
@pytest.mark.parametrize('pattern', ['none', 'head_only', 'last_k', 'pos', 'qkv'])
def test_buckets_cover_the_span_with_visited_triggers(bucket_layers, which, pattern):
    model = models()[which]
    freeze(model, pattern, k=1)
    layout, total = model._flat_layout()
    depth = model.config.num_hidden_layers
    span = model.trainable_span()
    offs = [layout[f'l{l}.ln1.w'][0] for l in range(depth)]
    sl = bucket_slices(offs, total, depth, bucket_layers, span.lowest, span.lo)
    # contiguous, in backward order, covering exactly [lo, total)
    assert sl[0][2] == total and sl[-1][1] == span.lo
    for (_, lo_a, _), (_, _, hi_b) in zip(sl, sl[1:]):
        assert hi_b == lo_a
    embedding_trains = span.lowest == -1
    for t, lo, hi in sl:
        assert hi > lo
        assert t >= max(span.lowest, 0) or (t == -1 and embedding_trains), (t, span.lowest)
    if pattern == 'head_only':
        assert sl == [(depth, span.lo, total)]
    if pattern == 'none':
        assert sl == bucket_slices(offs, total, depth, bucket_layers)


def test_group_map_puts_frozen_tensors_at_255():
    model = models()[0]
    freeze(model, 'qkv')
    model._layout, total = model._flat_layout()
    model._flat_p = torch.zeros(total)
    names = [tuple(n for n, p in model.named_parameters() if p.requires_grad)]
    gm = group_map(model, names)
    for key, (o, n, _, name) in model._layout.items():
        ids = gm[o // 64:(o + n + 63) // 64]
        assert bool((ids == (UNGROUPED if key == 'l1.qkv.w' else 0)).all()), key


def _trainer(model, **kw):
    tr = FusedTrainer(model, **kw)
    model._layout, total = model._flat_layout()
    model._flat_p = torch.zeros(total)
    tr._flat_ptr = model._flat_p.data_ptr()
    return tr


@pytest.mark.parametrize('pattern', ['none', 'head_only', 'pos', 'qkv'])
def test_plan_selects_the_kernels(pattern):
    model = models()[0]
    freeze(model, pattern)
    tr = _trainer(model)
    tr._plan()
    assert tr._span.lo == model.trainable_span().lo
    assert tr._grouped == (pattern == 'qkv')
    if tr._grouped:
        frozen = model.trainable_span().frozen
        for key, (o, n, _, _) in model._layout.items():
            assert int(tr._gmap[o // 64]) == (UNGROUPED if key in frozen else 0)
        assert len(tr._hyper_values(1)) == 18   # hyper block + one group (the trainer's lr / weight decay)
    else:
        assert len(tr._hyper_values(1)) == 16


def test_nothing_to_train_raises():
    model = models()[0]
    freeze(model, 'all')
    with pytest.raises(ValueError, match='nothing to train'):
        _trainer(model)._plan()


def test_defer_optimizer_with_a_frozen_tensor_raises():
    model = models()[0]
    freeze(model, 'head_only')
    with pytest.raises(ValueError, match='defer_optimizer'):
        _trainer(model, defer_optimizer=True)._plan()
    freeze(model, 'none')
    _trainer(model, defer_optimizer=True)._plan()


def test_graph_key_follows_the_flags():
    """the trainer's CUDA-graph key holds the span's flag key: flipping a flag (gradual unfreezing) changes it"""
    model = models()[0]
    freeze(model, 'head_only')
    k1 = model.trainable_span().key
    model.vit.transformer.layers[3][0].norm.weight.requires_grad_(True)
    k2 = model.trainable_span().key
    assert k1 != k2 and model.trainable_span().lowest == 3
    import inspect
    assert 'self._span.key' in inspect.getsource(FusedTrainer._graph_step)
