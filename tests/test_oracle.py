"""CPU tier: pins the travelling oracle against the committed golden vectors, which the reference's own wrapper,
transform classes and metrics produced (tests/golden/make_golden*.py)."""
import os

import numpy as np
import pytest
import torch
from torch import nn

from conftest import GOLDEN_CFG, golden_sample
from oracle.ecg_vit_oracle import OracleConfig, OracleEcgVit, OracleTrainer, NAMED_SIZES, lr_lambda, patch_matrix


def _load_state(model, golden, prefix):
    sd = {k[len(prefix):]: torch.from_numpy(v) for k, v in golden.items() if k.startswith(prefix)}
    model.load_state_dict(sd, strict=True)


def test_oracle_reproduces_golden_forward_backward(golden):
    m = OracleEcgVit(config=OracleConfig(**GOLDEN_CFG))
    _load_state(m, golden, 'init/')
    m.train()
    x, y = torch.from_numpy(golden['x']), torch.from_numpy(golden['y'])
    out = m(sample_values=x, labels=y)
    out.loss.backward()
    np.testing.assert_allclose(out.logits.detach().numpy(), golden['logits'], rtol=0, atol=1e-6)
    assert abs(out.loss.item() - float(golden['loss'])) < 1e-6
    for k, p in m.named_parameters():
        np.testing.assert_allclose(golden_sample(p.grad.numpy()), golden['grad/' + k], rtol=0, atol=1e-7)


@pytest.fixture
def golden_threads():
    """CPU reductions round according to how they are split over threads.  Where a weight's gradient cancels to the size
    of AdamW's eps (1e-8), that rounding reaches its update: one patch-embedding weight moves by 1.6e-7 after three
    steps with 1, 4 or 16 intra-op threads.  With 8 threads the oracle reproduces the golden vectors bit for bit, also
    on machines with fewer or more cores.  The split is one input of the rounding; the CPU's vector width is another:
    the vectors reproduce on AVX-512 CPUs, and a CPU with another vector width may still differ in the last bits."""
    threads = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(threads)


def test_oracle_reproduces_golden_three_steps(golden, golden_threads):
    m = OracleEcgVit(config=OracleConfig(**GOLDEN_CFG))
    _load_state(m, golden, 'init/')
    m.train()
    x, y = torch.from_numpy(golden['x']), torch.from_numpy(golden['y'])
    tr = OracleTrainer(m, learning_rate=3e-4, weight_decay=1e-2, schedule='constant', n_warmup=0)
    for step in (1, 2, 3):
        loss, _, norm = tr.step(x, y)
        assert abs(float(loss) - float(golden[f'loss{step}'])) < 1e-6
        assert abs(float(norm) - float(golden[f'norm{step}'])) < 1e-6
        if step in (1, 3):
            for k, v in m.state_dict().items():
                got = golden_sample(v.numpy()) if step == 1 else v.numpy()
                np.testing.assert_allclose(got, golden[f'step{step}/' + k], rtol=0, atol=1e-7)


def test_oracle_eval_loss_none(golden):
    m = OracleEcgVit(config=OracleConfig(**GOLDEN_CFG), loss_reduction='none')
    _load_state(m, golden, 'step3/')
    m.eval()
    with torch.no_grad():
        out = m(torch.from_numpy(golden['x']), torch.from_numpy(golden['y']))
    np.testing.assert_allclose(out.loss.numpy(), golden['eval_loss_none'], rtol=0, atol=1e-6)


def test_patch_matrix_matches_golden_index(golden):
    idx = torch.arange(2 * 12 * 500, dtype=torch.float32).reshape(2, 12, 500)
    assert np.array_equal(patch_matrix(idx, 50).numpy().astype(np.int32), golden['patch_index'])
    # closed form: A[b*n+w, t*C+c] = x[b, c, w*P+t]
    b, w, t, c = 1, 7, 13, 5
    assert golden['patch_index'][b * 10 + w, t * 12 + c] == (b * 12 + c) * 500 + w * 50 + t


def test_named_sizes_and_param_counts():
    # SURVEY.md 8a-S cross-checks: cfg1 3 341 895 params / 52 tensors; base (2500/50) 85 584 455 / 140
    c = OracleConfig(max_signal_length=2500, patch_size=50, hidden_size=256, num_hidden_layers=4,
                     num_attention_heads=8, intermediate_size=1024)
    m = OracleEcgVit(config=c)
    assert sum(p.numel() for p in m.parameters()) == 3_341_895 and len(list(m.parameters())) == 52
    assert NAMED_SIZES['base'] == (768, 12, 12, 3072)


def test_lr_lambda_matches_transformers():
    from transformers import get_constant_schedule_with_warmup, get_cosine_schedule_with_warmup
    p = nn.Parameter(torch.zeros(1))
    for name, mk in (('constant', lambda o: get_constant_schedule_with_warmup(o, num_warmup_steps=5)),
                     ('cosine', lambda o: get_cosine_schedule_with_warmup(o, num_warmup_steps=5, num_training_steps=40))):
        opt = torch.optim.AdamW([p], lr=1.0)
        sch = mk(opt)
        for s in range(45):
            assert abs(opt.param_groups[0]['lr'] - lr_lambda(name, s, 5, 40)) < 1e-12
            opt.step()
            sch.step()


def test_oracle_matches_reference_wrapper(golden, golden_threads):
    """The restated wrapper == the reference's verbatim `EcgVit`, bit for bit, through what that wrapper stored in the
    golden vectors (tests/golden/make_golden.py): its state_dict keys in its order, its initial weights from the same
    seed (parameter creation order and initialisers), and its logits, loss and gradients on those weights and inputs."""
    torch.manual_seed(77)
    ours = OracleEcgVit(config=OracleConfig(**GOLDEN_CFG))
    ref_init = {k[len('init/'):]: v for k, v in golden.items() if k.startswith('init/')}
    assert list(ours.state_dict().keys()) == list(ref_init.keys())
    for k, v in ours.state_dict().items():
        assert np.array_equal(v.numpy(), ref_init[k]), k
    ours.train()
    out = ours(sample_values=torch.from_numpy(golden['x']), labels=torch.from_numpy(golden['y']))
    assert np.array_equal(out.logits.detach().numpy(), golden['logits']) and out.loss.item() == float(golden['loss'])
    out.loss.backward()
    assert [k for k, _ in ours.named_parameters()] == [k[len('grad/'):] for k in golden if k.startswith('grad/')]
    for k, p in ours.named_parameters():
        assert np.array_equal(golden_sample(p.grad.numpy()), golden['grad/' + k]), k


# ---- input transforms (SURVEY 8f rank 1): oracle/transforms.py pinned by vectors the reference's own classes produced
@pytest.fixture(scope='module')
def transform_golden():
    return np.load(os.path.join(os.path.dirname(__file__), 'golden', 'input_transform.npz'))


@pytest.mark.parametrize('case', ['ragged', 'full_block', 'long'])
def test_transform_oracle_matches_reference_vectors(transform_golden, case):
    from oracle import transforms
    g = transform_golden
    rec, k = g[f'{case}/records'], int(g[f'{case}/k'])
    got_eval = transforms.pipeline(rec, g['mean'], g['std'], pad=k)
    got_train = transforms.pipeline(rec, g['mean'], g['std'], pad=k, spans=g[f'{case}/spans'])
    assert got_eval.dtype == np.float32
    assert np.array_equal(got_eval, g[f'{case}/eval'])      # bit-exact
    assert np.array_equal(got_train, g[f'{case}/train'])    # masking bit-exact
    if case == 'full_block':
        assert got_eval.shape[-1] == rec.shape[-1] + k      # TimeEndPad pads a whole block when L % k == 0


@pytest.mark.parametrize('case', ['ragged', 'full_block', 'long'])
def test_transform_oracle_draws_time_out_like_reference_classes(transform_golden, case):
    """The reference's `TimeOut` draws its span from torch's global RNG, one record after another, and the golden
    `train` output is what its classes produced after torch.manual_seed(1234) (tests/golden/make_golden_transform.py).
    `draw_time_out_span` must consume the RNG the same way: the same seed gives the same masked output, bit for bit."""
    from oracle import transforms
    g = transform_golden
    rec, k = g[f'{case}/records'], int(g[f'{case}/k'])
    torch.manual_seed(1234)
    spans = [transforms.draw_time_out_span(g[f'{case}/eval'].shape[-1]) for _ in range(rec.shape[0])]
    assert np.array_equal(transforms.pipeline(rec, g['mean'], g['std'], pad=k, spans=spans), g[f'{case}/train'])


# ---- evaluation metrics (SURVEY 8f rank 2): oracle/metrics.py pinned by the reference's own get_accuracy outputs
@pytest.mark.parametrize('case', ['sparse', 'ties', 'tiny'])
def test_metrics_oracle_matches_reference_vectors(case):
    from oracle import metrics
    g = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'eval_metrics.npz'))
    scalars, per_class = metrics.get_accuracy(g[f'{case}/preds'], g[f'{case}/labels'])
    assert np.allclose(scalars, g[f'{case}/scalars'], rtol=1e-12, atol=0)
    want = g[f'{case}/per_class_auc']
    assert np.array_equal(np.isnan(per_class), np.isnan(want))
    assert np.allclose(per_class[~np.isnan(want)], want[~np.isnan(want)], rtol=1e-12, atol=0)
    assert np.isnan(per_class[5]) and np.isnan(per_class[9])      # single-label classes are filtered (util/train.py:29)


def test_oracle_fp64_tie_breaker(golden):
    """SURVEY 8c: an fp64 run of the oracle is the referee when fp32 CPU and fp32 GPU disagree near 1e-5.  It also
    measures the fp32 noise floor of the golden vectors themselves: well below the 1e-5 bar the GPU tests apply."""
    m = OracleEcgVit(config=OracleConfig(**GOLDEN_CFG))
    _load_state(m, golden, 'init/')
    m = m.double().train()
    x, y = torch.from_numpy(golden['x']).double(), torch.from_numpy(golden['y']).double()
    out = m(sample_values=x, labels=y)
    out.loss.backward()
    want = torch.from_numpy(golden['logits']).double()
    rel = float((out.logits.detach() - want).norm() / want.norm())
    assert rel < 1e-6, rel
    assert abs(out.loss.item() - float(golden['loss'])) < 1e-6 * float(golden['loss'])
    worst = max(float((golden_sample(p.grad) - torch.from_numpy(golden['grad/' + k]).double()).norm() /
                      torch.from_numpy(golden['grad/' + k]).double().norm().clamp_min(1e-30))
                for k, p in m.named_parameters())
    assert worst < 1e-5, worst


@pytest.mark.parametrize('seed', range(6))
def test_metrics_oracle_matches_sklearn_on_random_cases(seed):
    """oracle/metrics.py against scikit-learn itself (the third-party code the reference calls, util/train.py:33-52) on
    random sizes, class balances and tie structures, with the reference's argument order for classification_report"""
    sk = pytest.importorskip('sklearn.metrics')
    from oracle import metrics
    rng = np.random.default_rng(seed)
    n, k = int(rng.integers(2, 400)), int(rng.integers(1, 12))
    quant = [None, 2, 8][seed % 3]
    logits = rng.standard_normal((n, k)) * 2
    if quant:
        logits = np.round(logits * quant) / quant
    preds = (1 / (1 + np.exp(-logits))).astype(np.float32)
    labels = (rng.random((n, k)) < rng.uniform(0.05, 0.6)).astype(np.float32)
    scalars, per_class = metrics.get_accuracy(preds, labels)
    two = np.any(labels != labels[0], axis=0)
    for c in range(k):
        if two[c]:
            assert abs(per_class[c] - sk.roc_auc_score(labels[:, c], preds[:, c])) < 1e-12
        else:
            assert np.isnan(per_class[c])
    pb, y = (preds >= 0.5).astype(np.float32).flatten(), labels.flatten()
    assert abs(scalars[0] - sk.accuracy_score(y, pb)) < 1e-12
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        assert abs(scalars[1] - sk.balanced_accuracy_score(y, pb)) < 1e-12
        rep = sk.classification_report(pb, y, labels=[0, 1], target_names=['neg', 'pos'], output_dict=True,
                                       zero_division=0)
    rec_pos, rec_neg = [rep[t]['recall'] for t in ['neg', 'pos']]            # util/train.py:50, names as swapped there
    assert abs(scalars[2] - rec_neg) < 1e-12 and abs(scalars[3] - rec_pos) < 1e-12


@pytest.mark.parametrize('seed', range(4))
def test_transform_oracle_random_shapes_against_numpy_semantics(seed):
    """TimeEndPad's length rule and TimeOut's span on random lengths; Normalize in fp32 like numpy broadcasting"""
    from oracle import transforms
    rng = np.random.default_rng(100 + seed)
    C, L, k = int(rng.integers(1, 13)), int(rng.integers(10, 700)), int(rng.integers(2, 90))
    rec = rng.standard_normal((2, C, L)).astype(np.float32)
    mean, std = rng.standard_normal(C), rng.random(C) + 0.1
    Lp = L + (k - L % k)
    spans = [(int(rng.integers(0, Lp // 2)), int(rng.integers(0, Lp // 2))) for _ in range(2)]
    out = transforms.pipeline(rec, mean, std, pad=k, spans=spans)
    assert out.shape == (2, C, Lp) and out.dtype == np.float32 and Lp % k == 0 and Lp > L
    want = (rec - mean.astype(np.float32)[None, :, None]) / std.astype(np.float32)[None, :, None]
    for b, (s, l) in enumerate(spans):
        keep = np.ones(Lp, bool)
        keep[s:s + l] = False
        assert np.array_equal(out[b][:, :L][:, keep[:L]], want[b][:, keep[:L]])
        assert not out[b][:, ~keep].any() and not out[b][:, L:].any()


def test_restated_blocks_match_an_independent_vit_implementation():
    """`oracle/vit_restated.py` cannot be pinned against vit-pytorch itself (absent, not installable offline).  Its block
    arithmetic -- pre-norm residual blocks, multi-head softmax attention scaled by dim_head^-0.5, exact-erf GELU MLP,
    LayerNorm eps 1e-5 -- is checked here against an independent implementation of the same published block
    (Hugging Face `ViTEncoder`, bias-free q/k/v) with the weights mapped across.  What stays pinned only by the
    reference's call sites and state_dict keys is vit-pytorch's wiring around the blocks (packed to_qkv, dropout
    placement, CLS / pos assembly, LayerNorm inside mlp_head)."""
    tv = pytest.importorskip('transformers.models.vit.modeling_vit')
    from transformers import ViTConfig
    from oracle.vit_restated import Transformer
    torch.manual_seed(3)
    dim, depth, heads, dh, mlp = 96, 3, 4, 24, 160
    ours = Transformer(dim, depth, heads, dh, mlp, dropout=0.0).eval()
    cfg = ViTConfig(hidden_size=dim, num_hidden_layers=depth, num_attention_heads=heads, intermediate_size=mlp,
                    qkv_bias=False, layer_norm_eps=1e-5, hidden_act='gelu', hidden_dropout_prob=0.0,
                    attention_probs_dropout_prob=0.0)
    cfg._attn_implementation = 'eager'
    theirs = tv.ViTEncoder(cfg).eval()
    with torch.no_grad():
        for (attn, ff), layer in zip(ours.layers, theirs.layer):
            q, k, v = attn.fn.to_qkv.weight.chunk(3, dim=0)
            layer.attention.attention.query.weight.copy_(q)
            layer.attention.attention.key.weight.copy_(k)
            layer.attention.attention.value.weight.copy_(v)
            layer.attention.output.dense.weight.copy_(attn.fn.to_out[0].weight)
            layer.attention.output.dense.bias.copy_(attn.fn.to_out[0].bias)
            layer.layernorm_before.weight.copy_(attn.norm.weight.uniform_(0.5, 1.5))
            layer.layernorm_before.bias.copy_(attn.norm.bias.uniform_(-0.2, 0.2))
            layer.layernorm_after.weight.copy_(ff.norm.weight.uniform_(0.5, 1.5))
            layer.layernorm_after.bias.copy_(ff.norm.bias.uniform_(-0.2, 0.2))
            layer.intermediate.dense.weight.copy_(ff.fn.net[0].weight)
            layer.intermediate.dense.bias.copy_(ff.fn.net[0].bias)
            layer.output.dense.weight.copy_(ff.fn.net[3].weight)
            layer.output.dense.bias.copy_(ff.fn.net[3].bias)
        x = torch.randn(2, 17, dim)
        got = ours(x)
        want = theirs(x)
        want = want.last_hidden_state if hasattr(want, 'last_hidden_state') else want[0]
    assert float((got - want).abs().max()) < 2e-5 * float(want.abs().max())
