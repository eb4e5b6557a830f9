import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a B200 (sm_100a) GPU; run with -m gpu on the GPU box')


@pytest.fixture(scope='session')
def golden():
    import numpy as np
    path = os.path.join(ROOT, 'tests', 'golden', 'ecgvit_small_step.npz')
    return dict(np.load(path))


def golden_sample(a):
    """The elements of a gradient (grad/) or step-1 weight (step1/) tensor that tests/golden/ecgvit_small_step.npz keeps:
    every 31st element of the flattened tensor (a prime stride, so every row and column of a 64-wide matrix is hit),
    or all of it up to 1024 elements.  Works on numpy arrays and torch tensors alike."""
    flat = a.reshape(-1)
    return flat[::31] if flat.shape[0] > 1024 else flat


GOLDEN_CFG = dict(max_signal_length=500, patch_size=50, num_channels=12, hidden_size=64, num_hidden_layers=2,
                  num_attention_heads=4, intermediate_size=128, hidden_dropout_prob=0.0,
                  attention_probs_dropout_prob=0.0)
