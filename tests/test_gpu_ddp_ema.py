"""GPU tier (needs >= 2 GPUs, skipped otherwise): the weight moving average under data parallelism -- bit-identical on
every rank, equal to the single-GPU run on the union batch."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

from conftest import ROOT


@pytest.mark.parametrize('mode', ['eager', 'graph'])
def test_two_rank_ema_is_identical_and_equals_union_batch(mode):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node=2', '--master-addr', '127.0.0.1',
           '--master-port', '29641', os.path.join(ROOT, 'tests', 'ddp_ema_worker.py'), mode]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and 'ddp ema ok' in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
