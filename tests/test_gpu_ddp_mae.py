"""GPU tier: data-parallel MAE-style pre-training == the oracle's step on the union batch with the masks every rank drew
(guards the gradient-bucket placement of the decoder and recon head, and the per-rank mask seeds).  With two
GPUs: NCCL, eager and graph-captured.  With one: both ranks share it and exchange through gloo (eager only: gloo
collectives cannot be captured)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

from conftest import ROOT


@pytest.mark.parametrize('mode', ['eager', 'graph'])
def test_two_rank_mae_step_equals_union_batch(mode):
    shared = torch.cuda.device_count() < 2
    if shared and mode == 'graph':
        pytest.skip('graph-captured collectives need NCCL, i.e. 2 GPUs')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node=2', '--master-addr', '127.0.0.1',
           '--master-port', '29649', os.path.join(ROOT, 'tests', 'ddp_mae_worker.py'), mode,
           'shared' if shared else 'own']
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and 'ddp mae ok' in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
