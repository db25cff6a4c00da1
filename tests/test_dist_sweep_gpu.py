"""GPU (needs >= 2 devices, otherwise skipped): the utterance-sharded SIF sweep (tools/sif_sweep_dist_check.py)
at 2 and 4 ranks, and 8 where the box has them.  One process per GPU via torchrun, rendezvous on 127.0.0.1."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize('world', [2, 4, 8])
def test_sharded_sweep_equals_sharded_path_and_single_gpu(world):
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip('needs >= 2 GPUs')
    if world > n:
        pytest.skip('needs %d GPUs' % world)
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(world),
           '--master-addr', '127.0.0.1', '--master-port', '29547', os.path.join(ROOT, 'tools', 'sif_sweep_dist_check.py')]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    sys.stdout.write(r.stdout[-6000:])
    sys.stderr.write(r.stderr[-4000:])
    assert r.returncode == 0
