"""GPU (needs >= 2 devices, otherwise skipped): the NCCL utterance-sharded SIF path equals the
single-GPU path.  One process per GPU via torchrun, rendezvous on 127.0.0.1."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sharded_equals_single_gpu():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip('needs >= 2 GPUs')
    world = 2 if n < 4 else 4
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(world),
           '--master-addr', '127.0.0.1', '--master-port', '29541', os.path.join(ROOT, 'tools', 'dist_check.py')]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    sys.stdout.write(r.stdout[-4000:])
    sys.stderr.write(r.stderr[-4000:])
    assert r.returncode == 0


def test_data_parallel_mmb_step_reproduces_reference_loop():
    """SURVEY.md 8e "MMB training": utterances sharded over 2 ranks, head gradients summed over NVLink peer
    memory, global-batch mean and BatchNorm statistics -- the reference loop's goldens (tools/dp_check.py)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs >= 2 GPUs')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
           '--master-addr', '127.0.0.1', '--master-port', '29543', os.path.join(ROOT, 'tools', 'dp_check.py')]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    sys.stdout.write(r.stdout[-4000:])
    sys.stderr.write(r.stderr[-6000:])
    assert r.returncode == 0
