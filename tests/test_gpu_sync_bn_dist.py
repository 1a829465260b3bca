"""Synchronised BatchNorm on two GPUs (skipped with fewer): two ranks x b images with --sync-bn against the CPU oracle at
the unsharded global batch; see tests/sync_bn_dist_worker.py.  The control run trains without --sync-bn and must miss
that oracle on the BatchNorm running statistics."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize('precision,mode,extra', [('fp32', 'eager', ''), ('fp32', 'graph', ''), ('bf16', 'graph', ''),
                                                  ('fp32', 'eager', 'control')])
def test_world2_sync_bn_matches_global_batch_oracle(precision, mode, extra):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    port = 29300 + (os.getpid() + hash((precision, mode, extra))) % 300
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
           '127.0.0.1', '--master-port', str(port), os.path.join(ROOT, 'tests', 'sync_bn_dist_worker.py'), precision,
           mode] + ([extra] if extra else [])
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT)
    sys.stdout.write(r.stdout[-4000:])
    assert r.returncode == 0, r.stderr[-4000:]
    assert 'SYNC_BN_OK' in r.stdout, r.stdout[-4000:]
