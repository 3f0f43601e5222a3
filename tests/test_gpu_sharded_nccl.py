"""Memory-sharded kNN-SV with the CUDA kernel and a real NCCL all-gather (world size 2), against the unsharded
kernel on rank 0.  Needs two GPUs on the box; the CPU / gloo twin is tests/test_sharded_gloo.py."""
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.gpu
@pytest.mark.parametrize('rows,cand,dim', [(5001, 160, 160), (20000, 1000, 512)])
def test_sharded_knn_sv_nccl_world2(rows, cand, dim):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    env = dict(os.environ, SWEEP_ROWS=str(rows), SWEEP_CAND=str(cand), SWEEP_DIM=str(dim))
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
           '--master-port', str(_free_port()), os.path.join(ROOT, 'tools', 'sharded_sweep.py')]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith('{')][-1])
    assert line['ok'] and line['n_gpus'] == 2, line
    assert line['max_abs_err_vs_unsharded'] < 2e-4
    assert line['top100_identical_fraction'] >= 0.98
