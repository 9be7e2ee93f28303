"""Multi-GPU correctness on real devices (skipped below two GPUs): the NCCL-broadcast cloud key must produce
bit-exact gates on ranks other than the one that generated it.  Reference model: examples/multi_gpu.py:86-104."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_rank1_gates_with_the_broadcast_key_equal_the_oracle():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip('needs two GPUs')
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
           '127.0.0.1', '--master-port', str(port), os.path.join(ROOT, 'tests', 'multi_gpu_worker.py')]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out[-3000:]
    assert 'rank 0 parity ok' in out and 'rank 1 parity ok' in out, out[-3000:]
    assert 'ranks ok: [1, 1]' in out, out[-3000:]
