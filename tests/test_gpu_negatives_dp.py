"""Pool negatives under data parallelism on real GPUs: launches tests/negatives_dp_check.py under torchrun when the box shows >= 2
GPUs (N ranks with synchronised BatchNorm draw and train as one process on N * B impressions).  Skipped on a 1-GPU box; the row
offset a rank draws with is checked on one GPU in tests/test_gpu_negatives.py."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def test_n_ranks_draw_and_train_as_one_process_on_the_whole_batch():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip('needs >= 2 GPUs')
    world = 2 if n < 4 else 4
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', f'--nproc-per-node={world}', '--master-addr', '127.0.0.1',
           '--master-port', str(_free_port()), os.path.join(ROOT, 'tests', 'negatives_dp_check.py')]
    out = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert out.returncode == 0 and '-> OK' in out.stdout, (out.stdout[-3000:], out.stderr[-3000:])
