"""-m gpu: the spatial "max" contrastive loss sharded over a real NCCL process group equals the single-GPU result
(op level and the whole model step, both precision modes, a different utterance length on every rank).  Launches
tools/sharded_spatial_check.py under torchrun; world 1 runs on a one-GPU box and covers the model wiring."""
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
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_sharded_spatial_max_equals_single_gpu(world):
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tools", "sharded_spatial_check.py"), "48"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert res.returncode == 0 and "SHARDED_SPATIAL_OK" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]
