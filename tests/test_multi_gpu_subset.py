"""Multi-GPU parity of the keyframe database's keyframe selections (keyframes=): spawns tools/test_multi_gpu_subset.py under
torchrun on all visible GPUs (>= 2) and writes the script's log to the test's temporary directory.  The host logic is covered on CPU by
tests/test_keyframe_db_subset.py (gloo); this is the device side."""
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


def test_sharded_subset_parity_on_all_gpus(tmp_path):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    n = 8 if n >= 8 else 4 if n >= 4 else 2
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tools", "test_multi_gpu_subset.py")]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=1200)
    with open(tmp_path / f"multi_gpu_subset_n{n}.log", "w") as f:
        f.write(r.stdout + "\n--- stderr ---\n" + r.stderr[-4000:])
    assert r.returncode == 0 and f"MULTI_GPU_SUBSET OK world={n}" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
