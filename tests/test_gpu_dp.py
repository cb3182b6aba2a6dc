"""Native data-parallel engines on real GPUs (needs >= 2): every engine -- torch.distributed collectives, NCCL inside the library
(replicated and ZeRO-1 sharded optimizer), and the peer-memory engine (one reduce + Adam + publish kernel between two NVLink flag
barriers, multimem.ld_reduce / multimem.st where the fabric has NVLS) -- keeps the replicas bit-identical and reproduces the
single-GPU training trajectory. The ranks are spawned by scripts/dp_parity.py (the driver's single-GPU test run skips this)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_data_parallel_engines_match_single_gpu(torch_cuda):
    torch = torch_cuda
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "dp_parity.py")], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "DP PARITY OK" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
