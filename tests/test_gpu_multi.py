"""Multi-GPU parity (-m gpu): launches tests/multi_gpu_worker.py under torchrun and requires every sharded mode — peer-store
gather, the pipelined frame ring, sharded views — to equal the single-GPU frame bit for bit (SURVEY.md §8(e): the result must not
depend on the partition). One rank per device with 2 and 4 devices (skipped with fewer); and two ranks sharing one device, which
runs the same multi-rank paths — IPC mappings, peer stores, ring flags between processes — on a machine with a single GPU."""
from __future__ import annotations

import os
import subprocess
import sys

import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def _device_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.parametrize("ranks", [2, 4])
def test_sharded_modes_equal_single_gpu(ranks):
    if _device_count() < ranks:
        pytest.skip(f"needs {ranks} CUDA devices")
    _run_worker(ranks, 29600 + ranks)


def test_sharded_modes_equal_single_gpu_two_ranks_on_one_device():
    if _device_count() < 1:
        pytest.skip("needs a CUDA device")
    _run_worker(2, 29610, {"CUDA_VISIBLE_DEVICES": os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]})


def _run_worker(ranks, port, env=None):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={ranks}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "multi_gpu_worker.py")]
    p = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900, env={**os.environ, **(env or {})})
    assert p.returncode == 0 and "MULTI-GPU CHECK PASSED" in p.stdout, p.stdout[-4000:]
