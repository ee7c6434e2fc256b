"""Tensor-parallel single-sample forward (BASELINE config 4) on >= 2 GPUs: logits within the bf16 tolerance of the
single-GPU forward (fp32 partial sums are all-reduced before the single rounding), ranks stay in lock-step."""
import os
import subprocess
import sys

import pytest
import torch

from helpers import ROOT

pytestmark = pytest.mark.gpu


def test_tensor_parallel_matches_single_gpu():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    tp = 2
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={tp}", "--master-addr", "127.0.0.1",
           "--master-port", "29631", os.path.join(ROOT, "tests", "_tp_worker.py")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    print(p.stdout[-2000:])
    assert p.returncode == 0, p.stderr[-3000:]
    assert "TP_CHECK_OK" in p.stdout
