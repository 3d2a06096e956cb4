"""GPU (needs >= 2 B200s on the box; skipped otherwise): DSGD over NCCL against the oracle."""
import os
import subprocess
import sys

import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def test_dsgd_two_ranks_parity(capi):
    if capi.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.join(ROOT, "tests", "dsgd_gpu_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "DSGD-CHECK OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
