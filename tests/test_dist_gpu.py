"""GPU (needs >= 2 GPUs, else skipped): genome-sharded query/profile over NCCL == single-GPU result."""
import os
import subprocess
import sys

import pytest

from tests.util import REPO

pytestmark = pytest.mark.gpu


def test_sharded_equals_single_gpu(tmp_path):
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29517", os.path.join(REPO, "scripts", "dist_check.py")]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    (tmp_path / "dist_check_2gpu.log").write_text(r.stdout)   # the whole log, kept with pytest's temporary files
    assert r.returncode == 0, r.stdout[-3000:]
    assert "sharded(2 ranks)" in r.stdout and "equal=True" in r.stdout and "equal=False" not in r.stdout
