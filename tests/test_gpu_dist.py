"""-m gpu, needs >= 2 visible GPUs (skipped otherwise): frame-sharded data parallelism with the SHARDED FlatAdam over NCCL
equals a single process that averages the cameras' gradients itself (tests/dist_check_sharded.py, launched with torchrun)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_flat_adam_over_nccl_matches_single_process():
    env = dict(os.environ, OMP_NUM_THREADS="4")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29577", os.path.join(ROOT, "tests", "dist_check_sharded.py")],
                       capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert r.returncode == 0 and "DIST_CHECK_OK" in r.stdout, (r.stdout[-1500:], r.stderr[-3000:])
