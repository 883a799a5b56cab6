"""Multi-GPU parity in the driver-run suite (pytest -m gpu): spawns one process per GPU with torchrun when the box has at
least two devices (skipped, with the reason, on a single-GPU box).  The worker compares the peer-memory multi-GPU engine
with the single-GPU engine: forces bit-equal, energies, a Langevin trajectory, identical state on every rank."""
import os
import subprocess
import sys
import pytest
from conftest import ROOT

pytestmark = pytest.mark.gpu


def _ngpu():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.parametrize("world,name", [(2, "water"), (2, "dhfr"), (4, "dhfr"), (8, "apoa1")])
def test_multi_gpu_engine_equals_single_gpu_engine(world, name):
    n = _ngpu()
    if n < world:
        pytest.skip("needs %d GPUs on one box, this one has %d (run python -m pytest tests/test_gpu_multi.py -m gpu on a box with %d)" % (world, n, world))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(29400 + world), os.path.join(ROOT, "tests", "multi_rank_worker.py"), name, "40"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0 and "MULTI_OK" in r.stdout, (r.stdout[-3000:], r.stderr[-3000:])
