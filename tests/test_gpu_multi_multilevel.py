"""Multi-GPU multilevel PARSDMM on z-slabs (3 levels, coarsening 2): device warm starts across slab boundaries
against the host warm starts (bit for bit) and against the CPU oracle.  Needs >= 2 GPUs on the box; skipped otherwise."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ngpu():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.parametrize("nproc", [2, 4])
def test_multilevel_slabs(nproc):
    if _ngpu() < nproc:
        pytest.skip("needs %d GPUs" % nproc)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc),
           "--master-addr", "127.0.0.1", "--master-port", str(29520 + nproc),
           os.path.join(ROOT, "tests", "mgpu_multilevel_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    sys.stdout.write(res.stdout[-6000:])
    sys.stderr.write(res.stderr[-4000:])
    assert res.returncode == 0
