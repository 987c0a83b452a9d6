"""Multi-GPU parity (needs >= 2 B200s on the box): the particle-sharded scan with one ncclAllGather per iteration
must reproduce the single-GPU scan.  Spawns tests/mgpu_worker.py under torch.distributed.run."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sharded_equals_single_gpu():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 2 if n < 4 else 4
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", "29517", os.path.join(ROOT, "tests", "mgpu_worker.py")]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    sys.stdout.write(r.stdout[-4000:])
    sys.stderr.write(r.stderr[-4000:])
    assert r.returncode == 0


def test_sharded_with_the_debug_library():
    """The same worker against libsvnicp_b200_dbg.so: every wait of the peer exchange checks that no rank is more than one
    iteration ahead (SVN_CHECK 40) -- a sequence-number disagreement shows up as an error instead of as luck (DESIGN.md section 5)."""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    from svn_icp_b200 import build as b
    dbg = b.LIB.replace(".so", "_dbg.so")
    if not os.path.exists(dbg):
        dbg = b.build(debug_bounds=True)
    world = 2 if n < 4 else 4
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", "29521", os.path.join(ROOT, "tests", "mgpu_worker.py")]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900, env=dict(os.environ, SVNICP_B200_LIB=dbg))
    sys.stdout.write(r.stdout[-4000:])
    sys.stderr.write(r.stderr[-4000:])
    assert r.returncode == 0
