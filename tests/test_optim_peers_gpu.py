"""The optimiser's peer-exchange forms (rlppo_norm_clip_adam_peers, _peers2) at 1, 2, 3 and min(GPUs, 8) ranks:
tests/optim_peers_check.py under torch.distributed.run --standalone.  One rank runs the peer code paths with nothing to
exchange; the rank-order sum and the two-shot slices need two ranks or more."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("world", [1, 2, 3, "all"])
def test_optimiser_peer_forms(world):
    n = min(torch.cuda.device_count(), 8)
    if world == "all":
        if n <= 3:
            pytest.skip(f"{n} GPUs: covered by the 2- and 3-rank runs")
        world = n
    if n < world:
        pytest.skip(f"needs {world} GPUs, the box has {n}")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc-per-node={world}",
           os.path.join(ROOT, "tests", "optim_peers_check.py")]
    # generous: a peer that never arrives traps the kernel after about two minutes
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0 and f"optim_peers_check OK world={world}" in out.stdout, \
        out.stdout[-4000:] + out.stderr[-4000:]
    print(out.stdout[-300:])
