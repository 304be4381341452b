"""Learner(data_parallel=True) end to end: tests/dp_learner_check.py under torch.distributed.run --standalone, at one rank
and, when the box has two GPUs, at two ranks (also with the NCCL gradient exchange, which carries the return statistics
with WelfordRunningStat.broadcast_ instead of a peer-memory read)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("world,collective", [(1, None), (2, None), (2, "nccl")])
def test_data_parallel_learner(tmp_path, world, collective):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    env = dict(os.environ)
    env.pop("RLPPO_DP_COLLECTIVE", None)
    if collective is not None:
        env["RLPPO_DP_COLLECTIVE"] = collective
    cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc-per-node={world}",
           os.path.join(ROOT, "tests", "dp_learner_check.py"), str(tmp_path)]
    out = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and f"dp_learner_check OK world={world}" in out.stdout, \
        out.stdout[-4000:] + out.stderr[-4000:]
    print(out.stdout[-500:])
