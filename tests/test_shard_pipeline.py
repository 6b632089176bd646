"""Runs tests/shard_pipeline_check.py under torchrun on 2 GPUs when the box has them."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
@pytest.mark.parametrize("exchange", ["p2p", "nccl"])
def test_two_gpu_rows_pipeline_after_the_fit(exchange, tmp_path):
    """Build, fit, contributors, reduce, refine, assign and save on row shards equal the
    same chain on one GPU; column sums by peer stores (default) or ncclAllReduce
    (MXB_NO_P2P=1)."""
    from mixemt_b200 import _lib
    if _lib.lib.mxb_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ)
    if exchange == "nccl":
        env["MXB_NO_P2P"] = "1"
    else:
        env.pop("MXB_NO_P2P", None)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29527" if exchange == "p2p" else "29528",
           os.path.join(ROOT, "tests", "shard_pipeline_check.py"), str(tmp_path)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert res.returncode == 0 and "SHARD_PIPELINE_OK" in res.stdout, \
        res.stdout[-2000:] + res.stderr[-4000:]
    assert ("exchange=%s" % exchange) in res.stdout, res.stdout[-2000:]
