"""Runs tests/multirank_check.py under torchrun on 2, 4 and 8 GPUs when the box has them: the
row- and restart-sharded EM against long double, with the column sums exchanged by peer stores
inside the EM tail (default) and by NCCL (MXB_NO_P2P=1)."""
import os
import subprocess
import sys

import pytest

import multirank_check
from test_shard_consumers_gpu import free_port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
@pytest.mark.parametrize("exchange", ["p2p", "nccl"])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_em_matches_long_double(world, exchange, tmp_path):
    from mixemt_b200 import _lib
    if _lib.lib.mxb_device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    refs = str(tmp_path / "refs.npz")
    n_cases = multirank_check.write_references(world, refs)
    env = dict(os.environ)
    if exchange == "nccl":
        env["MXB_NO_P2P"] = "1"
    else:
        env.pop("MXB_NO_P2P", None)
    env.pop("MXB_EM_NO_PACK", None)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
           "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(free_port()), os.path.join(ROOT, "tests", "multirank_check.py"),
           refs]
    try:
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    finally:
        os.remove(refs)     # several hundred MB
    print(res.stdout)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-5000:]
    ok = "MULTIRANK_OK world=%d exchange=%s cases=%d" % (world, exchange, n_cases)
    assert ok in res.stdout, res.stdout[-3000:]
