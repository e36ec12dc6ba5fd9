"""Document-sharded search on >= 2 GPUs (NCCL all-gather + on-device merge, shard.cuh)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("p2p", ["1", "0"])
def test_sharded_two_ranks(p2p):
    """p2p=1: the shard records travel by direct NVLink stores into IPC-mapped windows; p2p=0: by ncclAllGather."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    env = dict(os.environ, OC_SHARD_P2P=p2p)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29611" if p2p == "1" else "29612",
                        os.path.join(ROOT, "tests", "sharded_worker.py")], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0 and "SHARDED_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
