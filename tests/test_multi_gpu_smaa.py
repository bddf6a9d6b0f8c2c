"""SMAA in row-sharded frames on real GPUs against the single-GPU viewer, with both exchange paths of the edges:
peer-memory stores from the edge kernel (default) and NCCL broadcasts."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AA_SMAA_HIGH, AA_SMAA_ULTRA = 5, 6


def _gpu_count():
    import torch

    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.parametrize("exchange", ["peer", "nccl"])
@pytest.mark.parametrize("post_aa", [AA_SMAA_HIGH, AA_SMAA_ULTRA], ids=["smaa_high", "smaa_ultra"])
@pytest.mark.parametrize("world", [2, 4])
def test_sharded_smaa_frames_are_bit_identical(cuda, world, post_aa, exchange):
    n = _gpu_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs on the box")
    if n < world:
        pytest.skip(f"needs {world} GPUs on the box")
    port = 29631 + 4 * (world == 4) + 2 * (post_aa == AA_SMAA_ULTRA) + (exchange == "nccl")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "multi_gpu_smaa_worker.py"), "1280", "768", "300", str(post_aa)]
    env = dict(os.environ, GRB_SHARD_EXCHANGE=exchange)
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    sys.stdout.write(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "grb_smaa" not in r.stderr and "smaa-" not in r.stderr, r.stderr[-3000:]
    if exchange == "peer":
        assert "peer-memory exchange unavailable" not in r.stderr, "the box has NVLink peers: the peer path must be the one that ran"
