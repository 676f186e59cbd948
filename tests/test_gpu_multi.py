"""Two-rank run on two GPUs (NCCL halo exchange inside libpamg_cuda) against the single-GPU result.
Skipped when the box has fewer than 2 GPUs."""
import os
import subprocess
import sys

import pytest

from pamg_pkg import pamg

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.parametrize("xchg", ["sweep", "deep", "theta"])
@pytest.mark.parametrize("world", [2, 4])
def test_partitioned_smoother_and_vcycle_match_single_gpu(world, xchg):
    """theta: the default exchange with theta = 1/2 (the told strips of the cut faces are exchanged for the old-time terms);
    xchg = sweep: the producer warps of the sweeps send the cut-face values, an unpack launch runs between sweeps; k_halo
    copies, sends and receives after uploads and prolongations and on the levels without a producer warp; deep: nearly
    no agglomeration (PAMG_AGG_ELEMS=1024), so that every kernel family of the hierarchy runs partitioned with its own
    exchange."""
    if pamg.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    env = dict(os.environ)
    env.setdefault("PAMG_P2P_TIMEOUT_S", "30")
    if xchg == "deep":
        env["PAMG_AGG_ELEMS"] = "1024"
    if xchg == "theta":
        env["PAMG_TEST_THETA"] = "0.5"
    port = 29700 + (os.getpid() % 200)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(HERE, "multi_gpu_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "MULTI_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
