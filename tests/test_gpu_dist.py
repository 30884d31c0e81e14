"""Row-partitioned single LP over 2 GPUs (SURVEY.md §8e): needs two devices, skipped otherwise.  The host-side
partition logic is covered on the CPU below."""
import os
import subprocess
import sys

import numpy as np
import pytest

from activesetmethods_b200 import shard

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_row_partitioned_lp_two_gpus(gpu):
    if gpu.asm_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29517", os.path.join(ROOT, "tests", "dist_worker.py"), "case118", "1e-7"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    print(out.stdout[-2000:], out.stderr[-2000:])
    assert out.returncode == 0 and "DIST_OK" in out.stdout


def test_row_blocks_cover_and_balance():
    rng = np.random.default_rng(0)
    lens = rng.integers(0, 30, 1000)
    rp = np.concatenate([[0], np.cumsum(lens)])
    for world in (1, 2, 3, 8):
        cuts = shard.row_blocks(rp, world)
        assert cuts[0] == 0 and cuts[-1] == 1000 and all(a <= b for a, b in zip(cuts, cuts[1:]))
        nnz = [rp[b] - rp[a] for a, b in zip(cuts, cuts[1:])]
        assert sum(nnz) == rp[-1] and max(nnz) <= rp[-1] / world + 64


def test_partial_aty_sums_to_full():
    """The identity the all-reduce relies on: sum_g K_g' y_g == K' y for the row blocks of shard.row_blocks."""
    import scipy.sparse as sp
    K = sp.random(200, 120, density=0.05, random_state=1, format="csr")
    y = np.random.default_rng(2).standard_normal(200)
    cuts = shard.row_blocks(K.indptr, 4)
    parts = [K[a:b].T @ y[a:b] for a, b in zip(cuts, cuts[1:])]
    assert np.allclose(sum(parts), K.T @ y, rtol=0, atol=1e-13)
