"""N>1 path.

CPU (gloo, world_size 2, runs everywhere): the row-shard decomposition itself -- per-shard partial sums all-reduced with
the same int64-sum contract the GPUs use over NCCL reproduce the whole-snapshot reconcile, and the pending check of a
shard given the reduced status reproduces the whole-snapshot rows.  The oracle stands in for the per-rank device.

GPU (needs >= 2 GPUs, otherwise skipped): tools/multi_gpu_parity.py under torchrun -- the real engine, NCCL all-reduce,
stacked results bit-exact against the oracle on the whole snapshot."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _torchrun(nproc, script, *args, timeout=600):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
           "--master-port", str(29500 + (os.getpid() % 400)), script, *args]
    return subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=timeout)


def test_row_ranges_partition():
    from kube_throttler_b200 import shard

    for n in (0, 1, 7, 100, 100003):
        for world in (1, 2, 3, 8):
            rs = [shard.row_range(n, r, world) for r in range(world)]
            assert rs[0][0] == 0 and rs[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(rs, rs[1:]))
            assert max(hi - lo for lo, hi in rs) - min(hi - lo for lo, hi in rs) <= 1


def test_sharded_pass_with_gloo_allreduce():
    r = _torchrun(2, os.path.join("tests", "gloo_shard_worker.py"))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "gloo shard parity: OK" in r.stdout


@pytest.mark.gpu
def test_two_gpu_parity():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = _torchrun(2, os.path.join("tools", "multi_gpu_parity.py"), "C3")
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "OK" in r.stdout


@pytest.mark.gpu
def test_missing_rank_times_out_instead_of_hanging():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = _torchrun(2, os.path.join("tools", "multi_gpu_timeout.py"), timeout=300)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "multi-gpu timeout: OK" in r.stdout
