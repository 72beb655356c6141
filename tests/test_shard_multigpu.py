"""Multi-GPU (>= 2 B200s on the box; skipped otherwise): z-slab sharded volumes -- through the NCCL all-gather and through
the fused peer-memory epilogue (mp_query_grid_peers) -- are bit-identical to the single-GPU volume on every rank."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("fused", [False, True])
def test_sharded_volume_equals_single_gpu_volume(fused):
    n = _gpus()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 2 if n < 4 else 4
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr",
           "127.0.0.1", "--master-port", "29517", os.path.join(ROOT, "tools", "shard_check.py")] + (["--fused", "--octree"] if fused else [])
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "shard_check OK: identical volumes" in r.stdout
    if fused:
        assert "shard_check OK (fused slab exchange)" in r.stdout
        assert "shard_check OK (list-sharded octree engines)" in r.stdout
