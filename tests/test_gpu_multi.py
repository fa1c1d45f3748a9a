"""Multi-GPU checks as tests (marker `gpu_multi`; need >= 2 GPUs of one node, skipped otherwise -- also under `-m gpu`
on a one-GPU box and on the CPU box).  Each test launches scripts/multi_gpu_check.py under torchrun on every visible
GPU (at most 8): view-sharded sweeps (NCCL gather, peer-store ring with barriers, peer-store ring with device-side
flags and a consumer stream) and tile-row-sharded frames (NCCL strips, peer stores into one image, a band without
instances) must reproduce single-GPU frames bit for bit.

    gpurun --gpus 2 -- python -m pytest tests -m gpu_multi -q
"""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gpus():
    try:
        import torch
        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


pytestmark = [pytest.mark.gpu, pytest.mark.gpu_multi, pytest.mark.skipif(_gpus() < 2, reason="needs >= 2 GPUs on one node")]


def _run(extra, port, timeout=900):
    n = min(_gpus(), 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "scripts", "multi_gpu_check.py")] + extra
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    out = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert out["world"] == n
    return out


def test_sharded_frames_equal_single_gpu_frames():
    out = _run(["--config", "C3", "--gaussians", "400000"], 29541)
    for k in ("view_sharded_bit_exact", "view_sharded_peer_bit_exact", "view_sharded_flags_bit_exact", "tile_row_sharded_bit_exact",
              "tile_row_sharded_peer_bit_exact", "instances_partition_exactly", "empty_band_bit_exact"):
        assert out[k] is True, (k, out)
    assert out["empty_band_instances"] == 0


def test_full_size_c2_orbit_views_and_frame():
    """The C4 workload's scene at full size (6.1 M Gaussians, 1237x822)."""
    out = _run(["--config", "C2", "--gaussians", "6100000", "--capacity", "30000000"], 29542)
    assert out["view_sharded_peer_bit_exact"] and out["view_sharded_flags_bit_exact"] and out["tile_row_sharded_peer_bit_exact"]


def test_full_size_c5_tile_row_sharded_8k_frame():
    """The C5 frame at full size (10 M Gaussians, 7680x4320, 234 M instances) split by tile rows over the GPUs of the box,
    every band blended into one image on rank 0: bit-identical to rank 0's own single-GPU frame."""
    out = _run(["--config", "C5", "--gaussians", "10000000", "--capacity", "260000000", "--skip-views", "--views", "2"], 29543,
               timeout=1500)
    assert out["tile_row_sharded_peer_bit_exact"] and out["tile_row_sharded_bit_exact"] and out["instances_partition_exactly"]
    assert out["num_rendered"] > 150_000_000
