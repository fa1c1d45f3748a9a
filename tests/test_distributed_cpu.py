"""world_size-2 gloo tests (CPU) of the multi-GPU host logic: view sharding and tile-row sharding.

The renderer passed to the drivers is the CPU oracle here -- as the checker standing in for a GPU
rank -- so the assembled results can be compared bit for bit with a single-process frame.
"""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from luisacomputegaussiansplatting_b200 import distributed as D
from luisacomputegaussiansplatting_b200 import scenes
from oracle import oracle as orc

W, H, P = 200, 120, 1500


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _scene():
    sc, _ = scenes.make_config_scene("C3", P=P)
    return sc


def _frame(sc, pose, row0=0, row1=-1):
    vp = orc.view_params(orc.make_camera(*pose, W, H))
    return orc.forward(sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, vp, row0=row0, row1=row1)


class MemmapRing:
    """Stand-in for distributed.PeerFrameRing on CPU: the "peer-mapped device buffer" is a file every rank maps;
    ptr(slot) is a byte offset into it.  Same interface, same barriers."""

    def __init__(self, path, slots, dst=0):
        self.slots, self.dst, self.group = slots, dst, None
        self.frame_bytes = 3 * H * W * 4
        if dist.get_rank() == dst:
            np.zeros(slots * 3 * H * W, np.float32).tofile(path)
        dist.barrier()
        self.mem = np.memmap(path, dtype=np.float32, mode="r+", shape=(slots, 3, H, W))

    def ptr(self, slot):
        assert 0 <= slot < self.slots
        return slot * self.frame_bytes

    def write(self, ptr, img, rows=None):
        slot = ptr // self.frame_bytes
        if rows is None:
            self.mem[slot] = img
        else:
            self.mem[slot][:, rows[0]:rows[1], :] = img[:, rows[0]:rows[1], :]

    def complete(self):
        self.mem.flush()
        dist.barrier()

    def frame(self, slot):
        return np.array(self.mem[slot])

    def release(self):
        dist.barrier()


def _worker(rank, world, port, mode, q, ring_path):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sc = _scene()
    try:
        if mode == "rows_empty_band":
            # the last rank owns only the last tile row, which is never binned (Q1): its band has 0 instances and must
            # still overwrite the stale pixels of the slot with the background
            ring = MemmapRing(ring_path, slots=2)
            if rank == 0:
                ring.mem[1][:] = -7.0
            dist.barrier()
            gy = (H + 15) // 16
            pose = (scenes.CAM_POS, scenes.CAM_TARGET, scenes.WORLD_UP_COLMAP)
            bg = (0.25, 0.5, 0.75)

            def band(r0, r1, ptr):
                vp = orc.view_params(orc.make_camera(*pose, W, H))
                fr = orc.forward(sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, vp, bg=bg, row0=r0, row1=r1)
                assert (fr.num_rendered == 0) == (r0 == gy - 1)
                ring.write(ptr, fr.img, (min(H, 16 * r0), min(H, 16 * r1)))

            img, bands = D.render_frame_tile_row_sharded_peer(band, H, ring, slot=1, bands=[(0, gy - 1), (gy - 1, gy)])
            if rank == 0:
                q.put((img, bands))
        elif mode in ("views_peer", "rows_peer"):
            ring = MemmapRing(ring_path, slots=5)
            if mode == "views_peer":
                out = D.render_sweep_view_sharded_peer(
                    lambda k, ptr: ring.write(ptr, _frame(sc, scenes.orbit_pose(k * 13)).img), 5, ring)
                if rank == 0:
                    q.put(out)
            else:
                pose = (scenes.CAM_POS, scenes.CAM_TARGET, scenes.WORLD_UP_COLMAP)
                img, bands = D.render_frame_tile_row_sharded_peer(
                    lambda r0, r1, ptr: ring.write(ptr, _frame(sc, pose, r0, r1).img, (min(H, 16 * r0), min(H, 16 * r1))),
                    H, ring, slot=2)
                if rank == 0:
                    q.put((img, bands))
        elif mode == "views":
            nviews = 5  # odd on purpose: the last round has an idle rank
            out = D.render_sweep_view_sharded(lambda k: torch.from_numpy(_frame(sc, scenes.orbit_pose(k * 13)).img.copy()),
                                              nviews)
            if rank == 0:
                q.put([f.numpy() for f in out])
        else:
            pose = (scenes.CAM_POS, scenes.CAM_TARGET, scenes.WORLD_UP_COLMAP)
            weights = None if mode == "rows" else [1, 1, 1, 50, 1, 1, 1, 1]
            img, bands = D.render_frame_tile_row_sharded(
                lambda r0, r1: torch.from_numpy(_frame(sc, pose, r0, r1).img.copy()), H, weights)
            if rank == 0:
                q.put((img.numpy(), bands))
    finally:
        dist.destroy_process_group()


def _run(mode, ring_path=None, world=2):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, mode, q, ring_path)) for r in range(world)]
    for p in procs:
        p.start()
    res = q.get(timeout=240)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return res


def test_view_sharded_sweep_gathers_frames_in_view_order():
    frames = _run("views")
    sc = _scene()
    assert len(frames) == 5
    for k, f in enumerate(frames):
        want = _frame(sc, scenes.orbit_pose(k * 13)).img
        assert np.array_equal(f.view(np.uint32), want.view(np.uint32)), k


@pytest.mark.parametrize("mode", ["rows", "rows_weighted"])
def test_tile_row_sharded_frame_equals_single_device_frame(mode):
    img, bands = _run(mode)
    want = _frame(_scene(), (scenes.CAM_POS, scenes.CAM_TARGET, scenes.WORLD_UP_COLMAP)).img
    assert bands[0][0] == 0 and bands[-1][1] == (H + 15) // 16 and bands[0][1] == bands[1][0]
    assert np.array_equal(img.view(np.uint32), want.view(np.uint32))


def test_peer_drivers_assemble_the_same_frames(tmp_path):
    """The drivers of the gather-fused-into-the-render path (every rank writes straight into the destination's
    buffer; on a GPU box that buffer is peer-mapped device memory, here a shared file)."""
    frames = _run("views_peer", str(tmp_path / "views_ring.bin"))
    sc = _scene()
    assert len(frames) == 5
    for k, f in enumerate(frames):
        want = _frame(sc, scenes.orbit_pose(k * 13)).img
        assert np.array_equal(f.view(np.uint32), want.view(np.uint32)), k
    img, bands = _run("rows_peer", str(tmp_path / "rows_ring.bin"))
    want = _frame(sc, (scenes.CAM_POS, scenes.CAM_TARGET, scenes.WORLD_UP_COLMAP)).img
    assert bands[0][0] == 0 and bands[-1][1] == (H + 15) // 16
    assert np.array_equal(img.view(np.uint32), want.view(np.uint32))


def test_a_band_without_instances_still_writes_the_background(tmp_path):
    img, bands = _run("rows_empty_band", str(tmp_path / "ring.bin"))
    sc = _scene()
    vp = orc.view_params(orc.make_camera(scenes.CAM_POS, scenes.CAM_TARGET, scenes.WORLD_UP_COLMAP, W, H))
    want = orc.forward(sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, vp, bg=(0.25, 0.5, 0.75))
    assert want.num_rendered > 0 and bands[-1] == ((H + 15) // 16 - 1, (H + 15) // 16)
    assert np.array_equal(img.view(np.uint32), want.img.view(np.uint32)), "stale pixels left in the empty band"


def test_partitioning_helpers():
    assert D.shard_views(10, 4, 1) == [1, 5, 9]
    assert sorted(sum((D.shard_views(7, 3, r) for r in range(3)), [])) == list(range(7))
    for rows, world in [(68, 8), (270, 8), (3, 8), (1, 2), (52, 4)]:
        bands = D.split_tile_rows(rows, world)
        assert bands[0][0] == 0 and bands[-1][1] == rows
        assert all(a[1] == b[0] for a, b in zip(bands, bands[1:])) and all(r1 >= r0 for r0, r1 in bands)
        if rows >= world:
            assert max(r1 - r0 for r0, r1 in bands) - min(r1 - r0 for r0, r1 in bands) <= 1
    # heavy rows get narrow bands
    w = [1.0] * 20
    w[10] = 100.0
    bands = D.split_tile_rows(20, 4, w)
    sums = [sum(w[a:b]) for a, b in bands]
    assert max(sums) <= 100.0 + 10.0
    rg = torch.tensor([[0, 3], [3, 5], [0, 0], [5, 9]], dtype=torch.int32)
    assert D.row_weights_from_ranges(rg, 2) == [5.0, 4.0]
