"""bench.py --dump-outputs: the files it writes for a captured frame (synthetic arrays stand in for the GPU buffers)."""
import json
import os

import numpy as np
import pytest

import bench


def _frame():
    rng = np.random.default_rng(1)
    return {"img": (rng.random((3, 2000, 3000), dtype=np.float32), np.float32),             # 72 MB on its own
            "rgb8": (rng.integers(0, 256, (2000, 3000, 3), dtype=np.uint8), np.uint8),
            "keys_sorted": (rng.integers(0, 2**49, 5_000_000, dtype=np.uint64), np.uint64),
            "ranges": (rng.integers(0, 2**32, (500, 2), dtype=np.uint32), np.uint32),
            "num_rendered": (np.array([123456789], np.int64), np.int64)}


def test_dump_fits_the_budget_and_repeats_exactly(tmp_path):
    arrays = _frame()
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), arrays)
    a, b = tmp_path / "a", tmp_path / "b"
    assert sorted(os.listdir(a)) == sorted([k + ".npy" for k in arrays] + ["manifest.json"])
    assert sum(os.path.getsize(a / f) for f in os.listdir(a)) <= 64 * 10**6
    for k in arrays:
        x, y = np.load(a / (k + ".npy")), np.load(b / (k + ".npy"))
        assert x.dtype in (np.float32, np.float64) and np.array_equal(x, y), k

    man = json.load(open(a / "manifest.json"))
    # small outputs are written whole and exact
    assert man["ranges"]["sample"] is None and man["num_rendered"]["sample"] is None
    assert np.array_equal(np.load(a / "ranges.npy"), arrays["ranges"][0].astype(np.float64))
    assert np.load(a / "num_rendered.npy").tolist() == [123456789.0]
    # large ones keep the elements at the recorded indices, integers still exact
    for k in ("img", "keys_sorted"):
        s, src = man[k]["sample"], arrays[k][0]
        assert man[k]["shape"] == list(src.shape) and 0 < s["count"] < src.size
        idx = np.sort(np.random.default_rng(s["seed"]).choice(src.size, s["count"], replace=False))
        assert np.array_equal(np.load(a / (k + ".npy")).astype(src.dtype), src.reshape(-1)[idx]), k


def test_dump_refuses_integers_float64_cannot_hold(tmp_path):
    with pytest.raises(ValueError):
        bench.write_outputs(str(tmp_path), {"keys_sorted": (np.array([2**60 + 1], np.uint64), np.uint64)})


@pytest.mark.gpu
def test_dump_of_a_frame_holds_what_the_renderer_returns(tmp_path):
    from luisacomputegaussiansplatting_b200 import lcgs, scenes

    W, H, P = 320, 192, 8000
    sc, cfg = scenes.make_config_scene("C3", P=P)
    dev = lcgs.Device(0)
    r = lcgs.Renderer(dev, sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, W, H, list_capacity=1_000_000, rgb8=True)
    n = r.render(lcgs.make_camera(scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world), W, H))
    bench.write_outputs(str(tmp_path), bench.capture_frame(r, n))
    g = r.intermediates(n)
    g["rgb8"] = r.rgb8.cpu().numpy().reshape(H, W, 3)
    assert n > 0 and np.load(tmp_path / "num_rendered.npy").tolist() == [float(n)]
    for k in ("img", "rgb8", "depth", "radii", "tiles_touched", "offsets", "keys_sorted", "vals_sorted", "ranges", "means_2d",
              "conic", "color"):
        got = np.load(tmp_path / (k + ".npy"))
        assert got.shape == g[k].shape and np.array_equal(got.astype(g[k].dtype), g[k]), k
    dev.close()
