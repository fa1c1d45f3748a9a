"""The aux oracle (tests/oracle_aux/oracle_aux.c, orc_blend_aux): alpha = 1 - T, depth_map = sum of w * z in blend order
and n_contrib = entries blended, on hand-built tile lists; its image and examined counts equal orc_blend's bit for bit."""
import numpy as np

from luisacomputegaussiansplatting_b200 import scenes
from oracle import oracle as orc

import aux_oracle

f32 = np.float32
W, H = 32, 16      # two tiles; tile 1 never has a list
CX, CY = 5, 7      # every hand-built Gaussian is centred on this pixel
CONIC = (20.0, 0.0, 20.0)  # one pixel away: power -10, alpha <= 0.99 * e^-10 < 1/255 -- only the centre is reached


def run(entries):
    """entries: (opacity, z) front to back, all centred on (CX, CY); returns blend_aux's dict."""
    P = len(entries)
    means = np.tile(np.array([CX, CY], f32), (max(P, 1), 1))
    conic = np.tile(np.array(CONIC, f32), (max(P, 1), 1))
    opacity = np.array([e[0] for e in entries] or [0.0], f32)
    depth = np.array([e[1] for e in entries] or [0.0], f32)
    color = np.full((max(P, 1), 3), 0.5, f32)
    ranges = np.array([[0, P], [0, 0]], np.uint32)
    return aux_oracle.blend_aux(W, H, (0.0, 0.0, 0.0), ranges, np.arange(P, dtype=np.uint32), means, conic, opacity, color,
                         depth)


def walk(entries):
    """The oracle's walk for the centre pixel (power 0), restated in float32."""
    T, D, n = f32(1.0), f32(0.0), 0
    for op, z in entries:
        alpha = min(f32(0.99), f32(f32(op) * f32(orc.exp(0.0))))
        if alpha < f32(1.0) / f32(255.0):
            continue
        test_T = f32(T * f32(f32(1.0) - alpha))
        if test_T < f32(0.0001):
            break
        w = f32(T * alpha)
        D = f32(D + f32(w * f32(z)))
        n += 1
        T = test_T
    return f32(f32(1.0) - T), D, n


def check_centre(out, alpha, depth, n):
    assert out["alpha"][CY, CX] == f32(alpha)
    assert out["depth_map"][CY, CX] == f32(depth)
    assert out["n_contrib"][CY, CX] == n
    # nothing else is reached
    mask = np.ones((H, W), bool)
    mask[CY, CX] = False
    for k in ("alpha", "depth_map", "n_contrib"):
        assert not out[k][mask].any(), k


def test_single_gaussian():
    out = run([(0.5, 3.0)])
    check_centre(out, 0.5, 1.5, 1)
    assert walk([(0.5, 3.0)]) == (f32(0.5), f32(1.5), 1)


def test_two_stacked_gaussians():
    out = run([(0.5, 2.0), (0.5, 4.0)])
    check_centre(out, 0.75, 2.0, 2)


def test_alpha_test_skip_is_not_counted():
    entries = [(0.5, 2.0), (0.003, 9.0), (0.5, 4.0)]  # 0.003 < 1/255: skipped
    out = run(entries)
    check_centre(out, 0.75, 2.0, 2)
    assert out["n_examined"][CY, CX] == 3


def test_saturating_entry_is_not_counted():
    entries = [(0.95, 1.0), (0.95, 2.0), (0.95, 3.0), (0.95, 4.0), (0.95, 5.0)]
    a, d, n = walk(entries)
    assert n == 3  # T: 0.05, 0.0025, 0.000125, then 6.25e-6 < 1e-4 saturates
    out = run(entries)
    check_centre(out, a, d, n)
    assert out["n_examined"][CY, CX] == 4  # the walk stops at the saturating entry


def test_unreached_pixels_are_zero():
    out = run([])
    for k in ("alpha", "depth_map", "n_contrib"):
        assert not out[k].any(), k
    assert not out["img"].any()


def test_image_equals_orc_blend_bit_for_bit():
    sc, cfg = scenes.make_config_scene("C3", P=3000)
    Wf, Hf = 97, 61
    cam = orc.make_camera(scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world), Wf, Hf)
    fr = orc.forward(sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, orc.view_params(cam))
    assert fr.num_rendered > 0
    img, nex = orc.blend(Wf, Hf, (0.0, 0.0, 0.0), fr.ranges, fr.vals_sorted, fr.means_2d, fr.conic, sc.opacity, fr.color)
    stats = orc.blend_stats()
    out = aux_oracle.blend_aux(Wf, Hf, (0.0, 0.0, 0.0), fr.ranges, fr.vals_sorted, fr.means_2d, fr.conic, sc.opacity, fr.color,
                        fr.depth)
    assert np.array_equal(out["img"].view(np.uint32), img.view(np.uint32))
    assert np.array_equal(out["img"].view(np.uint32), fr.img.view(np.uint32))
    assert np.array_equal(out["n_examined"], nex)
    assert np.all(out["n_contrib"] <= nex)
    assert int(out["n_contrib"].sum()) == stats["E_contrib"]
    assert out["alpha"].min() >= 0.0 and out["alpha"].max() < 1.0
    assert np.array_equal(out["alpha"] > 0, out["n_contrib"] > 0)
    # the expected depth lies within the depths of the Gaussians that touch a tile
    zt = fr.depth[fr.tiles_touched > 0]
    hit = out["alpha"] > 0
    ez = out["depth_map"][hit] / out["alpha"][hit]
    assert ez.min() >= zt.min() * (1 - 1e-5) and ez.max() <= zt.max() * (1 + 1e-5)
