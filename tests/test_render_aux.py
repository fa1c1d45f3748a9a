"""Per-pixel alpha / depth / contributor-count planes on the GPU, against the aux oracle (tests/oracle_aux, orc_blend_aux).

Bars: alpha within 2e-3 (the image bar), depth_map within 2e-3 x the largest view depth of a touching Gaussian, and
n_contrib equal except at most ceil(1e-4 * W * H) pixels that differ by exactly 1 (a saturation decision on a rounding
tie moves one entry).  Turning the planes on changes no other output by a bit."""
import math
import os
import subprocess

import numpy as np
import pytest

from luisacomputegaussiansplatting_b200 import scenes
from oracle import oracle as orc

import aux_oracle

pytestmark = pytest.mark.gpu

CASES = [
    ("C3", 20_000, 640, 360),
    ("C1", 10_000, 200, 200),
    ("C2", 50_000, 1237, 822),
    ("C3", 3_000, 97, 61),
    ("C3", 1, 64, 64),
]


@pytest.fixture(scope="module")
def lcgs():
    from luisacomputegaussiansplatting_b200 import lcgs as m
    return m


@pytest.fixture(scope="module")
def dev(lcgs):
    d = lcgs.Device(0)
    yield d
    d.close()


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def pose_of(key, P):
    sc, cfg = scenes.make_config_scene(key, P=P)
    return sc, (scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world))


def oracle_aux(fr, opacity, W, H, row0=0, row1=-1):
    return aux_oracle.blend_aux(W, H, (0.0, 0.0, 0.0), fr.ranges, fr.vals_sorted, fr.means_2d, fr.conic, opacity, fr.color,
                         fr.depth, row0, row1)


def assert_aux_close(alpha, depth_map, n_contrib, want, fr):
    W, H = alpha.shape[1], alpha.shape[0]
    assert float(np.abs(alpha - want["alpha"]).max()) <= 2e-3, "alpha"
    touching = fr.tiles_touched > 0
    zmax = float(fr.depth[touching].max()) if touching.any() else 1.0
    assert float(np.abs(depth_map - want["depth_map"]).max()) <= 2e-3 * zmax, "depth_map"
    d = n_contrib.astype(np.int64) - want["n_contrib"].astype(np.int64)
    assert int((d != 0).sum()) <= math.ceil(1e-4 * W * H), "n_contrib: %d pixels differ" % int((d != 0).sum())
    assert int(np.abs(d).max()) <= 1, "n_contrib differs by more than one entry"


def render(lcgs, dev, sc, pose, W, H, cap, **kw):
    r = lcgs.Renderer(dev, sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, W, H, list_capacity=cap, **kw)
    n = r.render(lcgs.make_camera(*pose, W, H))
    return r, n


@pytest.mark.parametrize("key,P,W,H", CASES)
def test_aux_planes_match_the_oracle(lcgs, dev, key, P, W, H):
    sc, pose = pose_of(key, P)
    fr = orc.forward(sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, orc.view_params(orc.make_camera(*pose, W, H)))
    r, n = render(lcgs, dev, sc, pose, W, H, max(fr.num_rendered, 1) + 17, aux=True, rgb8=True)
    assert n == fr.num_rendered
    g = r.intermediates(n)
    assert_aux_close(g["alpha"], g["depth_map"], g["n_contrib"], oracle_aux(fr, sc.opacity, W, H), fr)
    e = r.expected_depth().cpu().numpy()
    hit = g["alpha"] > 0
    assert np.array_equal(e[~hit], np.zeros_like(e[~hit]))
    # aux on changes no other output by a bit
    r0, n0 = render(lcgs, dev, sc, pose, W, H, max(fr.num_rendered, 1) + 17, rgb8=True)
    g0 = r0.intermediates(n0)
    assert n0 == n
    for k, v in g0.items():
        if k == "num_rendered":
            continue
        assert np.array_equal(np.ascontiguousarray(v).view(np.uint8), np.ascontiguousarray(g[k]).view(np.uint8)), k
    assert np.array_equal(r.rgb8.cpu().numpy(), r0.rgb8.cpu().numpy()), "rgb8"


def test_full_size_c3(lcgs, dev):
    sc, cfg = scenes.make_config_scene("C3")
    pose = (scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world))
    W, H = cfg.W, cfg.H
    fr = orc.forward(sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, orc.view_params(orc.make_camera(*pose, W, H)))
    r, n = render(lcgs, dev, sc, pose, W, H, 20_000_000, aux=True, keep_intermediates=False)
    assert n == fr.num_rendered
    want = oracle_aux(fr, sc.opacity, W, H)
    assert_aux_close(r.alpha().cpu().numpy(), r.depth_map().cpu().numpy(),
                     r.n_contrib().cpu().numpy().view(np.uint32), want, fr)
    img_aux = r.image().cpu().numpy()
    r.c_frame.target_alpha = r.c_frame.target_depth = r.c_frame.target_n_contrib = None
    assert r.render(lcgs.make_camera(*pose, W, H)) == n
    assert np.array_equal(bits(r.image().cpu().numpy()), bits(img_aux))


def test_splat_forward_aux(lcgs, dev):
    """GSTileSplatter.forward (lcgs_b200_splat_forward) with aux targets in the output proxy."""
    import torch
    W, H, P = 512, 288, 30_000
    sc, pose = pose_of("C3", P)
    cam = lcgs.make_camera(*pose, W, H)
    fr = orc.forward(sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, orc.view_params(orc.make_camera(*pose, W, H)))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    d_pos, d_scale, d_rotq, d_sh, d_opacity = t(sc.pos), t(sc.scale), t(sc.rotq), t(sc.sh), t(sc.opacity)
    L = fr.num_rendered + 100
    gx, gy = (W + 15) // 16, (H + 15) // 16
    shp, proj, spl = lcgs.SHProcessor(), lcgs.GSProjector(), lcgs.GSTileSplatter()
    shp.create(dev), proj.create(dev), spl.create(dev)

    def run(aux):
        d_color = dev.create_buffer(torch.float32, 3 * P)
        d_means, d_depth, d_cov = (dev.create_buffer(torch.float32, k * P) for k in (2, 1, 3))
        accel = lcgs.GSTileSplatterAccelProxy(
            dev.create_buffer(torch.int32, P), dev.create_buffer(torch.int32, P), dev.create_buffer(torch.int64, L),
            dev.create_buffer(torch.int32, L), dev.create_buffer(torch.int64, L), dev.create_buffer(torch.int32, L),
            dev.create_buffer(torch.int32, 2 * gx * gy))
        out = lcgs.GSSplatForwardOutputProxy(H, W, dev.create_buffer(torch.float32, 3 * W * H), dev.create_buffer(torch.int32, P))
        if aux:
            out.target_alpha = torch.full((W * H,), 7.0, device="cuda")
            out.target_depth = torch.full((W * H,), 7.0, device="cuda")
            out.target_n_contrib = torch.full((W * H,), 7, dtype=torch.int32, device="cuda")
        shp.process(None, lcgs.GPUPointsProxy(P, 3, d_pos), cam, d_sh, d_color, 3, 3)
        proj.forward(None, lcgs.GSProjectorInputProxy(P, d_pos, d_scale, d_rotq, 1.0),
                     lcgs.GSProjectorOutputProxy(d_means, d_cov, d_depth), cam)
        inp = lcgs.GSTileSplatterInputProxy(P, (0.0, 0.0, 0.0), d_means, d_depth, d_cov, d_color, d_opacity)
        assert spl.forward(dev, None, accel, inp, out) == fr.num_rendered
        return out

    out = run(True)
    want = oracle_aux(fr, sc.opacity, W, H)
    assert_aux_close(out.target_alpha.view(H, W).cpu().numpy(), out.target_depth.view(H, W).cpu().numpy(),
                     out.target_n_contrib.view(H, W).cpu().numpy().view(np.uint32), want, fr)
    out0 = run(False)
    assert np.array_equal(bits(out.target_img.cpu().numpy()), bits(out0.target_img.cpu().numpy()))


def test_tile_row_bands_fill_the_same_planes(lcgs, dev):
    W, H, P = 640, 360, 20_000
    sc, pose = pose_of("C3", P)
    cam = lcgs.make_camera(*pose, W, H)
    whole, _ = render(lcgs, dev, sc, pose, W, H, 400_000, aux=True)
    gy = (H + 15) // 16
    r = lcgs.Renderer(dev, sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, W, H, list_capacity=400_000, aux=True)
    for t in (r.alpha_map, r.depth_plane, r.n_contrib_map):
        t.fill_(3)
    for r0, r1 in [(0, 9), (9, gy)]:
        r.set_tile_rows(r0, r1)
        r.render(cam)
    for a, b in ((r.alpha(), whole.alpha()), (r.depth_map(), whole.depth_map()), (r.n_contrib(), whole.n_contrib())):
        assert np.array_equal(a.cpu().numpy().view(np.uint32), b.cpu().numpy().view(np.uint32))


def test_empty_frame_zeroes_the_planes_and_keeps_the_image(lcgs, dev):
    W, H, P = 128, 96, 2000
    sc, pose = pose_of("C3", P)
    cam = lcgs.make_camera(*pose, W, H)
    behind = sc.pos.copy()
    behind[:] = np.array(scenes.CAM_POS, np.float32) - 5.0 * np.array(list(cam.front), np.float32)
    r = lcgs.Renderer(dev, behind, sc.scale, sc.rotq, sc.sh, sc.opacity, W, H, list_capacity=1000, aux=True)
    r.img.fill_(0.25)
    r.alpha_map.fill_(0.5), r.depth_plane.fill_(2.0), r.n_contrib_map.fill_(9)
    assert r.render(cam) == 0
    assert bool((r.img == 0.25).all())
    assert not bool(r.alpha_map.any()) and not bool(r.depth_plane.any()) and not bool(r.n_contrib_map.any())


def test_sub_allocated_planes_edges_and_alignment(lcgs, dev):
    import torch
    W, H, P = 200, 200, 10_000
    sc, pose = pose_of("C1", P)
    cam = lcgs.make_camera(*pose, W, H)
    r = lcgs.Renderer(dev, sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, W, H, list_capacity=400_000, aux=True)
    r.render(cam)
    ref = [t.clone() for t in (r.alpha_map, r.depth_plane, r.n_contrib_map)]
    pad = 37
    canary = 0x7F7F1234
    bufs = [torch.full((W * H + 2 * pad,), canary, dtype=torch.int32, device="cuda") for _ in range(3)]
    f = r.c_frame
    f.target_alpha, f.target_depth, f.target_n_contrib = (b.data_ptr() + 4 * pad for b in bufs)
    r.render(cam)
    for b, want in zip(bufs, ref):
        h = b.cpu().numpy()
        assert (h[:pad] == canary).all() and (h[pad + W * H:] == canary).all()
        assert np.array_equal(h[pad:pad + W * H], want.cpu().numpy().view(np.int32))
    # Q1: the last tile row and column are never binned -- nothing reaches them
    gx, gy = (W + 15) // 16, (H + 15) // 16
    for t in ref:
        p = t.view(H, W).cpu().numpy()
        assert not p[(gy - 1) * 16:, :].any() and not p[:, (gx - 1) * 16:].any()
    # a misaligned plane is rejected
    f.target_alpha = bufs[0].data_ptr() + 2
    with pytest.raises(lcgs.LcgsError) as e:
        r.render(cam)
    assert e.value.status == -1
    f.target_alpha, f.target_depth, f.target_n_contrib = (r.alpha_map.data_ptr(), r.depth_plane.data_ptr(),
                                                          r.n_contrib_map.data_ptr())


def test_cuda_graph_replay_and_pose_change(lcgs, dev):
    import torch
    W, H, P = 400, 240, 12_000
    sc, pose = pose_of("C3", P)
    vp = lcgs.view_params(lcgs.make_camera(*pose, W, H))
    pose2 = (tuple(np.array(scenes.CAM_POS) + np.array([0.4, -0.2, 0.3])), pose[1], pose[2])
    vp2 = lcgs.view_params(lcgs.make_camera(*pose2, W, H))
    r = lcgs.Renderer(dev, sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, W, H, list_capacity=400_000, aux=True)
    r.render_async(vp)
    dev.num_rendered()
    eager = [t.clone() for t in (r.alpha_map, r.depth_plane, r.n_contrib_map)]
    for t in (r.alpha_map, r.depth_plane, r.n_contrib_map):
        t.fill_(5)
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            r.render_async(vp, stream=s)
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip((r.alpha_map, r.depth_plane, r.n_contrib_map), eager):
        assert torch.equal(a, b)
    # another pose over the same planes overwrites every pixel: it equals a fresh renderer's frame
    r.render_async(vp2)
    dev.num_rendered()
    fresh = lcgs.Renderer(dev, sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, W, H, list_capacity=400_000, aux=True)
    fresh.render_async(vp2)
    dev.num_rendered()
    for a, b in zip((r.alpha_map, r.depth_plane, r.n_contrib_map), (fresh.alpha_map, fresh.depth_plane, fresh.n_contrib_map)):
        assert torch.equal(a, b)


@pytest.mark.parametrize("fused", [1, 0])
def test_cli_dumps_the_planes(tmp_path, fused):
    from luisacomputegaussiansplatting_b200 import build as native
    from luisacomputegaussiansplatting_b200 import plyio
    W, H, P = 320, 200, 6000
    sc, cfg = scenes.make_config_scene("C1", P=P)
    ply = str(tmp_path / "tiny_lego.ply")
    plyio.write_gs_ply(ply, sc.pos, sc.sh, sc.logit_opacity, sc.log_scale, sc.raw_rot)
    app = native.build_app()
    d = tmp_path / "dump"
    r = subprocess.run([app, "--ply=" + ply, "--out", str(tmp_path / "out"), "--world=blender", "--res", "%dx%d" % (W, H),
                        "--backend=cuda", "--fused", str(fused), "--capacity", "2000000", "--aux", "1", "--dump", str(d)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    pos, scale, rotq, opacity, sh = plyio.read_gs_ply(ply)
    cam = orc.make_camera(scenes.CAM_POS, scenes.CAM_TARGET, scenes.WORLD_UP_BLENDER, W, H)
    fr = orc.forward(pos, scale, rotq, sh, opacity, orc.view_params(cam))
    want = oracle_aux(fr, opacity, W, H)
    alpha = np.fromfile(os.path.join(d, "alpha.f32"), np.float32).reshape(H, W)
    dmap = np.fromfile(os.path.join(d, "depth_map.f32"), np.float32).reshape(H, W)
    ncon = np.fromfile(os.path.join(d, "n_contrib.u32"), np.uint32).reshape(H, W)
    assert_aux_close(alpha, dmap, ncon, want, fr)

