"""The backward pass on the GPU (lcgs_b200_render_backward, lcgs.DifferentiableRenderer) against the float64 torch
reference (tests/torch_reference.py) for L = sum(img * R), R a fixed random tensor.

Bars per gradient tensor: relative L2 error <= 1e-3 and cosine >= 0.9999.  The GPU walk makes the forward's own
decisions (ex2-based alpha, float32 T), the reference the oracle's (exact exp): a saturation decision on a rounding tie
can move one entry of one pixel, which the bars absorb."""
import ctypes as C

import numpy as np
import pytest
import torch

from luisacomputegaussiansplatting_b200 import scenes
from oracle import oracle as orc

import torch_reference as tr

pytestmark = pytest.mark.gpu

# test_render_aux.py's frame shapes, scaled down so that the float64 reference stays fast
CASES = [
    ("C3", 4_000, 320, 180),
    ("C1", 3_000, 200, 200),
    ("C2", 5_000, 320, 212),
    ("C3", 1_500, 97, 61),
    ("C3", 1, 64, 64),
]
NAMES = ("pos", "scale", "rotq", "sh", "opacity")


@pytest.fixture(scope="module")
def lcgs():
    from luisacomputegaussiansplatting_b200 import lcgs as m
    return m


@pytest.fixture(scope="module")
def dev(lcgs):
    d = lcgs.Device(0)
    yield d
    d.close()


def metrics(got, want):
    got, want = np.asarray(got, np.float64).ravel(), np.asarray(want, np.float64).ravel()
    nw, ng = np.linalg.norm(want), np.linalg.norm(got)
    if nw == 0.0:
        return (0.0 if ng == 0.0 else np.inf), 1.0
    return float(np.linalg.norm(got - want) / nw), float(got @ want / max(nw * ng, 1e-300))


def assert_close(name, got, want, errs):
    rel, cos = metrics(got, want)
    errs[name] = (rel, cos)
    assert rel <= 1e-3 and cos >= 0.9999, (name, rel, cos)


def scene_arrays(key, P, deg=3, dense=False):
    sc, cfg = scenes.make_config_scene(key, P=P)
    pose = (scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world))
    sh = np.ascontiguousarray(sc.sh[:, :(deg + 1) ** 2])
    scale, opacity = sc.scale, sc.opacity
    if dense:  # large, nearly opaque Gaussians: most pixels saturate
        scale = (scale * 4.0).astype(np.float32)
        opacity = np.full_like(opacity, 0.97)
    return [np.ascontiguousarray(a, np.float32) for a in (sc.pos, scale, sc.rotq, sh, opacity)], pose


def gpu_backward(lcgs, dev, arrays, pose, W, H, deg, bg, R, list_capacity=2_000_000, scale_modifier=1.0,
                 prepare_scene=True):
    """Render with Renderer, then lcgs_b200_render_backward with every output requested; returns (renderer, grads)."""
    r = lcgs.Renderer(dev, *arrays, W, H, list_capacity=list_capacity, sh_deg=deg, bg_color=bg,
                      scale_modifier=scale_modifier, prepare_scene=prepare_scene)
    cam = lcgs.make_camera(*pose, W, H)
    vp = lcgs.view_params(cam)
    r.render_async(vp)
    dev.num_rendered()
    return r, run_backward(lcgs, dev, r, vp, R)


def run_backward(lcgs, dev, r, vp, R):
    """lcgs_b200_render_backward of the frame `r` last rendered (with view `vp`), every output requested."""
    P = r.P
    out = {n: torch.zeros_like(t) for n, t in zip(NAMES, (r.pos, r.scale, r.rotq, r.sh, r.opacity))}
    out["means_2d"] = torch.zeros(P, 2, device="cuda")
    out["conic"] = torch.zeros(P, 3, device="cuda")
    out["color"] = torch.zeros(P, 3, device="cuda")
    dl = torch.from_numpy(np.ascontiguousarray(R, np.float32)).cuda()
    g = lcgs._capi.Grad()
    g.dl_dimg = dl.data_ptr()
    for n in out:
        setattr(g, "grad_" + n, out[n].data_ptr())
    dev.check(dev.lib.lcgs_b200_render_backward(dev.ctx, C.byref(r.c_scene), C.byref(vp), C.byref(r.c_frame), C.byref(g), None))
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def reference(arrays, pose, W, H, deg, bg, R, scale_modifier=1.0):
    vp = orc.view_params(orc.make_camera(*pose, W, H))
    fr = orc.forward(arrays[0], arrays[1], arrays[2], arrays[3], arrays[4], vp, bg=bg, sh_deg=deg,
                     scale_modifier=scale_modifier)
    L = [tr.leaf(a) for a in arrays]
    img, (means, conic, color) = tr.forward(*L, vp, fr, deg=deg, bg=bg, scale_modifier=scale_modifier, keep_2d=True)
    (img * torch.from_numpy(np.asarray(R, np.float64))).sum().backward()
    want = {n: x.grad.numpy() for n, x in zip(NAMES, L)}
    want.update(means_2d=means.grad.numpy(), conic=conic.grad.numpy(), color=color.grad.numpy())
    return fr, want, color.detach().numpy()


def check_case(lcgs, dev, key, P, W, H, deg=3, bg=(0.0, 0.0, 0.0), dense=False, seed=0):
    arrays, pose = scene_arrays(key, P, deg, dense)
    R = np.random.default_rng(seed).uniform(-1.0, 1.0, (3, H, W))
    r, got = gpu_backward(lcgs, dev, arrays, pose, W, H, deg, bg, R)
    fr, want, _ = reference(arrays, pose, W, H, deg, bg, R)
    assert np.array_equal(r.tiles_touched.cpu().numpy().view(np.uint32), fr.tiles_touched)
    errs = {}
    for n in want:
        assert_close(n, got[n], want[n], errs)
    # a Gaussian no tile holds gets exactly zero everywhere
    idle = fr.tiles_touched == 0
    for n in got:
        assert not np.any(got[n][idle]), n
    print(key, P, W, H, "deg", deg, "bg", bg, "dense" if dense else "", {k: "%.2e / %.7f" % v for k, v in errs.items()})
    return got, want, fr


@pytest.mark.parametrize("key,P,W,H", CASES)
def test_gradients_match_the_reference(lcgs, dev, key, P, W, H):
    check_case(lcgs, dev, key, P, W, H)


@pytest.mark.parametrize("deg", [0, 1, 2])
def test_sh_degrees(lcgs, dev, deg):
    check_case(lcgs, dev, "C3", 3_000, 256, 144, deg=deg)


def test_background(lcgs, dev):
    check_case(lcgs, dev, "C1", 3_000, 200, 200, bg=(0.3, 0.6, 0.15))


def test_dense_saturating_scene(lcgs, dev):
    got, want, fr = check_case(lcgs, dev, "C3", 6_000, 160, 96, dense=True)
    # most pixels end by saturating: the walk's stop is exercised
    assert fr.n_examined.mean() < np.diff(fr.ranges.astype(np.int64), axis=1).mean()


def test_zero_gradients_off_screen_near_culled_and_clamped(lcgs, dev):
    W, H, P = 160, 96, 3_000
    arrays, pose = scene_arrays("C3", P)
    cam = lcgs.make_camera(*pose, W, H)
    front = np.array(list(cam.front), np.float32)
    campos = np.array(scenes.CAM_POS, np.float32)
    arrays[0][:200] = campos + 0.1 * front            # near-culled (z < 0.2)
    arrays[0][200:400] = campos - 3.0 * front         # behind the camera
    arrays[0][400:600] = campos + 3.0 * front + 50.0 * np.array(list(cam.right), np.float32)  # far off-screen
    arrays[3][600:900, 0, :] = np.where(np.arange(300)[:, None] % 2 == 0, 8.0, -8.0)  # colours clamped at 1 / 0
    R = np.random.default_rng(5).uniform(-1.0, 1.0, (3, H, W))
    r, got = gpu_backward(lcgs, dev, arrays, pose, W, H, 3, (0.0, 0.0, 0.0), R)
    tt = r.tiles_touched.cpu().numpy()
    assert not tt[:600].any()
    for n in got:
        assert not np.any(got[n][:600]), n
    fr, want, color = reference(arrays, pose, W, H, 3, (0.0, 0.0, 0.0), R)
    t = lambda a: torch.from_numpy(np.asarray(a, np.float64))  # noqa: E731
    vp = orc.view_params(orc.make_camera(*pose, W, H))
    d = t(arrays[0]) - t(list(vp.cam_pos))[None]
    d = d / torch.linalg.norm(d, dim=1, keepdim=True)
    res = (torch.einsum("pk,pkc->pc", tr.sh_basis(d, 3), t(arrays[3])) + 0.5).numpy()
    clamped = ((res < -1e-4) | (res > 1 + 1e-4)) & (tt > 0)[:, None]
    assert clamped[600:900].sum() > 100
    for c in range(3):
        assert not np.any(got["sh"][clamped[:, c], :, c]), c
    assert np.any(got["color"][clamped])  # the post-clamp colour itself still has a gradient


def test_empty_frame(lcgs, dev):
    W, H, P = 128, 96, 2_000
    arrays, pose = scene_arrays("C3", P)
    cam = lcgs.make_camera(*pose, W, H)
    arrays[0][:] = np.array(scenes.CAM_POS, np.float32) - 5.0 * np.array(list(cam.front), np.float32)
    R = np.ones((3, H, W))
    r, got = gpu_backward(lcgs, dev, arrays, pose, W, H, 3, (0.1, 0.2, 0.3), R, list_capacity=1000)
    assert dev.num_rendered() == 0
    for n in got:
        assert not np.any(got[n]), n


def test_differentiable_renderer_image_is_bit_identical(lcgs, dev):
    W, H, P = 320, 180, 4_000
    arrays, pose = scene_arrays("C3", P)
    cam = lcgs.make_camera(*pose, W, H)
    r = lcgs.Renderer(dev, *arrays, W, H, list_capacity=2_000_000, bg_color=(0.2, 0.3, 0.4))
    r.render(cam)
    dr = lcgs.DifferentiableRenderer(dev, W, H, list_capacity=2_000_000, bg_color=(0.2, 0.3, 0.4), keep_means_2d_grad=True)
    leaves = [torch.tensor(a, device="cuda", requires_grad=True) for a in arrays]
    img = dr(*leaves, cam)
    assert img.shape == (3, H, W)
    assert torch.equal(img.detach().view(-1).view(torch.int32), r.img.view(torch.int32))
    R = torch.rand(3, H, W, device="cuda")
    (img * R).sum().backward()
    for x in leaves:
        assert x.grad is not None and x.grad.shape == x.shape and torch.isfinite(x.grad).all()
    assert dr.means_2d_grad is not None and dr.means_2d_grad.shape == (P, 2)
    # the same gradients as the C call on the Renderer's frame
    _, got = gpu_backward(lcgs, dev, arrays, pose, W, H, 3, (0.2, 0.3, 0.4), R.cpu().numpy())
    for n, x in zip(NAMES, leaves):
        rel, _ = metrics(x.grad.cpu().numpy(), got[n])
        assert rel <= 1e-5, (n, rel)
    rel, _ = metrics(dr.means_2d_grad.cpu().numpy(), got["means_2d"])
    assert rel <= 1e-5


def test_two_views_then_one_backward(lcgs, dev):
    W, H, P = 200, 120, 3_000
    arrays, pose = scene_arrays("C3", P)
    pose2 = (tuple(np.array(scenes.CAM_POS) + np.array([0.5, -0.3, 0.2])), pose[1], pose[2])
    cams = [lcgs.make_camera(*p, W, H) for p in (pose, pose2)]
    dr = lcgs.DifferentiableRenderer(dev, W, H, list_capacity=1_000_000)
    Rs = [torch.rand(3, H, W, device="cuda") for _ in cams]

    def grads(views):
        leaves = [torch.tensor(a, device="cuda", requires_grad=True) for a in arrays]
        loss = sum((dr(*leaves, cams[v]) * Rs[v]).sum() for v in views)
        loss.backward()
        return [x.grad.cpu().numpy() for x in leaves]

    both, a, b = grads([0, 1]), grads([0]), grads([1])
    for n, g, ga, gb in zip(NAMES, both, a, b):
        rel, _ = metrics(g, ga + gb)
        assert rel <= 1e-5, (n, rel)


def test_error_paths_and_canaries(lcgs, dev):
    W, H, P = 160, 96, 2_000
    arrays, pose = scene_arrays("C1", P)
    r = lcgs.Renderer(dev, *arrays, W, H, list_capacity=1_000_000)
    vp = lcgs.view_params(lcgs.make_camera(*pose, W, H))
    r.render_async(vp)
    dev.num_rendered()
    dl = torch.rand(3 * W * H, device="cuda")
    pad, canary = 37, 0x7F7F1234
    buf = torch.full((2 * pad + 3 * P,), canary, dtype=torch.int32, device="cuda")
    ref = torch.zeros(3 * P, device="cuda")

    def call(**fields):
        g = lcgs._capi.Grad()
        g.dl_dimg = dl.data_ptr()
        for k, v in fields.items():
            setattr(g, k, v)
        return dev.lib.lcgs_b200_render_backward(dev.ctx, C.byref(r.c_scene), C.byref(vp), C.byref(r.c_frame), C.byref(g), None)

    assert call(grad_pos=ref.data_ptr()) == 0
    assert call(grad_pos=buf.data_ptr() + 4 * pad) == 0
    torch.cuda.synchronize()
    h = buf.cpu().numpy()
    assert (h[:pad] == canary).all() and (h[pad + 3 * P:] == canary).all()
    sub = h[pad:pad + 3 * P].view(np.float32)
    rel, _ = metrics(sub, ref.cpu().numpy())
    assert rel <= 1e-5
    # NULL required pointer, misaligned pointer
    g = lcgs._capi.Grad()
    assert dev.lib.lcgs_b200_render_backward(dev.ctx, C.byref(r.c_scene), C.byref(vp), C.byref(r.c_frame), C.byref(g), None) == -1
    assert call(grad_pos=ref.data_ptr() + 2) == -1
    saved = r.c_frame.conic
    r.c_frame.conic = None
    assert call(grad_pos=ref.data_ptr()) == -1
    r.c_frame.conic = saved
    # a band of tile rows
    r.c_frame.tile_row_begin, r.c_frame.tile_row_end = 0, 3
    assert call(grad_pos=ref.data_ptr()) == -5
    r.c_frame.tile_row_begin, r.c_frame.tile_row_end = 0, -1


def test_run_to_run_spread(lcgs, dev):
    W, H, P = 320, 180, 20_000
    arrays, pose = scene_arrays("C3", P)
    R = np.random.default_rng(3).uniform(-1.0, 1.0, (3, H, W))
    _, a = gpu_backward(lcgs, dev, arrays, pose, W, H, 3, (0.0, 0.0, 0.0), R)
    _, b = gpu_backward(lcgs, dev, arrays, pose, W, H, 3, (0.0, 0.0, 0.0), R)
    spread = {n: metrics(a[n], b[n])[0] for n in a}
    print("run-to-run relative L2 spread", {k: "%.2e" % v for k, v in spread.items()})
    for n, v in spread.items():
        assert v <= 1e-5, (n, v)


def _optimise(lcgs, dev, learn_all, steps, seed=0):
    W, H, P = 128, 96, 1_500
    arrays, pose = scene_arrays("C3", P)
    cam = lcgs.make_camera(*pose, W, H)
    dr = lcgs.DifferentiableRenderer(dev, W, H, list_capacity=1_000_000)
    target = [torch.tensor(a, device="cuda") for a in arrays]
    with torch.no_grad():
        goal = dr(*target, cam).clone()
    g = torch.Generator(device="cpu").manual_seed(seed)
    noise = lambda t, s: (torch.randn(t.shape, generator=g) * s).cuda()  # noqa: E731
    logit = torch.logit(target[4].clamp(1e-4, 1 - 1e-4))
    sh = target[3].clone()
    sh[:, 0] += noise(sh[:, 0], 0.4)
    params = {"sh": sh.requires_grad_(), "logit": (logit + noise(logit, 1.5)).requires_grad_()}
    if learn_all:
        params["pos"] = (target[0] + noise(target[0], 0.01)).requires_grad_()
        params["log_scale"] = (torch.log(target[1]) + noise(target[1], 0.1)).requires_grad_()
        params["rotq"] = (target[2] + noise(target[2], 0.05)).requires_grad_()
    opt = torch.optim.Adam(params.values(), lr=0.02)
    losses = []
    for _ in range(steps):
        opt.zero_grad()
        pos = params.get("pos", target[0])
        scale = torch.exp(params["log_scale"]) if learn_all else target[1]
        rotq = params.get("rotq", target[2])
        img = dr(pos, scale, rotq, params["sh"], torch.sigmoid(params["logit"]), cam)
        loss = ((img - goal) ** 2).mean()
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    return losses


def test_optimisation_recovers_colour_and_opacity(lcgs, dev):
    losses = _optimise(lcgs, dev, learn_all=False, steps=100)
    print("L2 loss %.3e -> %.3e" % (losses[0], losses[-1]))
    assert losses[-1] <= 0.25 * losses[0]


def test_optimisation_of_all_five_arrays_decreases_the_loss(lcgs, dev):
    losses = _optimise(lcgs, dev, learn_all=True, steps=40, seed=1)
    print("L2 loss %.3e -> %.3e" % (losses[0], losses[-1]))
    assert losses[-1] < losses[0]
