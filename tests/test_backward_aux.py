"""The backward through the alpha and depth planes on the GPU (lcgs_b200_render_backward with dl_dalpha / dl_ddepth,
lcgs.DifferentiableRenderer(aux=True)) against the float64 torch reference with the planes
(tests/torch_reference_aux.py), for L = sum(img * R) + sum(alpha * Ra) + sum(depth * Rd), R, Ra, Rd fixed random
tensors.  Bars per gradient tensor as in test_backward.py: relative L2 error <= 1e-3 and cosine >= 0.9999."""
import ctypes as C

import numpy as np
import pytest
import torch

from luisacomputegaussiansplatting_b200 import scenes
from oracle import oracle as orc

import torch_reference_aux as tra
import torch_reference as tr
from test_backward import CASES, NAMES, assert_close, gpu_backward, metrics, scene_arrays

pytestmark = pytest.mark.gpu

OUTS = NAMES + ("means_2d", "conic", "color", "depth")


@pytest.fixture(scope="module")
def lcgs():
    from luisacomputegaussiansplatting_b200 import lcgs as m
    return m


@pytest.fixture(scope="module")
def dev(lcgs):
    d = lcgs.Device(0)
    yield d
    d.close()


def cuda32(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def render_aux_frame(lcgs, dev, arrays, pose, W, H, deg, bg, list_capacity=2_000_000, scale_modifier=1.0,
                     prepare_scene=True):
    r = lcgs.Renderer(dev, *arrays, W, H, list_capacity=list_capacity, sh_deg=deg, bg_color=bg, aux=True,
                      scale_modifier=scale_modifier, prepare_scene=prepare_scene)
    vp = lcgs.view_params(lcgs.make_camera(*pose, W, H))
    r.render_async(vp)
    dev.num_rendered()
    return r, vp


def grad_struct(lcgs, P, dl, da, dd, fill=0.0):
    """A Grad with every output requested (buffers pre-filled with `fill`); returns (struct, outputs, inputs kept)."""
    out = {n: torch.full((P, k), fill, device="cuda") for n, k in
           (("pos", 3), ("scale", 3), ("rotq", 4), ("opacity", 1), ("means_2d", 2), ("conic", 3), ("color", 3), ("depth", 1))}
    g = lcgs._capi.Grad()
    g.dl_dimg = dl.data_ptr()
    g.dl_dalpha = None if da is None else da.data_ptr()
    g.dl_ddepth = None if dd is None else dd.data_ptr()
    return g, out


def gpu_backward_aux(lcgs, dev, arrays, pose, W, H, deg, bg, R, Ra, Rd, list_capacity=2_000_000, scale_modifier=1.0,
                     prepare_scene=True):
    """Render with Renderer(aux=True), then lcgs_b200_render_backward with every output; Ra / Rd None = NULL."""
    r, vp = render_aux_frame(lcgs, dev, arrays, pose, W, H, deg, bg, list_capacity, scale_modifier, prepare_scene)
    dl, da, dd = cuda32(R), cuda32(Ra), cuda32(Rd)
    g, out = grad_struct(lcgs, r.P, dl, da, dd)
    out["sh"] = torch.zeros_like(r.sh)
    for n in out:
        setattr(g, "grad_" + n, out[n].data_ptr())
    dev.check(dev.lib.lcgs_b200_render_backward(dev.ctx, C.byref(r.c_scene), C.byref(vp), C.byref(r.c_frame), C.byref(g), None))
    torch.cuda.synchronize()
    got = {k: v.cpu().numpy().reshape(-1) if k in ("opacity", "depth") else v.cpu().numpy() for k, v in out.items()}
    return r, got


def reference_aux(arrays, pose, W, H, deg, bg, R, Ra, Rd, scale_modifier=1.0):
    vp = orc.view_params(orc.make_camera(*pose, W, H))
    fr = orc.forward(arrays[0], arrays[1], arrays[2], arrays[3], arrays[4], vp, bg=bg, sh_deg=deg,
                     scale_modifier=scale_modifier)
    L = [tr.leaf(a) for a in arrays]
    img, alpha, dmap, (means, conic, color, depth) = tra.forward_aux(*L, vp, fr, deg=deg, bg=bg,
                                                                     scale_modifier=scale_modifier)
    t = lambda a: torch.from_numpy(np.asarray(a, np.float64))  # noqa: E731
    loss = (img * t(R)).sum()
    if Ra is not None:
        loss = loss + (alpha * t(Ra)).sum()
    if Rd is not None:
        loss = loss + (dmap * t(Rd)).sum()
    loss.backward()
    want = {n: x.grad.numpy() for n, x in zip(NAMES, L)}
    # without a depth loss the blend's view-depth input is not on the graph
    dz = depth.grad.numpy() if depth.grad is not None else np.zeros(depth.shape)
    want.update(means_2d=means.grad.numpy(), conic=conic.grad.numpy(), color=color.grad.numpy(), depth=dz)
    return fr, want


def check_case(lcgs, dev, key, P, W, H, deg=3, bg=(0.0, 0.0, 0.0), dense=False, seed=0, planes="both", image=True):
    arrays, pose = scene_arrays(key, P, deg, dense)
    rng = np.random.default_rng(seed)
    R = rng.uniform(-1.0, 1.0, (3, H, W)) if image else np.zeros((3, H, W))
    Ra = rng.uniform(-1.0, 1.0, (H, W)) if planes in ("both", "alpha") else None
    Rd = rng.uniform(-1.0, 1.0, (H, W)) if planes in ("both", "depth") else None
    r, got = gpu_backward_aux(lcgs, dev, arrays, pose, W, H, deg, bg, R, Ra, Rd)
    fr, want = reference_aux(arrays, pose, W, H, deg, bg, R, Ra, Rd)
    assert np.array_equal(r.tiles_touched.cpu().numpy().view(np.uint32), fr.tiles_touched)
    errs = {}
    for n in want:
        if n == "color" and not image:
            assert not np.any(got[n]), n  # no image loss: the colour has no gradient
            continue
        if n == "depth" and Rd is None:
            assert not np.any(got[n]), n  # grad_depth without dl_ddepth is all zeros
            continue
        assert_close(n, got[n], want[n], errs)
    idle = fr.tiles_touched == 0
    for n in got:
        assert not np.any(got[n][idle]), n
    print(key, P, W, H, "deg", deg, "bg", bg, "dense" if dense else "", planes, "image" if image else "no image",
          {k: "%.2e / %.7f" % v for k, v in errs.items()})
    return got, want, fr


@pytest.mark.parametrize("key,P,W,H", CASES)
def test_aux_gradients_match_the_reference(lcgs, dev, key, P, W, H):
    check_case(lcgs, dev, key, P, W, H)


@pytest.mark.parametrize("planes", ["alpha", "depth"])
def test_one_plane_without_an_image_loss(lcgs, dev, planes):
    check_case(lcgs, dev, "C3", 4_000, 320, 180, planes=planes, image=False, seed=1)


def test_background_and_sh_degree_0(lcgs, dev):
    check_case(lcgs, dev, "C1", 3_000, 200, 200, deg=0, bg=(0.3, 0.6, 0.15), seed=2)


def test_dense_saturating_scene(lcgs, dev):
    _, _, fr = check_case(lcgs, dev, "C3", 6_000, 160, 96, dense=True, seed=3)
    assert fr.n_examined.mean() < np.diff(fr.ranges.astype(np.int64), axis=1).mean()


def test_empty_frame(lcgs, dev):
    W, H, P = 128, 96, 2_000
    arrays, pose = scene_arrays("C3", P)
    cam = lcgs.make_camera(*pose, W, H)
    arrays[0][:] = np.array(scenes.CAM_POS, np.float32) - 5.0 * np.array(list(cam.front), np.float32)
    ones = np.ones((H, W))
    r, got = gpu_backward_aux(lcgs, dev, arrays, pose, W, H, 3, (0.1, 0.2, 0.3), np.ones((3, H, W)), ones, ones,
                              list_capacity=1000)
    assert dev.num_rendered() == 0
    for n in got:
        assert not np.any(got[n]), n


def test_null_plane_gradients_equal_the_plain_backward(lcgs, dev):
    """An aux-rendered frame with dl_dalpha = dl_ddepth = NULL takes the image-only path: the plain backward's
    gradients (within the run-to-run bar) and a zero grad_depth, written over a NaN-filled buffer."""
    W, H, P = 320, 180, 4_000
    arrays, pose = scene_arrays("C3", P)
    R = np.random.default_rng(4).uniform(-1.0, 1.0, (3, H, W))
    _, plain = gpu_backward(lcgs, dev, arrays, pose, W, H, 3, (0.0, 0.0, 0.0), R)
    r, vp = render_aux_frame(lcgs, dev, arrays, pose, W, H, 3, (0.0, 0.0, 0.0))
    dl = cuda32(R)
    g, out = grad_struct(lcgs, P, dl, None, None, fill=float("nan"))
    out["sh"] = torch.zeros_like(r.sh)
    for n in out:
        setattr(g, "grad_" + n, out[n].data_ptr())
    dev.check(dev.lib.lcgs_b200_render_backward(dev.ctx, C.byref(r.c_scene), C.byref(vp), C.byref(r.c_frame), C.byref(g), None))
    torch.cuda.synchronize()
    assert torch.equal(out["depth"], torch.zeros_like(out["depth"]))
    for n in plain:
        rel, _ = metrics(out[n].cpu().numpy().reshape(plain[n].shape), plain[n])
        assert rel <= 1e-5, (n, rel)


def test_error_paths_and_canaries(lcgs, dev):
    W, H, P = 160, 96, 2_000
    arrays, pose = scene_arrays("C1", P)
    r, vp = render_aux_frame(lcgs, dev, arrays, pose, W, H, 3, (0.0, 0.0, 0.0), list_capacity=1_000_000)
    plain = lcgs.Renderer(dev, *arrays, W, H, list_capacity=1_000_000)
    plain.render_async(vp)
    dev.num_rendered()
    dl = torch.rand(3 * W * H, device="cuda")
    da = torch.rand(W * H + 1, device="cuda")
    dd = torch.rand(W * H + 1, device="cuda")
    pad, canary = 37, 0x7F7F1234
    buf = torch.full((2 * pad + P,), canary, dtype=torch.int32, device="cuda")
    ref = torch.zeros(P, device="cuda")

    def call(frame=r, **fields):
        g = lcgs._capi.Grad()
        g.dl_dimg = dl.data_ptr()
        for k, v in fields.items():
            setattr(g, k, v)
        return dev.lib.lcgs_b200_render_backward(dev.ctx, C.byref(frame.c_scene), C.byref(vp), C.byref(frame.c_frame),
                                                 C.byref(g), None)

    planes = dict(dl_dalpha=da.data_ptr(), dl_ddepth=dd.data_ptr())
    assert call(grad_depth=ref.data_ptr(), **planes) == 0
    assert call(grad_depth=buf.data_ptr() + 4 * pad, **planes) == 0
    torch.cuda.synchronize()
    h = buf.cpu().numpy()
    assert (h[:pad] == canary).all() and (h[pad + P:] == canary).all()
    rel, _ = metrics(h[pad:pad + P].view(np.float32), ref.cpu().numpy())
    assert rel <= 1e-5
    assert np.any(h[pad:pad + P].view(np.float32) != 0)
    # a plane gradient without its plane: a frame rendered without aux, or with the plane / the depth taken away
    assert call(frame=plain, dl_dalpha=da.data_ptr()) == -1
    assert call(frame=plain, dl_ddepth=dd.data_ptr()) == -1
    for field, want in (("target_alpha", dict(dl_dalpha=da.data_ptr())), ("target_depth", dict(dl_ddepth=dd.data_ptr())),
                        ("depth", dict(dl_ddepth=dd.data_ptr()))):
        saved = getattr(r.c_frame, field)
        setattr(r.c_frame, field, None)
        assert call(**want) == -1, field
        setattr(r.c_frame, field, saved)
    # the other plane's absence is fine
    saved = r.c_frame.target_depth
    r.c_frame.target_depth = None
    assert call(dl_dalpha=da.data_ptr()) == 0
    r.c_frame.target_depth = saved
    # misaligned pointers
    assert call(dl_dalpha=da.data_ptr() + 2) == -1
    assert call(dl_ddepth=dd.data_ptr() + 2) == -1
    assert call(grad_depth=ref.data_ptr() + 2, **planes) == -1
    # a band of tile rows
    r.c_frame.tile_row_begin, r.c_frame.tile_row_end = 0, 3
    assert call(**planes) == -5
    r.c_frame.tile_row_begin, r.c_frame.tile_row_end = 0, -1
    torch.cuda.synchronize()


def test_run_to_run_spread(lcgs, dev):
    W, H, P = 320, 180, 20_000
    arrays, pose = scene_arrays("C3", P)
    rng = np.random.default_rng(3)
    R, Ra, Rd = rng.uniform(-1.0, 1.0, (3, H, W)), rng.uniform(-1.0, 1.0, (H, W)), rng.uniform(-1.0, 1.0, (H, W))
    _, a = gpu_backward_aux(lcgs, dev, arrays, pose, W, H, 3, (0.0, 0.0, 0.0), R, Ra, Rd)
    _, b = gpu_backward_aux(lcgs, dev, arrays, pose, W, H, 3, (0.0, 0.0, 0.0), R, Ra, Rd)
    spread = {n: metrics(a[n], b[n])[0] for n in a}
    print("run-to-run relative L2 spread", {k: "%.2e" % v for k, v in spread.items()})
    for n, v in spread.items():
        assert v <= 1e-5, (n, v)


# ---- DifferentiableRenderer(aux=True) -------------------------------------------------------------------------------

def test_differentiable_renderer_outputs_are_bit_identical(lcgs, dev):
    W, H, P = 320, 180, 4_000
    arrays, pose = scene_arrays("C3", P)
    cam = lcgs.make_camera(*pose, W, H)
    bg = (0.2, 0.3, 0.4)
    r = lcgs.Renderer(dev, *arrays, W, H, list_capacity=2_000_000, bg_color=bg, aux=True)
    r.render(cam)
    plain = lcgs.DifferentiableRenderer(dev, W, H, list_capacity=2_000_000, bg_color=bg)
    dr = lcgs.DifferentiableRenderer(dev, W, H, list_capacity=2_000_000, bg_color=bg, aux=True)
    leaves = [torch.tensor(a, device="cuda") for a in arrays]
    with torch.no_grad():
        img0 = plain(*leaves, cam)
        img, alpha, depth = dr(*leaves, cam)
    bits = lambda t: t.contiguous().view(-1).view(torch.int32)  # noqa: E731
    assert img.shape == (3, H, W) and alpha.shape == (H, W) and depth.shape == (H, W)
    assert torch.equal(bits(img), bits(img0)) and torch.equal(bits(img), bits(r.image()))
    assert torch.equal(bits(alpha), bits(r.alpha())) and torch.equal(bits(depth), bits(r.depth_map()))
    assert float(alpha.max()) > 0.5


def test_differentiable_renderer_expected_depth_loss_matches_the_reference(lcgs, dev):
    W, H, P, deg = 200, 120, 3_000, 3
    arrays, pose = scene_arrays("C3", P)
    cam = lcgs.make_camera(*pose, W, H)
    dr = lcgs.DifferentiableRenderer(dev, W, H, list_capacity=1_000_000, aux=True)
    leaves = [torch.tensor(a, device="cuda", requires_grad=True) for a in arrays]
    img, alpha, depth = dr(*leaves, cam)
    mask = (alpha > 0.2).detach()
    assert int(mask.sum()) > 100
    target = torch.from_numpy(np.random.default_rng(6).uniform(-0.5, 0.5, (H, W))).float().cuda() + (
        (depth / alpha.clamp_min(1e-3)).detach())

    def loss_of(img, alpha, depth, target, mask):
        ed = depth / torch.where(mask, alpha, torch.ones_like(alpha))
        return ((ed - target) ** 2 * mask).sum() / mask.sum() + 0.1 * img.mean()

    loss_of(img, alpha, depth, target, mask).backward()
    vp = orc.view_params(orc.make_camera(*pose, W, H))
    fr = orc.forward(*arrays, vp, sh_deg=deg)
    L = [tr.leaf(a) for a in arrays]
    rimg, ralpha, rdepth, _ = tra.forward_aux(*L, vp, fr, deg=deg)
    loss_of(rimg, ralpha, rdepth, target.double().cpu(), mask.cpu()).backward()
    errs = {}
    for n, x, y in zip(NAMES, leaves, L):
        assert_close(n, x.grad.cpu().numpy(), y.grad.numpy(), errs)
    print("expected-depth loss", {k: "%.2e / %.7f" % v for k, v in errs.items()})


def test_differentiable_renderer_two_views_then_one_backward(lcgs, dev):
    W, H, P = 200, 120, 3_000
    arrays, pose = scene_arrays("C3", P)
    pose2 = (tuple(np.array(scenes.CAM_POS) + np.array([0.5, -0.3, 0.2])), pose[1], pose[2])
    cams = [lcgs.make_camera(*p, W, H) for p in (pose, pose2)]
    dr = lcgs.DifferentiableRenderer(dev, W, H, list_capacity=1_000_000, aux=True)
    Rs = [(torch.rand(3, H, W, device="cuda"), torch.rand(H, W, device="cuda"), torch.rand(H, W, device="cuda"))
          for _ in cams]

    def grads(views):
        leaves = [torch.tensor(a, device="cuda", requires_grad=True) for a in arrays]
        loss = 0.0
        for v in views:
            img, alpha, depth = dr(*leaves, cams[v])
            loss = loss + (img * Rs[v][0]).sum() + (alpha * Rs[v][1]).sum() + (depth * Rs[v][2]).sum()
        loss.backward()
        return [x.grad.cpu().numpy() for x in leaves]

    both, a, b = grads([0, 1]), grads([0]), grads([1])
    for n, g, ga, gb in zip(NAMES, both, a, b):
        rel, _ = metrics(g, ga + gb)
        assert rel <= 1e-5, (n, rel)


def _fit(lcgs, dev, which, steps):
    """Adam on a perturbed scene against the target scene's own mask (alpha) or depth plane; returns the losses."""
    W, H, P = 128, 96, 1_500
    arrays, pose = scene_arrays("C3", P)
    cam = lcgs.make_camera(*pose, W, H)
    dr = lcgs.DifferentiableRenderer(dev, W, H, list_capacity=1_000_000, aux=True)
    target = [torch.tensor(a, device="cuda") for a in arrays]
    with torch.no_grad():
        _, goal_alpha, goal_depth = [t.clone() for t in dr(*target, cam)]
    g = torch.Generator(device="cpu").manual_seed(0)
    noise = lambda t, s: (torch.randn(t.shape, generator=g) * s).cuda()  # noqa: E731
    logit = torch.logit(target[4].clamp(1e-4, 1 - 1e-4))
    params = {"logit": (logit + noise(logit, 1.5)).requires_grad_()}
    groups = [{"params": [params["logit"]], "lr": 0.02}]
    if which == "depth":
        params["pos"] = (target[0] + noise(target[0], 0.01)).requires_grad_()
        groups.append({"params": [params["pos"]], "lr": 0.002})
    opt = torch.optim.Adam(groups)
    losses = []
    for _ in range(steps):
        opt.zero_grad()
        _, alpha, depth = dr(params.get("pos", target[0]), *target[1:4], torch.sigmoid(params["logit"]), cam)
        loss = ((alpha - goal_alpha) ** 2).mean() if which == "alpha" else ((depth - goal_depth) ** 2).mean()
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    return losses


@pytest.mark.parametrize("which", ["alpha", "depth"])
def test_optimisation_fits_a_mask_and_a_depth_map(lcgs, dev, which):
    losses = _fit(lcgs, dev, which, steps=60)
    print(which, "loss %.3e -> %.3e" % (losses[0], losses[-1]))
    assert min(losses[-5:]) < 0.5 * losses[0]
