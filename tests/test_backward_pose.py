"""The camera-pose gradient on the GPU (lcgs_b200_grad's grad_view / grad_cam_pos, DifferentiableRenderer's
world_to_camera / camera_position) against the float64 torch reference, differentiated with respect to the view
matrix and the camera position.  Bars as in test_backward.py: relative L2 error <= 1e-3 and cosine >= 0.9999."""
import ctypes as C
import shutil

import numpy as np
import pytest
import torch

from luisacomputegaussiansplatting_b200 import scenes
from oracle import oracle as orc

import torch_reference as tr
import torch_reference_aux as tra
import torch_reference_pose as tp
from test_backward import CASES, NAMES, metrics, scene_arrays

pytestmark = pytest.mark.gpu

SPREAD = 1e-5  # run-to-run relative L2 spread of the float atomics (test_backward_edges.py)
VIEW_IDX = [(j // 3) * 4 + j % 3 for j in range(12)]
PER_GAUSSIAN = NAMES + ("means_2d", "conic", "color", "depth")


@pytest.fixture(scope="module")
def lcgs():
    from luisacomputegaussiansplatting_b200 import lcgs as m
    return m


@pytest.fixture(scope="module")
def dev(lcgs):
    d = lcgs.Device(0)
    yield d
    d.close()


def render(lcgs, dev, arrays, pose, W, H, deg=3, bg=(0.0, 0.0, 0.0), aux=False, list_capacity=2_000_000):
    r = lcgs.Renderer(dev, *arrays, W, H, list_capacity=list_capacity, sh_deg=deg, bg_color=bg, aux=aux)
    vp = lcgs.view_params(lcgs.make_camera(*pose, W, H))
    r.render_async(vp)
    dev.num_rendered()
    return r, vp


def backward(lcgs, dev, r, vp, outputs, R=None, RA=None, RD=None):
    """lcgs_b200_render_backward of the frame `r` last rendered, with the outputs named in `outputs` (scene arrays,
    means_2d, conic, color, depth, view, cam_pos) and the loss sum(img R) + sum(alpha RA) + sum(depth plane RD)."""
    P, W, H = r.P, r.W, r.H
    like = dict(zip(NAMES, (r.pos, r.scale, r.rotq, r.sh, r.opacity)))
    shapes = dict(means_2d=(P, 2), conic=(P, 3), color=(P, 3), depth=(P,), view=(16,), cam_pos=(3,))
    out = {n: (torch.zeros_like(like[n]) if n in like else torch.zeros(shapes[n], device="cuda")) for n in outputs}
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()  # noqa: E731
    dl = t(R) if R is not None else torch.zeros(3 * W * H, device="cuda")
    planes = [None if a is None else t(a) for a in (RA, RD)]
    g = lcgs._capi.Grad()
    g.dl_dimg = dl.data_ptr()
    g.dl_dalpha, g.dl_ddepth = [None if p is None else p.data_ptr() for p in planes]
    for n in out:
        setattr(g, "grad_" + n, out[n].data_ptr())
    dev.check(dev.lib.lcgs_b200_render_backward(dev.ctx, C.byref(r.c_scene), C.byref(vp), C.byref(r.c_frame), C.byref(g), None))
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def pose_reference(arrays, pose, W, H, deg=3, bg=(0.0, 0.0, 0.0), R=None, RA=None, RD=None):
    """(dL/dview [16], dL/dcam_pos [3]) of the float64 reference for the same loss as backward()."""
    vp = orc.view_params(orc.make_camera(*pose, W, H))
    fr = orc.forward(*arrays, vp, bg=bg, sh_deg=deg)
    V, cp = tp.vp_pose(vp)
    t = [torch.from_numpy(np.asarray(a, np.float64)) for a in arrays]
    dec = tr.decisions(fr, arrays[4], W, H)
    means, conic, color, vz = tp.preprocess(*t[:4], vp, V, cp, deg)
    img, alpha, dmap = tra.render_aux(means, conic, color, vz, t[4], dec, W, H, bg)
    f = lambda a: torch.from_numpy(np.asarray(a, np.float64))  # noqa: E731
    loss = torch.zeros((), dtype=tr.F64)
    if R is not None:
        loss = loss + (img * f(R).reshape(3, H, W)).sum()
    if RA is not None:
        loss = loss + (alpha * f(RA).reshape(H, W)).sum()
    if RD is not None:
        loss = loss + (dmap * f(RD).reshape(H, W)).sum()
    loss.backward()
    return V.grad.numpy(), (np.zeros(3) if cp.grad is None else cp.grad.numpy()), fr


def check_pose(lcgs, dev, key, P, W, H, deg=3, bg=(0.0, 0.0, 0.0), losses=("img",), seed=0):
    arrays, pose = scene_arrays(key, P, deg)
    rng = np.random.default_rng(seed)
    R = rng.uniform(-1.0, 1.0, (3, H, W)) if "img" in losses else None
    RA = rng.uniform(-1.0, 1.0, (H, W)) if "alpha" in losses else None
    RD = rng.uniform(-1.0, 1.0, (H, W)) if "depth" in losses else None
    r, vp = render(lcgs, dev, arrays, pose, W, H, deg, bg, aux=RA is not None or RD is not None)
    got = backward(lcgs, dev, r, vp, ("view", "cam_pos"), R, RA, RD)
    gv, gc, _ = pose_reference(arrays, pose, W, H, deg, bg, R, RA, RD)
    assert not got["view"][[3, 7, 11, 15]].any()
    errs = {n: metrics(got[n], want) for n, want in (("view", gv), ("cam_pos", gc))}
    print(key, P, W, H, "deg", deg, "bg", bg, losses, {k: "%.2e / %.7f" % v for k, v in errs.items()})
    for n, (rel, cos) in errs.items():
        assert rel <= 1e-3 and cos >= 0.9999, (n, rel, cos)
    if deg == 0:
        assert not got["cam_pos"].any()
    return got


@pytest.mark.parametrize("key,P,W,H", CASES)
def test_pose_gradient_matches_the_reference(lcgs, dev, key, P, W, H):
    check_pose(lcgs, dev, key, P, W, H)


@pytest.mark.parametrize("deg", [0, 1, 2])
def test_pose_gradient_sh_degrees(lcgs, dev, deg):
    check_pose(lcgs, dev, "C3", 3_000, 256, 144, deg=deg)


def test_pose_gradient_with_a_background(lcgs, dev):
    check_pose(lcgs, dev, "C1", 3_000, 200, 200, bg=(0.3, 0.6, 0.15))


@pytest.mark.parametrize("losses", [("depth",), ("alpha",), ("img", "alpha", "depth")])
def test_pose_gradient_of_the_planes(lcgs, dev, losses):
    check_pose(lcgs, dev, "C3", 4_000, 320, 180, losses=losses, seed=1)


@pytest.fixture(scope="module")
def gm_pose(tmp_path_factory):
    """The host builds of the pose terms (tests/grad_mirror/grad_mirror_pose.cpp), float and double."""
    if shutil.which("g++") is None:
        pytest.skip("no C++ compiler")
    from test_backward_pose_cpu import build_mirror
    return build_mirror(tmp_path_factory.mktemp("gmp"), False), build_mirror(tmp_path_factory.mktemp("gmp64"), True)


def test_reduction_at_full_size(lcgs, dev, gm_pose):
    """The full C3 frame: the GPU's pose gradient against the host mirror's per-Gaussian terms from the GPU's own 2D
    gradients (means, conic, colour, depth), summed in float64.  This isolates the reduction from the blend: against
    the float build the kernel's own arithmetic, against the double build the exact algebra."""
    from test_backward_pose_cpu import mirror_terms

    sc, cfg = scenes.make_config_scene("C3")
    W, H = cfg.W, cfg.H
    arrays = [np.ascontiguousarray(a, np.float32) for a in (sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity)]
    pose = (scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world))
    r, vp = render(lcgs, dev, arrays, pose, W, H, aux=True, list_capacity=20_000_000)
    rng = np.random.default_rng(2)
    R = rng.uniform(-1.0, 1.0, (3, H, W)).astype(np.float32)
    RD = rng.uniform(-0.1, 0.1, (H, W)).astype(np.float32)
    got = backward(lcgs, dev, r, vp, ("means_2d", "conic", "color", "depth", "view", "cam_pos"), R=R, RD=RD)
    vis = r.tiles_touched.cpu().numpy() > 0
    n = int(vis.sum())
    g2 = np.zeros((n, 12), np.float32)
    g2[:, 0:2], g2[:, 2:5] = got["means_2d"][vis], got["conic"][vis]
    g2[:, 6:9], g2[:, 9] = got["color"][vis], got["depth"][vis]
    sel = [np.ascontiguousarray(a[vis]) for a in arrays[:4]]
    gpu = np.concatenate([got["view"][VIEW_IDX], got["cam_pos"]])
    errs = {}
    for name, lib, double in (("float", gm_pose[0], False), ("double", gm_pose[1], True)):
        want = mirror_terms(lib, double, n, 3, *sel, 1.0, vp, g2).astype(np.float64).sum(0)
        errs[name] = (metrics(gpu[:12], want[:12])[0], metrics(gpu[12:], want[12:])[0])
    print("P", r.P, "visible", n, "view / cam_pos rel L2 against the float mirror %.2e / %.2e, the double mirror %.2e / %.2e"
          % (*errs["float"], *errs["double"]))
    for name in errs:
        assert max(errs[name]) <= 1e-4, (name, errs[name])


def _noisy_extra(arrays, pose, W, H, lcgs, n=300):
    """The scene plus n Gaussians behind the camera and n far off screen (none touches a tile)."""
    cam = lcgs.make_camera(*pose, W, H)
    front, right = np.array(list(cam.front), np.float32), np.array(list(cam.right), np.float32)
    campos = np.array(scenes.CAM_POS, np.float32)
    extra = [np.concatenate([a, a[:2 * n]]) for a in arrays]
    extra[0][-2 * n:-n] = campos - 3.0 * front
    extra[0][-n:] = campos + 3.0 * front + 50.0 * right
    return [np.ascontiguousarray(a) for a in extra]


def test_pose_outputs_change_nothing_else(lcgs, dev):
    W, H, P = 320, 180, 20_000
    arrays, pose = scene_arrays("C3", P)
    rng = np.random.default_rng(3)
    R, RD = rng.uniform(-1.0, 1.0, (3, H, W)), rng.uniform(-0.1, 0.1, (H, W))
    r, vp = render(lcgs, dev, arrays, pose, W, H, aux=True)
    plain = [backward(lcgs, dev, r, vp, PER_GAUSSIAN, R, RD=RD) for _ in range(2)]
    full = [backward(lcgs, dev, r, vp, PER_GAUSSIAN + ("view", "cam_pos"), R, RD=RD) for _ in range(2)]
    for n in PER_GAUSSIAN:
        spread = metrics(plain[0][n], plain[1][n])[0]
        rel = metrics(full[0][n], plain[0][n])[0]
        print("%s: with / without the pose %.2e, repeats %.2e" % (n, rel, spread))
        assert rel <= max(SPREAD, 3.0 * spread), (n, rel, spread)
    for n in ("view", "cam_pos"):
        rel = metrics(full[1][n], full[0][n])[0]
        print("%s run-to-run %.2e" % (n, rel))
        assert rel <= SPREAD, (n, rel)
    # tracking only: no scene gradient, the same pose gradient
    track = backward(lcgs, dev, r, vp, ("view", "cam_pos"), R, RD=RD)
    for n in ("view", "cam_pos"):
        assert metrics(track[n], full[0][n])[0] <= SPREAD, n
    # Gaussians that touch no tile add nothing
    more = _noisy_extra(arrays, pose, W, H, lcgs)
    r2, _ = render(lcgs, dev, more, pose, W, H, aux=True)
    assert not r2.tiles_touched.cpu().numpy()[P:].any()
    extra = backward(lcgs, dev, r2, vp, ("view", "cam_pos"), R, RD=RD)
    for n in ("view", "cam_pos"):
        rel = metrics(extra[n], full[0][n])[0]
        print("%s with %d idle Gaussians added %.2e" % (n, len(more[0]) - P, rel))
        assert rel <= SPREAD, (n, rel)


def test_empty_frame_and_error_paths(lcgs, dev):
    W, H, P = 128, 96, 2_000
    arrays, pose = scene_arrays("C3", P)
    cam = lcgs.make_camera(*pose, W, H)
    pad, canary = 5, 0x7F7F1234
    buf = torch.full((4 * pad + 19,), canary, dtype=torch.int32, device="cuda")
    view_at, cam_at = buf.data_ptr() + 4 * pad, buf.data_ptr() + 4 * (3 * pad + 16)  # [pad][16][2 pad][3][pad]
    dl = torch.rand(3 * W * H, device="cuda")

    def call(r, vp, **fields):
        g = lcgs._capi.Grad()
        g.dl_dimg = dl.data_ptr()
        for k, v in fields.items():
            setattr(g, k, v)
        return dev.lib.lcgs_b200_render_backward(dev.ctx, C.byref(r.c_scene), C.byref(vp), C.byref(r.c_frame), C.byref(g), None)

    def check_canaries():
        torch.cuda.synchronize()
        h = buf.cpu().numpy()
        assert (h[:pad] == canary).all() and (h[pad + 16:3 * pad + 16] == canary).all() and (h[3 * pad + 19:] == canary).all()
        return h[pad:pad + 16].view(np.float32), h[3 * pad + 16:3 * pad + 19].view(np.float32)

    # every Gaussian behind the camera: an empty frame gives zeros
    empty = [a.copy() for a in arrays]
    empty[0][:] = np.array(scenes.CAM_POS, np.float32) - 5.0 * np.array(list(cam.front), np.float32)
    r, vp = render(lcgs, dev, empty, pose, W, H, list_capacity=1000)
    assert dev.num_rendered() == 0
    assert call(r, vp, grad_view=view_at, grad_cam_pos=cam_at) == 0
    v, c = check_canaries()
    assert not v.any() and not c.any()
    # a scene: the same values as through plain buffers, nothing written outside
    r, vp = render(lcgs, dev, arrays, pose, W, H)
    ref = torch.zeros(19, device="cuda")
    assert call(r, vp, grad_view=ref.data_ptr(), grad_cam_pos=ref.data_ptr() + 64) == 0
    assert call(r, vp, grad_view=view_at, grad_cam_pos=cam_at) == 0
    v, c = check_canaries()
    refh = ref.cpu().numpy()
    assert metrics(v, refh[:16])[0] <= SPREAD and metrics(c, refh[16:])[0] <= SPREAD and v.any()
    # one output alone
    assert call(r, vp, grad_cam_pos=cam_at) == 0
    check_canaries()
    # misaligned, and a band of tile rows
    assert call(r, vp, grad_view=view_at + 2) == -1
    assert call(r, vp, grad_cam_pos=cam_at + 1) == -1
    r.c_frame.tile_row_begin, r.c_frame.tile_row_end = 0, 3
    assert call(r, vp, grad_view=view_at) == -5
    r.c_frame.tile_row_begin, r.c_frame.tile_row_end = 0, -1
    check_canaries()
    # a scene of no Gaussian at all
    buf[pad:pad + 16] = 1
    r.c_scene.num_gaussians = 0
    assert call(r, vp, grad_view=view_at, grad_cam_pos=cam_at) == 0
    r.c_scene.num_gaussians = P
    v, c = check_canaries()
    assert not v.any() and not c.any()


def _leaves(arrays, grad=True):
    return [torch.tensor(a, device="cuda", requires_grad=grad) for a in arrays]


def test_differentiable_renderer_with_the_camera_pose(lcgs, dev):
    W, H, P = 320, 180, 4_000
    arrays, pose = scene_arrays("C3", P)
    cam = lcgs.make_camera(*pose, W, H)
    bg = (0.2, 0.3, 0.4)
    dr = lcgs.DifferentiableRenderer(dev, W, H, list_capacity=2_000_000, bg_color=bg)
    R = torch.rand(3, H, W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
    plain = _leaves(arrays)
    img0 = dr(*plain, cam)
    (img0 * R).sum().backward()
    # the camera's own pose as tensors: the same image, the same scene gradients
    posed = _leaves(arrays)
    M = torch.tensor(lcgs.world_to_camera(cam), dtype=torch.float64, requires_grad=True)
    cp = torch.tensor(list(cam.position), dtype=torch.float32, requires_grad=True)
    img1 = dr(*posed, cam, world_to_camera=M, camera_position=cp)
    assert torch.equal(img1.detach().view(torch.int32), img0.detach().view(torch.int32))
    (img1 * R).sum().backward()
    for n, a, b in zip(NAMES, plain, posed):
        assert metrics(b.grad.cpu().numpy(), a.grad.cpu().numpy())[0] <= SPREAD, n
    assert M.grad is not None and M.grad.dtype == torch.float64 and M.grad.device.type == "cpu"
    assert not M.grad[3].any() and cp.grad is not None and cp.grad.device.type == "cpu"
    # the gradient on M with the default camera_position, against the reference chained through torch
    M2 = torch.tensor(lcgs.world_to_camera(cam), dtype=torch.float64, requires_grad=True)
    img2 = dr(*[torch.tensor(a, device="cuda") for a in arrays], cam, world_to_camera=M2)
    assert float((img2.detach() - img0.detach()).abs().max()) <= 1e-5  # cam_pos from M differs in the last bits
    (img2 * R).sum().backward()
    vp = orc.view_params(orc.make_camera(*pose, W, H))
    fr = orc.forward(*arrays, vp, bg=bg)
    Mr = M2.detach().clone().requires_grad_()
    ref = tp.forward(*[torch.from_numpy(np.asarray(a, np.float64)) for a in arrays], vp, fr, Mr.T.reshape(16),
                     -torch.linalg.solve(Mr[:3, :3], Mr[:3, 3]), bg=bg)
    (ref * R.double().cpu()).sum().backward()
    rel, cos = metrics(M2.grad.numpy(), Mr.grad.numpy())
    print("dL/dM rel L2 %.2e cosine %.7f" % (rel, cos))
    assert rel <= 1e-3 and cos >= 0.9999


def test_differentiable_renderer_depth_loss_on_the_pose(lcgs, dev):
    W, H, P = 256, 144, 4_000
    arrays, pose = scene_arrays("C3", P)
    cam = lcgs.make_camera(*pose, W, H)
    dr = lcgs.DifferentiableRenderer(dev, W, H, list_capacity=2_000_000, aux=True)
    M = torch.tensor(lcgs.world_to_camera(cam), dtype=torch.float64, requires_grad=True)
    RD = torch.rand(H, W, dtype=torch.float64, generator=torch.Generator().manual_seed(4)) - 0.5
    img, alpha, depth = dr(*[torch.tensor(a, device="cuda") for a in arrays], cam, world_to_camera=M)
    (depth.double().cpu() * RD).sum().backward()  # a depth-plane loss alone: img and alpha get no gradient
    vp = orc.view_params(orc.make_camera(*pose, W, H))
    fr = orc.forward(*arrays, vp)
    Mr = M.detach().clone().requires_grad_()
    t = [torch.from_numpy(np.asarray(a, np.float64)) for a in arrays]
    means, conic, color, vz = tp.preprocess(*t[:4], vp, Mr.T.reshape(16), -torch.linalg.solve(Mr[:3, :3], Mr[:3, 3]))
    _, _, dmap = tra.render_aux(means, conic, color, vz, t[4], tr.decisions(fr, arrays[4], W, H), W, H)
    (dmap * RD).sum().backward()
    rel, cos = metrics(M.grad.numpy(), Mr.grad.numpy())
    print("depth loss dL/dM rel L2 %.2e cosine %.7f" % (rel, cos))
    assert rel <= 1e-3 and cos >= 0.9999


def _hat(xi):
    """4x4 matrix of the twist xi = (omega, v)."""
    w, v = xi[:3], xi[3:]
    z = torch.zeros((), dtype=xi.dtype)
    return torch.stack([torch.stack([z, -w[2], w[1], v[0]]), torch.stack([w[2], z, -w[0], v[1]]),
                        torch.stack([-w[1], w[0], z, v[2]]), torch.stack([z, z, z, z])])


def test_pose_refinement_recovers_a_perturbed_camera(lcgs, dev):
    """Render a target from the true camera, perturb the pose by 1 degree and 2 % of the camera distance, and refine a
    twist with Adam against the image loss, the scene frozen.  Measured on a B200: rotation 1.0 -> below 1e-4 degrees
    and translation 0.108 -> 0.00027 (about 400x) in 150 steps; the bar asks for 5x each."""
    W, H, P = 256, 144, 20_000
    arrays, pose = scene_arrays("C3", P)
    cam = lcgs.make_camera(*pose, W, H)
    dr = lcgs.DifferentiableRenderer(dev, W, H, list_capacity=4_000_000)
    scene = [torch.tensor(a, device="cuda") for a in arrays]
    M_true = torch.tensor(lcgs.world_to_camera(cam), dtype=torch.float64)
    with torch.no_grad():
        goal = dr(*scene, cam).clone()
    g = torch.Generator().manual_seed(7)
    axis = torch.randn(3, generator=g, dtype=torch.float64)
    axis /= axis.norm()
    dist = float(np.linalg.norm(np.subtract(scenes.CAM_POS, scenes.CAM_TARGET)))
    shift = torch.randn(3, generator=g, dtype=torch.float64)
    shift *= 0.02 * dist / shift.norm()
    M0 = torch.linalg.matrix_exp(_hat(torch.cat([axis * np.deg2rad(1.0), shift]))) @ M_true

    def errors(M):
        dR = M[:3, :3] @ M_true[:3, :3].T
        ang = float(torch.rad2deg(torch.arccos(((torch.trace(dR) - 1) / 2).clamp(-1, 1))))
        c = -torch.linalg.solve(M[:3, :3], M[:3, 3])
        c_true = -torch.linalg.solve(M_true[:3, :3], M_true[:3, 3])
        return ang, float((c - c_true).norm())

    xi = torch.zeros(6, dtype=torch.float64, requires_grad=True)
    opt = torch.optim.Adam([xi], lr=5e-3)
    sched = torch.optim.lr_scheduler.ExponentialLR(opt, gamma=0.98)
    curve = []
    for step in range(150):
        opt.zero_grad()
        M = torch.linalg.matrix_exp(_hat(xi)) @ M0
        loss = ((dr(*scene, cam, world_to_camera=M) - goal) ** 2).mean()
        loss.backward()
        opt.step()
        sched.step()
        if step % 10 == 0 or step == 149:
            curve.append((step, float(loss.detach()), *errors(M.detach())))
    M = (torch.linalg.matrix_exp(_hat(xi)) @ M0).detach()
    a0, t0 = errors(M0)
    a1, t1 = errors(M)
    for row in curve:
        print("step %3d loss %.3e rotation %.4f deg translation %.5f" % row)
    print("rotation %.4f -> %.4f deg, translation %.5f -> %.5f (camera distance %.3f)" % (a0, a1, t0, t1, dist))
    assert a1 <= a0 / 5 and t1 <= t0 / 5
