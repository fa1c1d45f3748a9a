"""The backward through the alpha and depth planes without a GPU: the float64 reference's planes
(tests/torch_reference_aux.py) against the aux oracle and torch.autograd.gradcheck, the aux per-entry step of
csrc/lcgs_grad.cuh (built with g++ from tests/grad_mirror/grad_mirror_aux.cpp) against autograd on hand-built pixel
lists, the depth term of project_backward (the existing tests/grad_mirror/grad_mirror.cpp with slot kG2Depth set)
against autograd, and the SASS of blend_backward_aux_kernel."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from luisacomputegaussiansplatting_b200 import build, scenes
from oracle import oracle as orc

import aux_oracle
import torch_reference as tr
import torch_reference_aux as tra
from sass_ops import kernel_ops

HERE = os.path.dirname(os.path.abspath(__file__))
MIRROR_SRC = os.path.join(HERE, "grad_mirror", "grad_mirror.cpp")
MIRROR_AUX_SRC = os.path.join(HERE, "grad_mirror", "grad_mirror_aux.cpp")
CXX = ["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-Wno-unknown-pragmas"]

SCENES = [("C3", 4000, 320, 180), ("C1", 3000, 200, 200), ("C3", 1500, 97, 61)]


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def rel_l2(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return float(np.linalg.norm(got - want) / max(np.linalg.norm(want), 1e-30))


def t64(a):
    return torch.from_numpy(np.asarray(a, np.float64))


@pytest.mark.parametrize("key,P,W,H", SCENES)
def test_reference_planes_match_the_aux_oracle(key, P, W, H):
    sc, cfg = scenes.make_config_scene(key, P=P)
    vp = orc.view_params(orc.make_camera(scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world), W, H))
    fr = orc.forward(sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, vp)
    want = aux_oracle.blend_aux(W, H, (0.0, 0.0, 0.0), fr.ranges, fr.vals_sorted, fr.means_2d, fr.conic, sc.opacity,
                                fr.color, fr.depth)
    assert want["alpha"].max() > 0.5
    dec = tr.decisions(fr, sc.opacity, W, H)
    img, alpha, dmap = tra.render_aux(t64(fr.means_2d), t64(fr.conic), t64(fr.color), t64(fr.depth), t64(sc.opacity), dec,
                                      W, H)
    assert float(np.abs(img.numpy() - fr.img).max()) <= 1e-5
    assert float(np.abs(alpha.numpy() - want["alpha"]).max()) <= 1e-5
    # depth plane: float32 sums of w * z with z of a few units
    assert float(np.abs(dmap.numpy() - want["depth_map"]).max()) <= 1e-5 * max(1.0, float(np.abs(fr.depth).max()))
    # the whole float64 chain: its view depth is the oracle's
    _, _, _, depth = tr.preprocess(*[t64(a) for a in (sc.pos, sc.scale, sc.rotq, sc.sh)], vp)
    vis = fr.tiles_touched > 0
    assert float(np.abs(depth.numpy()[vis] - fr.depth[vis]).max()) <= 1e-5 * float(np.abs(fr.depth[vis]).max())


def tiny_scene(P=5, seed=3):
    """A few Gaussians in front of the camera, away from every clamp and from the 0.99 cap."""
    rng = np.random.default_rng(seed)
    cam = orc.make_camera((0.0, 0.0, -3.0), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), 32, 32)
    vp = orc.view_params(cam)
    pos = rng.uniform(-0.3, 0.3, (P, 3)).astype(np.float32)
    scale = rng.uniform(0.05, 0.12, (P, 3)).astype(np.float32)
    q = rng.normal(size=(P, 4)).astype(np.float32)
    rotq = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    sh = (rng.normal(size=(P, 16, 3)) * 0.05).astype(np.float32)
    sh[:, 0] = rng.uniform(-0.6, 0.6, (P, 3))
    opacity = rng.uniform(0.2, 0.6, P).astype(np.float32)
    return vp, pos, scale, rotq, sh, opacity


@pytest.mark.parametrize("plane", ["alpha", "depth", "expected_depth"])
def test_reference_gradcheck_of_plane_losses(plane):
    vp, pos, scale, rotq, sh, opacity = tiny_scene()
    fr = orc.forward(pos, scale, rotq, sh, opacity, vp)
    assert fr.num_rendered > 0
    dec = tr.decisions(fr, opacity, 32, 32)
    assert float(opacity.max()) < 0.9
    R = t64(np.random.default_rng(1).uniform(-1.0, 1.0, (32, 32)))
    target = t64(np.random.default_rng(2).uniform(2.5, 3.5, (32, 32)))

    def f(p, s, q, h, o):
        _, alpha, dmap, _ = tra.forward_aux(p, s, q, h, o, vp, fr, dec=dec)
        if plane == "alpha":
            return (alpha * R).sum()
        if plane == "depth":
            return (dmap * R).sum()
        m = alpha > 1e-3
        return ((dmap[m] / alpha[m] - target[m]) ** 2).mean()

    inputs = [tr.leaf(a) for a in (pos, scale, rotq, sh, opacity)]
    assert torch.autograd.gradcheck(f, inputs, eps=1e-6, atol=1e-6, rtol=1e-4)


@pytest.fixture(scope="module")
def gm_aux(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("no C++ compiler")
    so = str(tmp_path_factory.mktemp("grad_mirror_aux") / "libgrad_mirror_aux.so")
    subprocess.run([*CXX, "-fvisibility=hidden", "-x", "c++", MIRROR_AUX_SRC, "-o", so], check=True)
    lib = C.CDLL(so)
    lib.gm_blend_pixel_aux.restype = None
    return lib


def pixel_case(kind, rng, n=12):
    mx, my = rng.uniform(-3, 3, n), rng.uniform(-3, 3, n)
    cn = np.stack([rng.uniform(0.05, 0.4, n), rng.uniform(-0.05, 0.05, n), rng.uniform(0.05, 0.4, n)], 1)
    logo = np.log(rng.uniform(0.1, 0.7, n))
    if kind == "cap":
        logo[[2, 5]] = np.log(1.5)  # o e^power > 0.99 there
        mx[[2, 5]], my[[2, 5]] = 0.01, -0.02
    if kind == "saturate":
        logo[:] = np.log(0.985)
        mx[:], my[:] = rng.uniform(-0.05, 0.05, n), rng.uniform(-0.05, 0.05, n)
    logo[4] = np.log(0.001)  # rejected by the alpha test
    return mx, my, cn, logo, rng.uniform(0, 1, (n, 3)), rng.uniform(1.0, 6.0, n)


@pytest.mark.parametrize("kind", ["plain", "cap", "saturate"])
@pytest.mark.parametrize("weights", ["all", "alpha_only", "depth_only"])
def test_mirror_aux_blend_pixel_matches_autograd(gm_aux, kind, weights):
    """Hand-built pixel lists through the aux step: ordinary entries, an alpha-test reject, the 0.99 cap and a
    saturating entry; with dL/dC = 0 and only dL/dA or only dL/dD non-zero as well."""
    rng = np.random.default_rng(11)
    mx, my, cn, logo, rgb, z = pixel_case(kind, rng)
    n = mx.size
    f = np.float32
    dx, dy = mx.astype(f), my.astype(f)  # pixel at the origin
    a, b, c = (-0.5 * cn[:, 0]).astype(f), (-cn[:, 1]).astype(f), (-0.5 * cn[:, 2]).astype(f)
    power = (a * dx * dx + b * dx * dy + c * dy * dy).astype(f)
    araw = (np.exp(logo) * np.exp(power.astype(np.float64))).astype(f)
    ok = (power <= 0) & (araw >= 1.0 / 255.0)
    e = np.ascontiguousarray(np.stack([dx, dy, a, b, c, ok.astype(f), araw], 1), f)
    G = rng.normal(size=3).astype(f)
    GA, GD = f(rng.normal()), f(rng.normal() * 0.3)
    if weights == "alpha_only":
        G[:], GD = 0.0, f(0.0)
    elif weights == "depth_only":
        G[:], GA = 0.0, f(0.0)
    # decisions in float64, as the reference does
    alpha = np.minimum(0.99, araw.astype(np.float64))
    T, blended = 1.0, []
    for i in range(n):
        if not ok[i]:
            blended.append(False)
            continue
        if T * (1 - alpha[i]) < 1e-4:
            blended += [False] * (n - i)
            break
        blended.append(True)
        T *= 1 - alpha[i]
    blended = np.array(blended[:n])
    Mx, My, Cn, Lo, Rgb, Z = (torch.tensor(np.asarray(v, np.float64), requires_grad=True) for v in (mx, my, cn, logo, rgb, z))
    pw = -0.5 * (Cn[:, 0] * Mx * Mx + Cn[:, 2] * My * My) - Cn[:, 1] * Mx * My
    al = torch.where(torch.from_numpy(blended), torch.clamp(torch.exp(Lo + pw), max=0.99), torch.zeros(n, dtype=torch.float64))
    Tx = torch.cumprod(torch.cat([torch.ones(1, dtype=torch.float64), 1 - al[:-1]]), 0)
    bg = torch.tensor([0.3, 0.2, 0.1], dtype=torch.float64)
    Tf = Tx[-1] * (1 - al[-1])
    Cpix = ((Tx * al)[:, None] * Rgb).sum(0) + Tf * bg
    Apix = 1.0 - Tf
    Dpix = (Tx * al * Z).sum()
    loss = (Cpix * t64(G)).sum() + Apix * float(GA) + Dpix * float(GD)
    loss.backward()
    g = np.zeros((n, 10), np.float32)
    bl = np.zeros(n, np.int32)
    Cf = np.ascontiguousarray(Cpix.detach().numpy(), np.float32)
    zf = np.ascontiguousarray(z, np.float32)
    gm_aux.gm_blend_pixel_aux(C.c_int(n), _p(e), _p(np.ascontiguousarray(rgb, np.float32)), _p(zf), _p(Cf), _p(G),
                              C.c_float(float(Apix.detach())), C.c_float(float(Dpix.detach())), C.c_float(float(GA)), C.c_float(float(GD)),
                              _p(g), _p(bl))
    assert np.array_equal(bl.astype(bool), blended)
    want = np.concatenate([Mx.grad.numpy()[:, None], My.grad.numpy()[:, None], Cn.grad.numpy(), Lo.grad.numpy()[:, None],
                           Rgb.grad.numpy(), Z.grad.numpy()[:, None]], 1)
    scale = max(1.0, float(np.abs(want).max()))
    assert np.allclose(g, want, rtol=1e-4, atol=2e-6 * scale), np.abs(g - want).max()
    assert np.all(g[~blended] == 0)
    capped = blended & (araw >= 0.99)
    assert np.all(g[capped, :6] == 0)  # the cap: alpha has no gradient
    if weights != "all":
        assert np.any(g[:, :6] != 0)  # the plane alone moves the geometry and the opacity
        assert np.all(g[:, 6:9] == 0)  # and no colour


def _preprocess_lib(tmp_path_factory, double):
    if shutil.which("g++") is None:
        pytest.skip("no C++ compiler")
    d = tmp_path_factory.mktemp("grad_mirror_depth64" if double else "grad_mirror_depth")
    if double:
        src = d / "grad_mirror64.cpp"
        src.write_text("#include <math.h>\n#define sqrtf sqrt\n#define fminf fmin\n#define fmaxf fmax\n#define float double\n"
                       '#include "%s"\n' % MIRROR_SRC)
        so = str(d / "libgrad_mirror64.so")
        subprocess.run([*CXX, str(src), "-o", so], check=True)
    else:
        so = str(d / "libgrad_mirror.so")
        subprocess.run([*CXX, "-fvisibility=hidden", "-x", "c++", MIRROR_SRC, "-o", so], check=True)
    return C.CDLL(so)


class ViewParams64(C.Structure):
    _fields_ = [("view", C.c_double * 16), ("proj", C.c_double * 16), ("tanfovx", C.c_double), ("tanfovy", C.c_double),
                ("focalx", C.c_double), ("focaly", C.c_double), ("cam_pos", C.c_double * 3), ("width", C.c_int),
                ("height", C.c_int)]


def vp64(vp):
    v = ViewParams64()
    v.view[:], v.proj[:], v.cam_pos[:] = list(vp.view), list(vp.proj), list(vp.cam_pos)
    v.tanfovx, v.tanfovy, v.focalx, v.focaly, v.width, v.height = vp.tanfovx, vp.tanfovy, vp.focalx, vp.focaly, vp.width, vp.height
    return v


@pytest.mark.parametrize("double", [False, True], ids=["float", "double"])
def test_mirror_depth_gradient_reaches_pos(tmp_path_factory, double):
    """The packed 2D gradient with slot kG2Depth (9) set: project_backward adds it to dL/d(view z), so grad_pos matches
    autograd of a loss with a depth term.  Bars as the existing mirror test: 1e-6 for the double build (the algebra),
    2e-3 for the float build."""
    lib = _preprocess_lib(tmp_path_factory, double)
    rng = np.random.default_rng(21)
    vp = orc.view_params(orc.make_camera(scenes.CAM_POS, scenes.CAM_TARGET, scenes.WORLD_UP_BLENDER, 640, 360))
    P, deg = 4000, 3
    cam = np.array(list(vp.cam_pos), np.float64)
    V = np.array(list(vp.view), np.float64).reshape(4, 4)
    right, up, front = V[:3, 0], V[:3, 1], V[:3, 2]
    zz = rng.uniform(1.0, 6.0, P)
    lat = rng.uniform(-0.9, 0.9, (P, 2))
    pos = cam + front[None] * zz[:, None] + (right[None] * lat[:, :1] * vp.tanfovx + up[None] * lat[:, 1:] * vp.tanfovy) * zz[:, None]
    scale = 10 ** rng.uniform(-2.0, -0.8, (P, 3))
    rotq = rng.normal(size=(P, 4))
    sh = rng.normal(size=(P, 16, 3)) * 0.1
    opacity = rng.uniform(0.05, 0.95, P)
    f32 = lambda a: np.ascontiguousarray(a, np.float32)  # noqa: E731
    pos, scale, rotq, sh, opacity = (f32(a) for a in (pos, scale, rotq, sh, opacity))
    g2 = np.zeros((P, 12), np.float32)
    g2[:, :9] = rng.normal(size=(P, 9))
    g2[:, 2:5] *= 50.0
    g2[:, 9] = rng.normal(size=P) * 100.0  # dL/d(view depth)
    outs = [np.zeros((P, 3)), np.zeros((P, 3)), np.zeros((P, 4)), np.zeros((P, 16, 3)), np.zeros(P)]
    if double:
        d64 = lambda a: np.ascontiguousarray(a, np.float64)  # noqa: E731
        lib.gm_preprocess_backward(C.c_int(P), C.c_int(deg), _p(d64(pos)), _p(d64(scale)), _p(d64(rotq)), _p(d64(sh)),
                                   _p(d64(opacity)), C.c_double(1.0), C.byref(vp64(vp)), _p(d64(g2)), *[_p(o) for o in outs])
    else:
        outs = [o.astype(np.float32) for o in outs]
        lib.gm_preprocess_backward(C.c_int(P), C.c_int(deg), _p(pos), _p(scale), _p(rotq), _p(sh), _p(opacity), C.c_float(1.0),
                                   C.byref(vp), _p(g2), *[_p(o) for o in outs])
    L = [tr.leaf(a) for a in (pos, scale, rotq, sh, opacity)]
    means, conic, color, depth = tr.preprocess(L[0], L[1], L[2], L[3], vp, deg)
    g = torch.from_numpy(g2.astype(np.float64))
    loss = ((means * g[:, 0:2]).sum() + (conic * g[:, 2:5]).sum() + (torch.log(L[4]) * g[:, 5]).sum()
            + (color * g[:, 6:9]).sum() + (depth * g[:, 9]).sum())
    loss.backward()
    err = rel_l2(outs[0], L[0].grad.numpy())
    print("double" if double else "float", "grad_pos rel L2", err)
    assert err <= (1e-6 if double else 2e-3), err
    # the depth term, dL/dz * d(view z)/d(pos) = g2[9] * (V[2], V[6], V[10]), is a sizeable part of the result, so a
    # kernel that dropped it would fail the bar above
    dz_part = g2[:, 9:10].astype(np.float64) * V[:3, 2][None]
    assert np.linalg.norm(dz_part) > 0.1 * np.linalg.norm(L[0].grad.numpy())


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not available")
def test_blend_backward_aux_kernel_sass():
    archs, funcs = kernel_ops(build.build_native())
    assert archs == {"sm_100a"}
    hits = [(k, v) for k, v in funcs.items() if "blend_backward_aux_kernel" in k]
    assert len(hits) == 1, [k for k in funcs if "backward" in k]
    ops = hits[0][1]
    assert ops["STL"] == 0 and ops["LDL"] == 0
    assert ops["LDGSTS"] >= 4  # the three record planes and the view depth, staged with cp.async
    assert ops["RED"] + ops["REDG"] + ops["ATOMG"] >= 1
    for op in ("UTCMMA", "HMMA", "UBLKCP", "UTMALDG"):
        assert not [k for k in ops if k.startswith(op)], op
    res = subprocess.run(["cuobjdump", "-res-usage", build.build_native()], capture_output=True, text=True, check=True).stdout
    lines = res.splitlines()
    for i, ln in enumerate(lines):
        if "blend_backward" in ln and "Function" in ln and i + 1 < len(lines):
            print(ln.strip(), lines[i + 1].strip())
