"""The backward pass without a GPU: the float64 torch reference (tests/torch_reference.py) against the oracle and
torch.autograd.gradcheck, the CUDA path's derivative header (csrc/lcgs_grad.cuh, built with g++ from
tests/grad_mirror) against the reference's autograd, the ctypes Grad struct against the C header, and the SASS of
the backward kernels."""
import collections
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from luisacomputegaussiansplatting_b200 import _capi, build, scenes
from oracle import oracle as orc

import torch_reference as tr

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
MIRROR_SRC = os.path.join(HERE, "grad_mirror", "grad_mirror.cpp")

SCENES = [("C3", 4000, 320, 180), ("C1", 3000, 200, 200), ("C2", 5000, 320, 212), ("C3", 1500, 97, 61)]


def frame_of(key, P, W, H, **kw):
    sc, cfg = scenes.make_config_scene(key, P=P)
    vp = orc.view_params(orc.make_camera(scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world), W, H))
    return sc, vp, orc.forward(sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, vp, **kw)


def rel_l2(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return float(np.linalg.norm(got - want) / max(np.linalg.norm(want), 1e-30))


@pytest.mark.parametrize("key,P,W,H", SCENES)
def test_reference_image_matches_the_oracle(key, P, W, H):
    sc, vp, fr = frame_of(key, P, W, H)
    dec = tr.decisions(fr, sc.opacity, W, H)
    t = lambda a: torch.from_numpy(np.asarray(a, np.float64))  # noqa: E731
    # the blend walk alone, from the oracle's own 2D inputs: the decisions are the oracle's
    img = tr.render(t(fr.means_2d), t(fr.conic), t(fr.color), t(sc.opacity), dec, W, H)
    assert float(np.abs(img.numpy() - fr.img).max()) <= 1e-5
    # the whole chain in float64: the oracle's float32 preprocess moves means by ~3e-5 px, the image by ~2e-5
    full = tr.forward(*[t(a) for a in (sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity)], vp, fr, dec=dec)
    assert float(np.abs(full.numpy() - fr.img).max()) <= 1e-4
    m, c, col, _ = tr.preprocess(*[t(a) for a in (sc.pos, sc.scale, sc.rotq, sc.sh)], vp)
    vis = fr.tiles_touched > 0
    assert float(np.abs(m.numpy()[vis] - fr.means_2d[vis]).max()) <= 1e-3
    assert float(np.abs(col.numpy()[vis] - fr.color[vis]).max()) <= 1e-6


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


def test_reference_gradcheck_on_a_tiny_scene():
    vp, pos, scale, rotq, sh, opacity = tiny_scene()
    fr = orc.forward(pos, scale, rotq, sh, opacity, vp, bg=(0.2, 0.1, 0.3))
    assert fr.num_rendered > 0
    dec = tr.decisions(fr, opacity, 32, 32)
    # nothing near a clamp: colours inside (0, 1), tx/ty inside the frustum margin, alpha below the cap
    t = lambda a: torch.from_numpy(np.asarray(a, np.float64))  # noqa: E731
    _, _, col, _ = tr.preprocess(t(pos), t(scale), t(rotq), t(sh), vp)
    assert float(col.min()) > 0.05 and float(col.max()) < 0.95
    assert float(opacity.max()) < 0.9

    def f(p, s, q, h, o):
        return tr.forward(p, s, q, h, o, vp, fr, dec=dec, bg=(0.2, 0.1, 0.3))

    inputs = [tr.leaf(a) for a in (pos, scale, rotq, sh, opacity)]
    assert torch.autograd.gradcheck(f, inputs, eps=1e-6, atol=1e-6, rtol=1e-4)


@pytest.fixture(scope="module")
def gm(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("no C++ compiler")
    so = str(tmp_path_factory.mktemp("grad_mirror") / "libgrad_mirror.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-fvisibility=hidden",
                    "-Wno-unknown-pragmas", "-x", "c++", MIRROR_SRC, "-o", so], check=True)
    return C.CDLL(so)


@pytest.fixture(scope="module")
def gm64(tmp_path_factory):
    """The same header compiled with every float as a double: checks the derivative algebra apart from roundoff."""
    if shutil.which("g++") is None:
        pytest.skip("no C++ compiler")
    d = tmp_path_factory.mktemp("grad_mirror64")
    src = d / "grad_mirror64.cpp"
    src.write_text("#include <math.h>\n#define sqrtf sqrt\n#define fminf fmin\n#define fmaxf fmax\n#define float double\n"
                   '#include "%s"\n' % MIRROR_SRC)
    so = str(d / "libgrad_mirror64.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-Wno-unknown-pragmas", str(src),
                    "-o", so], check=True)
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


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def random_gaussians(P, rng, vp):
    """Gaussians around the view of `vp`: some far off-axis (tx/ty clamped), some with saturated colours."""
    cam = np.array(list(vp.cam_pos), np.float64)
    V = np.array(list(vp.view), np.float64).reshape(4, 4)  # column-major: V[c][r]
    right, up, front = V[:3, 0], V[:3, 1], V[:3, 2]
    z = rng.uniform(1.0, 6.0, P)
    lat = rng.uniform(-1.0, 1.0, (P, 2)) * np.where(rng.random(P) < 0.2, 2.5, 0.9)[:, None]  # 20 % beyond the clamp
    pos = cam + front[None] * z[:, None] + (right[None] * lat[:, :1] * vp.tanfovx + up[None] * lat[:, 1:] * vp.tanfovy) * z[:, None]
    scale = 10 ** rng.uniform(-2.3, -0.7, (P, 3))
    q = rng.normal(size=(P, 4))
    q *= rng.uniform(0.5, 1.5, (P, 1))  # unnormalised, as the forward allows
    sh = rng.normal(size=(P, 16, 3)) * 0.3
    sh[:, 0] *= np.where(rng.random(P) < 0.3, 6.0, 1.0)[:, None]  # 30 %: colours clamped on some channels
    opacity = rng.uniform(0.02, 1.0, P)
    f = lambda a: np.ascontiguousarray(a, np.float32)  # noqa: E731
    return f(pos), f(scale), f(q), f(sh), f(opacity)


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_mirror_preprocess_backward_matches_autograd(gm, gm64, deg):
    """Bars: the double build within 1e-6 (the algebra), the float build within 2e-3 relative L2 per tensor (what the
    kernel runs: a few very thin Gaussians seen edge-on carry ~0.5 % roundoff of the float32 covariance; measured
    9.6e-4 for the scale gradient at degree 1, below 1e-4 elsewhere)."""
    rng = np.random.default_rng(10 + deg)
    vp = orc.view_params(orc.make_camera(scenes.CAM_POS, scenes.CAM_TARGET, scenes.WORLD_UP_BLENDER, 640, 360))
    P = 10_000
    pos, scale, rotq, sh, opacity = random_gaussians(P, rng, vp)
    feat = (deg + 1) ** 2
    sh = np.ascontiguousarray(sh[:, :feat])
    g2 = np.zeros((P, 12), np.float32)
    g2[:, :9] = rng.normal(size=(P, 9))
    g2[:, 2:5] *= 50.0  # conic entries are small numbers: give their gradient a comparable weight
    outs = [np.zeros((P, 3), np.float32), np.zeros((P, 3), np.float32), np.zeros((P, 4), np.float32),
            np.zeros((P, feat, 3), np.float32), np.zeros(P, np.float32)]
    gm.gm_preprocess_backward(C.c_int(P), C.c_int(deg), _p(pos), _p(scale), _p(rotq), _p(sh), _p(opacity), C.c_float(1.3),
                              C.byref(vp), _p(g2), *[_p(o) for o in outs])
    d = lambda a: np.ascontiguousarray(a, np.float64)  # noqa: E731
    outs64 = [np.zeros(o.shape, np.float64) for o in outs]
    gm64.gm_preprocess_backward(C.c_int(P), C.c_int(deg), _p(d(pos)), _p(d(scale)), _p(d(rotq)), _p(d(sh)), _p(d(opacity)),
                                C.c_double(1.3), C.byref(vp64(vp)), _p(d(g2)), *[_p(o) for o in outs64])
    L = [tr.leaf(a) for a in (pos, scale, rotq, sh, opacity)]
    means, conic, color, _ = tr.preprocess(L[0], L[1], L[2], L[3], vp, deg, scale_modifier=1.3)
    g = torch.from_numpy(g2.astype(np.float64))
    loss = (means * g[:, 0:2]).sum() + (conic * g[:, 2:5]).sum() + (torch.log(L[4]) * g[:, 5]).sum() + (color * g[:, 6:9]).sum()
    loss.backward()
    # the cases the clamps matter for are present
    col = color.detach().numpy()
    assert ((col == 0) | (col == 1)).any(axis=1).mean() > 0.1
    names = ("pos", "scale", "rotq", "sh", "opacity")
    errs = {n: rel_l2(o, x.grad.numpy()) for n, o, x in zip(names, outs, L)}
    errs64 = {n: rel_l2(o, x.grad.numpy()) for n, o, x in zip(names, outs64, L)}
    print(deg, errs, errs64)
    for n in names:
        assert errs64[n] <= 1e-6, (n, errs64[n])
        assert errs[n] <= 2e-3, (n, errs[n])
    # clamped colour channels pass no gradient to the SH coefficients of that channel
    clamped = (col == 0) | (col == 1)
    assert np.all(outs[3][:, 0, :][clamped] == 0.0)


def test_mirror_blend_pixel_matches_autograd(gm):
    """Hand-built pixel lists: ordinary entries, an alpha-test reject, the 0.99 cap, and a saturating entry that ends
    the walk (itself and everything after it get no gradient)."""
    rng = np.random.default_rng(7)
    cases = []
    n = 12
    for kind in ("plain", "cap", "saturate"):
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
        cases.append((mx, my, cn, logo, rng.uniform(0, 1, (n, 3))))
    for mx, my, cn, logo, rgb in cases:
        f = np.float32
        dx, dy = mx.astype(f), my.astype(f)  # pixel at the origin
        a, b, c = (-0.5 * cn[:, 0]).astype(f), (-cn[:, 1]).astype(f), (-0.5 * cn[:, 2]).astype(f)
        power = (a * dx * dx + b * dx * dy + c * dy * dy).astype(f)
        araw = (np.exp(logo) * np.exp(power.astype(np.float64))).astype(f)
        ok = (power <= 0) & (araw >= 1.0 / 255.0)
        e = np.ascontiguousarray(np.stack([dx, dy, a, b, c, ok.astype(f), araw], 1), f)
        G = rng.normal(size=3).astype(f)
        # the reference first: decisions and the final colour in float64
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
        Mx, My, Cn, Lo, Rgb = (torch.tensor(np.asarray(v, np.float64), requires_grad=True) for v in (mx, my, cn, logo, rgb))
        pw = -0.5 * (Cn[:, 0] * Mx * Mx + Cn[:, 2] * My * My) - Cn[:, 1] * Mx * My
        al = torch.where(torch.from_numpy(blended), torch.clamp(torch.exp(Lo + pw), max=0.99), torch.zeros(n, dtype=torch.float64))
        Tx = torch.cumprod(torch.cat([torch.ones(1, dtype=torch.float64), 1 - al[:-1]]), 0)
        bg = torch.tensor([0.3, 0.2, 0.1], dtype=torch.float64)
        Cpix = ((Tx * al)[:, None] * Rgb).sum(0) + Tx[-1] * (1 - al[-1]) * bg
        (Cpix * torch.from_numpy(G.astype(np.float64))).sum().backward()
        g = np.zeros((n, 9), np.float32)
        bl = np.zeros(n, np.int32)
        Cf = np.ascontiguousarray(Cpix.detach().numpy(), np.float32)
        gm.gm_blend_pixel(C.c_int(n), _p(e), _p(np.ascontiguousarray(rgb, np.float32)), _p(Cf), _p(G), _p(g), _p(bl))
        assert np.array_equal(bl.astype(bool), blended)
        want = np.concatenate([Mx.grad.numpy()[:, None], My.grad.numpy()[:, None], Cn.grad.numpy(), Lo.grad.numpy()[:, None],
                               Rgb.grad.numpy()], 1)
        assert np.allclose(g, want, rtol=1e-4, atol=2e-6), np.abs(g - want).max()
        assert np.all(g[~blended] == 0)
        capped = blended & (araw >= 0.99)
        assert np.all(g[capped, :6] == 0)  # the cap: alpha has no gradient; the colour still has one


@pytest.mark.skipif(shutil.which("cc") is None, reason="no C compiler")
def test_ctypes_grad_matches_the_header(tmp_path):
    fields = [name for name, _ in _capi.Grad._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "lcgs_b200.h"\nint main(void) {\n'
                   '    printf("sizeof %zu\\n", sizeof(lcgs_b200_grad));\n'
                   + "".join('    printf("%s %%zu\\n", offsetof(lcgs_b200_grad, %s));\n' % (f, f) for f in fields)
                   + "    return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["cc", "-I", os.path.join(REPO, "include"), str(src), "-o", str(exe)], check=True)
    out = dict(ln.split() for ln in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out["sizeof"]) == C.sizeof(_capi.Grad)
    for f in fields:
        assert int(out[f]) == getattr(_capi.Grad, f).offset, f
    assert "lcgs_b200_render_backward" in _capi.EXPORTED_SYMBOLS


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not available")
def test_backward_kernels_sass():
    lib = build.build_native()
    sass = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    funcs, name, archs = collections.OrderedDict(), None, set()
    for ln in sass.splitlines():
        m = re.search(r"arch = (sm_\w+)", ln)
        if m:
            archs.add(m.group(1))
        m = re.search(r"Function : (\S+)", ln)
        if m:
            name = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip()
            funcs[name] = collections.Counter()
        elif name:
            m = re.match(r"\s+/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", ln)
            if m:
                funcs[name][m.group(1)] += 1
    assert archs == {"sm_100a"}
    for part in ("rebuild_records_kernel", "blend_backward_kernel", "preprocess_backward_kernel"):
        hits = [v for k, v in funcs.items() if part in k]
        assert len(hits) == 1, part
        ops = hits[0]
        assert ops["STL"] == 0 and ops["LDL"] == 0, part
        for op in ("UTCMMA", "HMMA", "UBLKCP", "UTMALDG"):
            assert not [k for k in ops if k.startswith(op)], (part, op)
    blend = [v for k, v in funcs.items() if "blend_backward_kernel" in k][0]
    assert blend["LDGSTS"] >= 3  # the three record planes, staged as in the forward
    assert blend["RED"] + blend["REDG"] + blend["ATOMG"] >= 1
