"""The camera-pose gradient without a GPU: the derivative header's pose terms (csrc/lcgs_grad.cuh, built with g++ from
tests/grad_mirror/grad_mirror_pose.cpp, in float and in double) against torch float64 autograd of the pose reference
(tests/torch_reference_pose.py) with respect to the view matrix and the camera position, gradcheck of a tiny frame's
reference image with respect to both, lcgs.world_to_camera, and the SASS of the new kernels."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from luisacomputegaussiansplatting_b200 import build, scenes
from oracle import oracle as orc

import torch_reference as tr
import torch_reference_pose as tp
from sass_ops import kernel_ops
from test_backward_cpu import random_gaussians, tiny_scene, vp64

HERE = os.path.dirname(os.path.abspath(__file__))
MIRROR_SRC = os.path.join(HERE, "grad_mirror", "grad_mirror_pose.cpp")
VIEW_IDX = [(j // 3) * 4 + j % 3 for j in range(12)]  # pose term j -> vp.view index


def build_mirror(tmp, double):
    if shutil.which("g++") is None:
        pytest.skip("no C++ compiler")
    src = MIRROR_SRC
    if double:  # every float as a double: the derivative algebra apart from roundoff
        src = str(tmp / "grad_mirror_pose64.cpp")
        with open(src, "w") as fh:
            fh.write("#include <math.h>\n#define sqrtf sqrt\n#define fminf fmin\n#define fmaxf fmax\n#define float double\n"
                     '#include "%s"\n' % MIRROR_SRC)
    so = str(tmp / ("libgrad_mirror_pose%s.so" % ("64" if double else "")))
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-fvisibility=hidden",
                    "-Wno-unknown-pragmas", "-x", "c++", src, "-o", so], check=True)
    return C.CDLL(so)


@pytest.fixture(scope="module")
def gm(tmp_path_factory):
    return build_mirror(tmp_path_factory.mktemp("gm_pose"), False)


@pytest.fixture(scope="module")
def gm64(tmp_path_factory):
    return build_mirror(tmp_path_factory.mktemp("gm_pose64"), True)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def mirror_terms(lib, double, P, deg, pos, scale, rotq, sh, scale_modifier, vp, g2):
    """[P, 15] per-Gaussian pose terms from the host build of lcgs_grad.cuh."""
    dt = np.float64 if double else np.float32
    a = [np.ascontiguousarray(x, dt) for x in (pos, scale, rotq, sh, g2)]
    out = np.zeros((P, 15), dt)
    sm = C.c_double(scale_modifier) if double else C.c_float(scale_modifier)
    lib.gm_pose_terms(C.c_int(P), C.c_int(deg), _p(a[0]), _p(a[1]), _p(a[2]), _p(a[3]), sm,
                      C.byref(vp64(vp) if double else vp), _p(a[4]), _p(out))
    return out


def pose_vector(view_grad, cam_grad):
    """The 15 pose terms from a [16] view gradient and a [3] camera-position gradient."""
    return np.concatenate([np.asarray(view_grad)[VIEW_IDX], np.asarray(cam_grad)])


def rel_l2(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return float(np.linalg.norm(got - want) / max(np.linalg.norm(want), 1e-30))


def test_mirror_view_index_is_the_kernels(gm):
    assert [gm.gm_pose_view_index(C.c_int(j)) for j in range(12)] == VIEW_IDX


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_mirror_pose_terms_match_autograd(gm, gm64, deg):
    """Random Gaussians around the C3 view: 20 % beyond the tx/ty clamp, 30 % with clamped colour channels, random
    upstream gradients of the means, the conic, the colour and the depth (slot 9).  Bars on the 15-vector of summed
    terms and on each Gaussian's own terms: the double build within 1e-6 (the algebra; its literals stay float).  The
    float build (what the kernel runs) within 5e-4 for the sum and 1e-5 for the median Gaussian: its sums measured
    1.8e-6 to 9.4e-5, the largest at degree 3, from the float32 covariance chain of a few thin Gaussians."""
    rng = np.random.default_rng(40 + deg)
    vp = orc.view_params(orc.make_camera(scenes.CAM_POS, scenes.CAM_TARGET, scenes.WORLD_UP_BLENDER, 640, 360))
    P = 400
    pos, scale, rotq, sh, _ = random_gaussians(P, rng, vp)
    feat = (deg + 1) ** 2
    sh = np.ascontiguousarray(sh[:, :feat])
    g2 = np.zeros((P, 12), np.float32)
    g2[:, :9] = rng.normal(size=(P, 9))
    g2[:, 2:5] *= 50.0
    g2[:, 9] = rng.normal(size=P)  # dL/d(view depth) of the depth plane
    t32 = mirror_terms(gm, False, P, deg, pos, scale, rotq, sh, 1.3, vp, g2)
    t64 = mirror_terms(gm64, True, P, deg, pos, scale, rotq, sh, 1.3, vp, g2)

    # autograd, one Gaussian at a time for the per-Gaussian bar (the sum is their sum)
    V, cp = tp.vp_pose(vp)
    L = [torch.from_numpy(np.asarray(a, np.float64)) for a in (pos, scale, rotq, sh)]
    means, conic, color, depth = tp.preprocess(*L, vp, V, cp, deg, scale_modifier=1.3)
    g = torch.from_numpy(g2.astype(np.float64))
    per = (means * g[:, 0:2]).sum(1) + (conic * g[:, 2:5]).sum(1) + (color * g[:, 6:9]).sum(1) + depth * g[:, 9]
    want = np.zeros((P, 15))
    for i in range(P):
        gv, gc = torch.autograd.grad(per[i], (V, cp), retain_graph=True, allow_unused=True)
        want[i] = pose_vector(gv.numpy(), np.zeros(3) if gc is None else gc.numpy())  # degree 0: cam_pos is unused
        assert not gv.numpy()[[3, 7, 11, 15]].any()
    col = color.detach().numpy()
    clamped = (col == 0) | (col == 1)
    assert clamped.any(axis=1).mean() > 0.1
    V_ = np.array(list(vp.view), np.float64).reshape(4, 4)
    pv = np.asarray(pos, np.float64) @ V_[:3, :3] + V_[3, :3]
    lim = 1.3 * np.array([vp.tanfovx, vp.tanfovy])
    assert (np.abs(pv[:, :2] / pv[:, 2:3]) > lim).any(axis=1).mean() > 0.05  # the tx/ty clamp is active

    e64 = rel_l2(t64.sum(0), want.sum(0))
    e32 = rel_l2(t32.astype(np.float64).sum(0), want.sum(0))
    rows = np.linalg.norm(want, axis=1)
    per64 = np.linalg.norm(t64 - want, axis=1) / np.maximum(rows, 1e-30)
    per32 = np.linalg.norm(t32 - want, axis=1) / np.maximum(rows, 1e-30)
    print("deg", deg, "sum rel L2 double %.2e float %.2e; per-Gaussian max double %.2e, median float %.2e"
          % (e64, e32, per64.max(), np.median(per32)))
    assert e64 <= 1e-6 and per64.max() <= 1e-6
    assert e32 <= 5e-4
    assert np.median(per32) <= 1e-5
    if deg == 0:
        assert not t32[:, 12:].any() and not t64[:, 12:].any()  # no view direction: exactly zero
    else:
        assert np.abs(want[:, 12:]).sum() > 0
    # all three channels clamped: the view direction gets nothing
    full = clamped.all(axis=1)
    if full.any():
        assert not t32[full, 12:].any()


def test_reference_gradcheck_of_the_pose():
    vp, pos, scale, rotq, sh, opacity = tiny_scene()
    fr = orc.forward(pos, scale, rotq, sh, opacity, vp, bg=(0.2, 0.1, 0.3))
    assert fr.num_rendered > 0
    dec = tr.decisions(fr, opacity, 32, 32)
    t = lambda a: torch.from_numpy(np.asarray(a, np.float64))  # noqa: E731
    scene = [t(a) for a in (pos, scale, rotq, sh, opacity)]

    def f(view, cam_pos):
        return tp.forward(*scene, vp, fr, view, cam_pos, dec=dec, bg=(0.2, 0.1, 0.3))

    V, cp = tp.vp_pose(vp)
    assert torch.autograd.gradcheck(f, (V, cp), eps=1e-6, atol=1e-6, rtol=1e-4)
    # with vp's own pose the pose reference is torch_reference's forward exactly
    assert torch.equal(f(V.detach(), cp.detach()), tr.forward(*scene, vp, fr, dec=dec, bg=(0.2, 0.1, 0.3)))


def test_world_to_camera_is_the_view_matrix():
    from luisacomputegaussiansplatting_b200 import lcgs

    for pose in [(scenes.CAM_POS, scenes.CAM_TARGET, scenes.WORLD_UP_BLENDER), ((1.0, -2.0, 0.5), (0.0, 0.3, 0.1), (0.0, 1.0, 0.0))]:
        cam = lcgs.make_camera(*pose, 64, 48)
        M = lcgs.world_to_camera(cam)
        assert M.dtype == np.float32 and M.shape == (4, 4) and M.flags.c_contiguous
        assert np.array_equal(M, lcgs.world_to_local_matrix(cam).reshape(4, 4).T)
        assert np.array_equal(M.T.ravel(), np.array(list(lcgs.view_params(cam).view), np.float32))
        # p_cam = M[:3, :3] p + M[:3, 3]: the camera centre maps to the origin
        c = np.array(list(cam.position), np.float64)
        assert np.abs(M[:3, :3].astype(np.float64) @ c + M[:3, 3]).max() < 1e-5


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not available")
def test_pose_kernels_sass():
    archs, funcs = kernel_ops(build.build_native())
    assert archs == {"sm_100a"}
    for part in ("preprocess_pose_grad_kernel", "pose_grad_reduce_kernel"):
        hits = [v for k, v in funcs.items() if part in k]
        assert len(hits) == 1, part
        ops = hits[0]
        assert ops["STL"] == 0 and ops["LDL"] == 0, part
        for op in ("UTCHMMA", "UTCQMMA", "UTCMMA", "HMMA", "LDTM", "STTM", "UBLKCP", "UTMALDG", "UTMASTG"):
            assert not [k for k in ops if k.startswith(op)], (part, op)
    pose = [v for k, v in funcs.items() if "preprocess_pose_grad_kernel" in k][0]
    assert pose["SHFL"] >= 15  # the warp reduction of the 15 terms
    # the names the existing SASS tests count stay unique
    for part in ("build_records_kernel", "blend_backward_kernel", "preprocess_backward_kernel"):
        assert len([k for k in funcs if part in k]) == 1, part
