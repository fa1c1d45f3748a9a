"""The SSIM loss without a GPU: the float64 torch reference (tests/torch_reference_ssim.py) against an independent
scipy restatement and gradcheck, the closed-form gradient the kernels compute against autograd, the per-pixel header
(csrc/ssim_math.cuh, built with g++ from tests/ssim_mirror/ssim_mirror.cpp, in float and in double) against torch
float64 autograd, the float32 torch formulation's errors that the GPU test's bars are built from, and the SASS of the
new kernels."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from luisacomputegaussiansplatting_b200 import build

import torch_reference_ssim as rs
from sass_ops import kernel_ops
from test_ssim import CASES, TORCH32

HERE = os.path.dirname(os.path.abspath(__file__))
MIRROR_SRC = os.path.join(HERE, "ssim_mirror", "ssim_mirror.cpp")
SIZES = [(1, 1), (5, 7), (11, 11), (3, 20), (16, 9), (33, 17), (64, 96)]  # (W, H)


@pytest.mark.parametrize("W,H", SIZES)
def test_conv2d_reference_matches_scipy(W, H):
    for kind in ("uniform", "wide", "zero_one"):
        x, y = rs.case_images(kind, H, W)
        t = torch.from_numpy(x).double(), torch.from_numpy(y).double()
        v_torch = float(rs.ssim_torch(*t))
        v_scipy = rs.ssim_scipy(x, y)
        assert abs(v_torch - v_scipy) <= 1e-12, (kind, v_torch, v_scipy)
        # the moments themselves: conv2d with padding 5 is correlate1d with zero padding, separably
        g = torch.from_numpy(rs.gauss1d())
        win = torch.outer(g, g).expand(3, 1, 11, 11).contiguous()
        mx = torch.nn.functional.conv2d(t[0][None], win, padding=5, groups=3)[0].numpy()
        assert np.abs(mx - rs.moments(x, y)[0]).max() <= 1e-12


def test_reference_gradcheck():
    rng = np.random.default_rng(3)
    x = torch.from_numpy(rng.random((3, 9, 13))).requires_grad_()
    y = torch.from_numpy(rng.random((3, 9, 13)))
    assert torch.autograd.gradcheck(lambda a: rs.ssim_torch(a, y), (x,), eps=1e-6, atol=1e-8, rtol=1e-5)


@pytest.mark.parametrize("W,H", SIZES)
def test_closed_form_gradient_matches_autograd(W, H):
    for kind in ("uniform", "wide", "zero_one"):
        x, y = rs.case_images(kind, H, W, seed=1)
        _, want = rs.reference(x, y)
        got = rs.closed_form_grad(x, y)
        assert np.abs(got - want).max() <= 1e-10 * max(np.abs(want).max(), 1e-300) + 1e-300, kind


def build_mirror(tmp, double):
    if shutil.which("g++") is None:
        pytest.skip("no C++ compiler")
    src = MIRROR_SRC
    if double:  # every float as a double: the algebra apart from roundoff (the window literals stay float)
        src = str(tmp / "ssim_mirror64.cpp")
        with open(src, "w") as fh:
            fh.write('#include <math.h>\n#include <cmath>\n#include <stdint.h>\n#define float double\n#include "%s"\n' % MIRROR_SRC)
    so = str(tmp / ("libssim_mirror%s.so" % ("64" if double else "")))
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-fvisibility=hidden",
                    "-x", "c++", src, "-o", so], check=True)
    lib = C.CDLL(so)
    lib.sm_ssim_weight.restype = C.c_double if double else C.c_float
    return lib


@pytest.fixture(scope="module")
def sm(tmp_path_factory):
    return build_mirror(tmp_path_factory.mktemp("ssim_mirror"), False)


@pytest.fixture(scope="module")
def sm64(tmp_path_factory):
    return build_mirror(tmp_path_factory.mktemp("ssim_mirror64"), True)


def mirror_pixel(lib, double, m):
    """[4, n] (s, P0, P1, P2) of the host build from moments [5, n]."""
    dt = np.float64 if double else np.float32
    m = np.ascontiguousarray(m, dt)
    out = np.zeros((4, m.shape[1]), dt)
    lib.sm_ssim_pixel(C.c_int(m.shape[1]), m.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
    return out


def autograd_pixel(m):
    """[4, n] (s, ds/dmx, ds/dexx, ds/dexy) of torch float64 autograd of the 3DGS per-pixel formula."""
    t = torch.from_numpy(np.asarray(m, np.float64)).requires_grad_()
    mx, my, exx, eyy, exy = t
    s = ((2 * mx * my + rs.C1) * (2 * (exy - mx * my) + rs.C2)) / ((mx * mx + my * my + rs.C1) *
                                                                   ((exx - mx * mx) + (eyy - my * my) + rs.C2))
    (g,) = torch.autograd.grad(s.sum(), t)
    return np.stack([s.detach().numpy(), g[0].numpy(), g[2].numpy(), g[4].numpy()])


def moment_cases():
    """Moments of random windows (consistent: from actual pixel values), and degenerate ones."""
    rng = np.random.default_rng(11)
    n = 2000
    vals = rng.uniform(-0.5, 1.5, (2, n, 16))
    w = rng.dirichlet(np.ones(16), n)  # positive window weights summing to 1
    x, y = vals
    m = np.stack([(w * x).sum(1), (w * y).sum(1), (w * x * x).sum(1), (w * y * y).sum(1), (w * x * y).sum(1)])
    const = rng.uniform(0, 1, 50)  # sigma = 0: flat windows
    flat = np.stack([const, const[::-1], const ** 2, const[::-1] ** 2, const * const[::-1]])
    zero = np.zeros((5, 1))        # mx = my = 0 and sigma = 0 (all-black windows)
    mz = np.stack([np.zeros(40), np.zeros(40), rng.uniform(0, 1, 40), rng.uniform(0, 1, 40), rng.uniform(-0.5, 0.5, 40)])
    same = m.copy()                # x == y
    same[1], same[3], same[4] = same[0], same[2], same[2]
    return dict(random=m, flat=flat, zero=zero, mean_zero=mz, identical=same)


def test_mirror_weights_are_the_window_rounded_once(sm):
    got = np.array([sm.sm_ssim_weight(C.c_int(k)) for k in range(11)], np.float32)
    assert np.array_equal(got, rs.gauss1d().astype(np.float32))


@pytest.mark.parametrize("name", ["random", "flat", "zero", "mean_zero", "identical"])
def test_mirror_pixel_matches_autograd(sm, sm64, name):
    m = moment_cases()[name]
    want = autograd_pixel(m)
    got64 = mirror_pixel(sm64, True, m)
    # moments are inputs here: the float build sees them rounded to float, so is compared with autograd at those
    m32 = m.astype(np.float32).astype(np.float64)
    want32 = autograd_pixel(m32)
    got32 = mirror_pixel(sm, False, m32).astype(np.float64)
    # errors against each row's scale, and at least 1e-3 of the largest term (P0 is exactly 0 for x == y)
    scale = lambda w: np.maximum(np.abs(w).max(axis=1, keepdims=True), 1e-3 * np.abs(w).max())  # noqa: E731
    e64 = (np.abs(got64 - want) / scale(want)).max()
    e32 = (np.abs(got32 - want32) / scale(want32)).max(axis=1)
    print(name, "double %.2e, float per row %s" % (e64, ["%.1e" % e for e in e32]))
    assert e64 <= 1e-12
    assert (e32 <= 5e-4).all()  # measured up to 1e-4, for flat windows: sigma^2 = exx - mx^2 cancels in float
    if name == "identical":  # A == Cc and B == D bit for bit: s exactly 1 and ds/dmx exactly 0
        got32 = mirror_pixel(sm, False, m32.astype(np.float32).copy())
        assert (got32[0] == 1.0).all() and (got32[1] == 0.0).all()
        assert np.array_equal(got32[3], -2.0 * got32[2])


@pytest.mark.parametrize("case", CASES[:-1], ids=lambda c: "%s-%dx%d" % c)
def test_float32_torch_errors_behind_the_gpu_bars(case):
    """The float32 torch formulation's errors against float64, measured here for each GPU case, are those recorded in
    test_ssim.TORCH32 (within 1.5x: the CPU's convolution order may differ).  The 7680x4320 case reuses the
    1920x1080 uniform figures (per-pixel i.i.d. inputs: the relative error does not depend on the size) and is not
    measured here: its float64 reference takes minutes on a CPU."""
    kind, W, H = case
    x, y = rs.rendered_pair(W, H) if kind == "rendered" else rs.case_images(kind, H, W)
    v64, g64 = rs.reference(x, y)
    v32, g32 = rs.torch32(x, y)
    e, r = abs(v32 - v64), rs.rel_l2(g32, g64)
    rec_e, rec_r = TORCH32[case]
    print(case, "value %.2e (recorded %.1e), gradient rel L2 %.2e (recorded %.1e)" % (e, rec_e, r, rec_r))
    assert e <= 1.5 * rec_e + 1e-9 and r <= 1.5 * rec_r
    assert r >= rec_r / 1.5 or rec_r < 1e-6


def test_identical_pair_gradient_of_float32_torch():
    """(x, x): the reference gradient is about 0; float32 torch reaches a max-abs gradient well under 1e-3 of that of
    (x, x + 0.01 noise), the bar the GPU test applies."""
    x, _ = rs.case_images("uniform", 64, 96)
    noise = np.random.default_rng(5).standard_normal(x.shape).astype(np.float32)
    _, g_same = rs.torch32(x, x)
    _, g_near = rs.torch32(x, (x + 0.01 * noise).astype(np.float32))
    ratio = np.abs(g_same).max() / np.abs(g_near).max()
    print("float32 torch identical-pair ratio %.1e" % ratio)
    assert ratio <= 1e-4


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not available")
def test_ssim_kernels_sass():
    archs, funcs = kernel_ops(build.build_native())
    assert archs == {"sm_100a"}
    names = ("ssim_forward_kernel<false>", "ssim_forward_kernel<true>", "ssim_backward_kernel", "ssim_reduce_kernel")
    for part in names:
        hits = [v for k, v in funcs.items() if part in k]
        assert len(hits) == 1, part
        ops = hits[0]
        assert ops["STL"] == 0 and ops["LDL"] == 0, part
        for op in ("UTCHMMA", "UTCQMMA", "UTCMMA", "HMMA", "LDTM", "STTM", "UBLKCP", "UTMALDG", "UTMASTG"):
            assert not [k for k in ops if k.startswith(op)], (part, op)
    for part in names[:3]:  # the taps are FMAs: 55 per pixel each way in the forward, 33 in the backward
        ops = [v for k, v in funcs.items() if part in k][0]
        ffma = ops["FFMA"] + 2 * ops["FFMA2"]
        assert ffma >= (110 if "forward" in part else 66), (part, ffma)
