"""The SSIM loss on the GPU (lcgs_b200_ssim, lcgs.ssim) against the float64 torch formulation of the 3DGS training
code's ssim() (tests/torch_reference_ssim.py).

Bars, per case: the SSIM error <= 2 x the float32 torch formulation's + 1e-6, the gradient's relative L2 error <= 2 x
float32 torch's + 1e-5, and its cosine >= 0.99999.  The float32 torch errors are in TORCH32, measured on a CPU before
any GPU run and checked again by tests/test_ssim_cpu.py."""

import numpy as np
import pytest
import torch

import torch_reference_ssim as rs

pytestmark = pytest.mark.gpu

# (kind, W, H); the last case is the one 7680x4320 frame
CASES = [("uniform", 1, 1), ("uniform", 5, 7), ("uniform", 11, 11), ("uniform", 16, 16), ("uniform", 33, 17),
         ("uniform", 257, 129), ("uniform", 1237, 822), ("uniform", 1920, 1080), ("wide", 16, 16), ("wide", 257, 129),
         ("wide", 1920, 1080), ("zero_one", 1, 1), ("zero_one", 11, 11), ("zero_one", 257, 129),
         ("rendered", 256, 256), ("uniform", 7680, 4320)]
# (|SSIM error|, gradient relative L2 error) of the float32 torch formulation against float64, measured on a CPU
TORCH32 = {
    ("uniform", 1, 1): (3.2e-08, 2.0e-07), ("uniform", 5, 7): (3.1e-08, 2.5e-07),
    ("uniform", 11, 11): (3.6e-09, 4.2e-07), ("uniform", 16, 16): (1.4e-08, 4.7e-07),
    ("uniform", 33, 17): (5.1e-08, 5.4e-07), ("uniform", 257, 129): (2.0e-08, 6.3e-07),
    ("uniform", 1237, 822): (1.7e-08, 6.5e-07), ("uniform", 1920, 1080): (1.6e-08, 6.4e-07),
    ("wide", 16, 16): (2.0e-08, 2.7e-07), ("wide", 257, 129): (6.2e-09, 3.3e-07),
    ("wide", 1920, 1080): (5.1e-09, 3.5e-07), ("zero_one", 1, 1): (4.8e-11, 1.8e-07),
    ("zero_one", 11, 11): (9.4e-11, 2.1e-05), ("zero_one", 257, 129): (5.3e-11, 1.4e-06),
    ("rendered", 256, 256): (3.3e-08, 2.1e-06),
    ("uniform", 7680, 4320): (1.6e-08, 6.4e-07),  # the 1920x1080 uniform figures (i.i.d. pixels)
}


@pytest.fixture(scope="module")
def lcgs():
    from luisacomputegaussiansplatting_b200 import lcgs as m
    return m


@pytest.fixture(scope="module")
def dev(lcgs):
    d = lcgs.Device(0)
    yield d
    d.close()


def call(dev, W, H, x, y, out, grad=None):
    """lcgs_b200_ssim on the current stream with device pointers (ints) or tensors; returns the status."""
    p = lambda t: None if t is None else (t if isinstance(t, int) else t.data_ptr())  # noqa: E731
    return dev.lib.lcgs_b200_ssim(dev.ctx, W, H, p(x), p(y), p(out), p(grad), torch.cuda.current_stream().cuda_stream or None)


def gpu_ssim(dev, x, y, grad=True):
    """(SSIM, gradient or None) of the kernels for float32 numpy or CUDA tensor images [3, H, W]."""
    xt = torch.as_tensor(x).float().cuda().contiguous()
    yt = torch.as_tensor(y).float().cuda().contiguous()
    H, W = xt.shape[1:]
    out = torch.full((), -7.0, device="cuda")
    g = torch.full_like(xt, -7.0) if grad else None
    assert call(dev, W, H, xt, yt, out, g) == 0
    torch.cuda.synchronize()
    return out, g


def case_pair(kind, W, H):
    return rs.rendered_pair(W, H) if kind == "rendered" else rs.case_images(kind, H, W)


@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s-%dx%d" % c)
def test_ssim_matches_the_reference(dev, case):
    kind, W, H = case
    x, y = case_pair(kind, W, H)
    want_v, want_g = rs.reference(x, y, device="cuda")
    v, g = gpu_ssim(dev, x, y)
    e = abs(float(v) - want_v)
    rel, cos = rs.rel_l2(g.cpu().numpy(), want_g), rs.cosine(g.cpu().numpy(), want_g)
    e32, r32 = TORCH32[case]
    print(case, "SSIM %.7f error %.2e (float32 torch %.1e), gradient rel L2 %.2e (float32 torch %.1e) cosine %.9f"
          % (want_v, e, e32, rel, r32, cos))
    assert e <= 2 * e32 + 1e-6
    assert rel <= 2 * r32 + 1e-5 and cos >= 0.99999


@pytest.mark.parametrize("W,H", [(1, 1), (11, 11), (257, 129), (1920, 1080)])
def test_identical_pairs(dev, W, H):
    """(x, x) has SSIM 1 and a gradient of about 0: within 1e-6 of 1, and a max-abs gradient <= 1e-3 x that of
    (x, x + 0.01 noise)."""
    x, _ = rs.case_images("uniform", H, W)
    noise = np.random.default_rng(9).standard_normal(x.shape).astype(np.float32)
    _, g_near = gpu_ssim(dev, x, (x + 0.01 * noise).astype(np.float32))
    ref_scale = float(g_near.abs().max())
    assert ref_scale > 0
    for img in (x, np.zeros_like(x), np.ones_like(x)):
        v, g = gpu_ssim(dev, img, img.copy())
        print("identical %dx%d: |1 - SSIM| %.1e, max |grad| / noisy %.1e" % (W, H, abs(1 - float(v)),
                                                                             float(g.abs().max()) / ref_scale))
        assert abs(1.0 - float(v)) <= 1e-6
        assert float(g.abs().max()) <= 1e-3 * ref_scale


def test_bit_reproducible_and_value_without_gradient(dev):
    x, y = rs.case_images("wide", 1080, 1920)
    v1, g1 = gpu_ssim(dev, x, y)
    v2, g2 = gpu_ssim(dev, x, y)
    v3, _ = gpu_ssim(dev, x, y, grad=False)
    assert torch.equal(v1.view(torch.int32), v2.view(torch.int32))
    assert torch.equal(g1.view(torch.int32), g2.view(torch.int32))
    assert torch.equal(v1.view(torch.int32), v3.view(torch.int32))
    # a larger call in between grows and overwrites the workspace: the same bits after it
    big = rs.case_images("uniform", 2000, 2500)
    gpu_ssim(dev, *big)
    v4, g4 = gpu_ssim(dev, x, y)
    assert torch.equal(v1.view(torch.int32), v4.view(torch.int32)) and torch.equal(g1.view(torch.int32), g4.view(torch.int32))


def test_cuda_graph_capture_and_replay(dev):
    W, H = 640, 360
    xt = torch.rand(3, H, W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    yt = torch.rand(3, H, W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
    out, g = torch.zeros((), device="cuda"), torch.zeros_like(xt)
    assert call(dev, W, H, xt, yt, out, g) == 0  # the first call at this size grows the workspace
    torch.cuda.synchronize()
    v0, g0 = out.clone(), g.clone()
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            assert call(dev, W, H, xt, yt, out, g) == 0
    torch.cuda.current_stream().wait_stream(s)
    out.zero_()
    g.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out.view(torch.int32), v0.view(torch.int32)) and torch.equal(g.view(torch.int32), g0.view(torch.int32))


def test_error_paths_leave_outputs_untouched(dev):
    W, H = 64, 48
    x = torch.rand(3, H, W, device="cuda")
    y = torch.rand(3, H, W, device="cuda")
    pad, canary, n = 4, 0x7F7F1234, 3 * W * H
    buf = torch.full((2 * pad + 1 + 1 + n + pad,), canary, dtype=torch.int32, device="cuda")
    base = buf.data_ptr()
    out_at, grad_at = base + 4 * pad, base + 4 * (2 * pad + 2)  # [pad][out][pad][1][grad n][pad]: grad 8-byte aligned
    bad = [
        (W, H, 0, y.data_ptr(), out_at, grad_at),
        (W, H, x.data_ptr(), 0, out_at, grad_at),
        (W, H, x.data_ptr(), y.data_ptr(), 0, grad_at),
        (0, H, x.data_ptr(), y.data_ptr(), out_at, grad_at),
        (W, -1, x.data_ptr(), y.data_ptr(), out_at, grad_at),
        (W, H, x.data_ptr() + 2, y.data_ptr(), out_at, grad_at),
        (W, H, x.data_ptr(), y.data_ptr() + 1, out_at, grad_at),
        (W, H, x.data_ptr(), y.data_ptr(), out_at + 2, grad_at),
        (W, H, x.data_ptr(), y.data_ptr(), out_at, grad_at + 2),
    ]
    for args in bad:
        assert call(dev, *args) == -1, args
        assert dev.lib.lcgs_b200_last_error(dev.ctx)
    assert dev.lib.lcgs_b200_ssim(None, W, H, x.data_ptr(), y.data_ptr(), out_at, grad_at, None) == -1
    torch.cuda.synchronize()
    assert (buf == canary).all()
    # a good call writes exactly its outputs
    assert call(dev, W, H, x, y, out_at, grad_at) == 0
    torch.cuda.synchronize()
    h = buf.cpu().numpy()
    assert (h[:pad] == canary).all() and (h[pad + 1:2 * pad + 2] == canary).all() and (h[2 * pad + 2 + n:] == canary).all()
    v, g = gpu_ssim(dev, x, y)
    assert h[pad] == int(v.view(torch.int32)) and np.array_equal(h[2 * pad + 2:2 * pad + 2 + n], g.view(torch.int32).cpu().numpy().ravel())


def test_lcgs_ssim_autograd(lcgs, dev):
    x, y = rs.case_images("uniform", 90, 160, seed=4)
    img = torch.tensor(x, device="cuda", requires_grad=True)
    ref = torch.tensor(y, device="cuda")
    v = lcgs.ssim(dev, img, ref)
    assert v.dim() == 0 and v.requires_grad
    (3.0 * v).backward()
    want_v, want_g = rs.reference(x, y)
    assert abs(float(v) - want_v) <= 1e-6
    rel, cos = rs.rel_l2(img.grad.cpu().numpy(), 3.0 * want_g), rs.cosine(img.grad.cpu().numpy(), want_g)
    assert rel <= 2e-5 and cos >= 0.99999, (rel, cos)
    # without grad: the value alone, the same bits
    v2 = lcgs.ssim(dev, img.detach(), ref)
    assert not v2.requires_grad and torch.equal(v2.view(torch.int32), v.detach().view(torch.int32))
    with pytest.raises(ValueError):
        lcgs.ssim(dev, img, ref.clone().requires_grad_())
    with pytest.raises(ValueError):
        lcgs.ssim(dev, img, ref[:, :, 1:])
    with pytest.raises(ValueError):
        lcgs.ssim(dev, img[0], ref[0])


def test_training_loss_through_the_renderer(lcgs, dev):
    """0.8 L1 + 0.2 (1 - ssim) through DifferentiableRenderer on a C1 scene: the five scene gradients match those from
    the float64 reference's dL/dimg fed through the same renderer (the backward's bars)."""
    from test_backward import NAMES, metrics, scene_arrays

    W, H, P = 200, 200, 3_000
    arrays, pose = scene_arrays("C1", P)
    cam = lcgs.make_camera(*pose, W, H)
    dr = lcgs.DifferentiableRenderer(dev, W, H, list_capacity=2_000_000)
    moved = [a.copy() for a in arrays]
    moved[0] = (moved[0] + np.random.default_rng(2).normal(0, 0.01, moved[0].shape)).astype(np.float32)
    with torch.no_grad():
        target = dr(*[torch.tensor(a, device="cuda") for a in moved], cam)
    leaves = [torch.tensor(a, device="cuda", requires_grad=True) for a in arrays]
    img = dr(*leaves, cam)
    loss = 0.8 * (img - target).abs().mean() + 0.2 * (1.0 - lcgs.ssim(dev, img, target))
    loss.backward()
    # the same loss, its dL/dimg from the float64 reference
    leaves2 = [torch.tensor(a, device="cuda", requires_grad=True) for a in arrays]
    img2 = dr(*leaves2, cam)
    assert torch.equal(img2.detach(), img.detach())
    x64 = img2.detach().double().cpu()
    _, g_ssim = rs.reference(x64.numpy(), target.double().cpu().numpy())
    dl = 0.8 * torch.sign(x64 - target.double().cpu()) / x64.numel() - 0.2 * torch.from_numpy(g_ssim)
    img2.backward(dl.float().cuda())
    for n, a, b in zip(NAMES, leaves, leaves2):
        rel, cos = metrics(a.grad.cpu().numpy(), b.grad.cpu().numpy())
        print("%s rel L2 %.2e cosine %.7f" % (n, rel, cos))
        assert rel <= 1e-3 and cos >= 0.9999, n


def test_gradient_ascent_restores_a_noisy_image(lcgs, dev):
    H, W = 96, 128
    yy, xx = np.meshgrid(np.linspace(0, 1, H), np.linspace(0, 1, W), indexing="ij")
    clean = np.stack([0.5 + 0.4 * np.sin(6 * xx + c) * np.cos(4 * yy - c) for c in range(3)]).astype(np.float32)
    noisy = clean + 0.1 * np.random.default_rng(3).standard_normal(clean.shape).astype(np.float32)
    ref = torch.tensor(clean, device="cuda")
    img = torch.tensor(noisy, device="cuda", requires_grad=True)
    opt = torch.optim.Adam([img], lr=5e-3)
    first = float(lcgs.ssim(dev, img.detach(), ref))
    for _ in range(300):
        opt.zero_grad()
        (-lcgs.ssim(dev, img, ref)).backward()
        opt.step()
    last = float(lcgs.ssim(dev, img.detach(), ref))
    print("SSIM %.4f -> %.4f" % (first, last))
    assert first < 0.7 and last > 0.99
