"""Restatements of the SSIM loss (lcgs_b200_ssim, csrc/ssim_math.cuh) for the tests.

- `ssim_torch`: the usual torch formulation of the 3DGS training code's ssim() (utils/loss_utils.py): depthwise 11x11
  conv2d with padding 5 and groups 3, in the dtype of its inputs.  In float64 it is the reference the kernels are held
  to; in float32 it is the formulation users write, whose error sets the bars.
- `ssim_scipy`: an independent float64 restatement with scipy.ndimage.correlate1d (zero padding), separable.
- `closed_form_grad`: the gradient as the kernels compute it (partials P0..P2 of the pixel SSIM, filtered), float64.
"""
import numpy as np
import torch
from scipy import ndimage

F64 = torch.float64
C1, C2 = 0.01 ** 2, 0.03 ** 2


def gauss1d() -> np.ndarray:
    """The 11 window taps in float64: exp(-(k-5)^2 / 4.5), normalised."""
    g = np.exp(-((np.arange(11) - 5.0) ** 2) / 4.5)
    return g / g.sum()


def ssim_torch(x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    """Mean SSIM of [3, H, W] x against y, conv2d formulation, in x's dtype (the window is rounded once from
    float64)."""
    g = torch.from_numpy(gauss1d()).to(x.dtype).to(x.device)
    win = torch.outer(g, g).expand(3, 1, 11, 11).contiguous()
    conv = lambda t: torch.nn.functional.conv2d(t[None], win, padding=5, groups=3)[0]  # noqa: E731
    mx, my = conv(x), conv(y)
    sx, sy, sxy = conv(x * x) - mx * mx, conv(y * y) - my * my, conv(x * y) - mx * my
    s = ((2 * mx * my + C1) * (2 * sxy + C2)) / ((mx * mx + my * my + C1) * (sx + sy + C2))
    return s.mean()


def _filt(a: np.ndarray) -> np.ndarray:
    """The separable window over the last two axes, zero padding: G*a."""
    g = gauss1d()
    a = ndimage.correlate1d(a, g, axis=-1, mode="constant", cval=0.0)
    return ndimage.correlate1d(a, g, axis=-2, mode="constant", cval=0.0)


def moments(x: np.ndarray, y: np.ndarray):
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    return _filt(x), _filt(y), _filt(x * x), _filt(y * y), _filt(x * y)


def pixel(mx, my, exx, eyy, exy):
    """(s, P0, P1, P2) per pixel from the five moments, float64 (the formulas of ssim_math.cuh)."""
    A, B = 2 * mx * my + C1, 2 * (exy - mx * my) + C2
    Cc, D = mx * mx + my * my + C1, (exx - mx * mx) + (eyy - my * my) + C2
    s = A * B / (Cc * D)
    p0 = 2 * my * B / (Cc * D) - 2 * mx * s / Cc + 2 * mx * s / D - 2 * my * A / (Cc * D)
    return s, p0, -s / D, 2 * A / (Cc * D)


def ssim_scipy(x: np.ndarray, y: np.ndarray) -> float:
    return float(pixel(*moments(x, y))[0].mean())


def closed_form_grad(x: np.ndarray, y: np.ndarray) -> np.ndarray:
    """d(mean SSIM)/dx = (1/N) (G*P0 + 2 x G*P1 + y G*P2), float64."""
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    _, p0, p1, p2 = pixel(*moments(x, y))
    return (_filt(p0) + 2 * x * _filt(p1) + y * _filt(p2)) / x.size


def reference(x, y, device="cpu"):
    """(SSIM, dSSIM/dx) of the float64 torch formulation, as numpy float64."""
    xt = torch.as_tensor(np.asarray(x), device=device).to(F64).requires_grad_()
    yt = torch.as_tensor(np.asarray(y), device=device).to(F64)
    v = ssim_torch(xt, yt)
    (g,) = torch.autograd.grad(v, xt)
    return float(v.detach()), g.cpu().numpy()


def torch32(x, y, device="cpu"):
    """(SSIM, dSSIM/dx) of the float32 torch formulation, as numpy float64."""
    xt = torch.as_tensor(np.asarray(x, np.float32), device=device).requires_grad_()
    yt = torch.as_tensor(np.asarray(y, np.float32), device=device)
    v = ssim_torch(xt, yt)
    (g,) = torch.autograd.grad(v, xt)
    return float(v.detach()), g.double().cpu().numpy()


def rel_l2(got, want) -> float:
    got, want = np.asarray(got, np.float64).ravel(), np.asarray(want, np.float64).ravel()
    return float(np.linalg.norm(got - want) / max(np.linalg.norm(want), 1e-300))


def cosine(got, want) -> float:
    got, want = np.asarray(got, np.float64).ravel(), np.asarray(want, np.float64).ravel()
    return float(got @ want / max(np.linalg.norm(got) * np.linalg.norm(want), 1e-300))


def case_images(kind: str, H: int, W: int, seed: int = 0):
    """(x, y) float32 [3, H, W] pairs of the tests: 'uniform' (both U[0, 1)), 'wide' (both U[-0.5, 1.5)),
    'zero_one' (all 0 against all 1)."""
    rng = np.random.default_rng([seed, H, W])
    if kind == "uniform":
        return rng.random((3, H, W), dtype=np.float32), rng.random((3, H, W), dtype=np.float32)
    if kind == "wide":
        return ((rng.random((3, H, W), dtype=np.float32) * 2 - 0.5).astype(np.float32),
                (rng.random((3, H, W), dtype=np.float32) * 2 - 0.5).astype(np.float32))
    if kind == "zero_one":
        return np.zeros((3, H, W), np.float32), np.ones((3, H, W), np.float32)
    raise ValueError(kind)


def rendered_pair(W: int = 256, H: int = 256, P: int = 20_000):
    """A C1 frame rendered by the CPU oracle, and the frame of the same scene with perturbed positions and colours,
    both float32 [3, H, W]."""
    from luisacomputegaussiansplatting_b200 import scenes
    from oracle import oracle as orc

    sc, cfg = scenes.make_config_scene("C1", P=P)
    vp = orc.view_params(orc.make_camera(scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world), W, H))
    arrays = [sc.pos, sc.scale, sc.rotq, np.ascontiguousarray(sc.sh), sc.opacity]
    a = orc.forward(*arrays, vp).img
    rng = np.random.default_rng(7)
    pert = [a_.copy() for a_ in arrays]
    pert[0] = (pert[0] + rng.normal(0.0, 0.01, pert[0].shape)).astype(np.float32)
    pert[3] = (pert[3] + rng.normal(0.0, 0.1, pert[3].shape)).astype(np.float32)
    b = orc.forward(*pert, vp).img
    return np.asarray(a, np.float32).reshape(3, H, W), np.asarray(b, np.float32).reshape(3, H, W)
