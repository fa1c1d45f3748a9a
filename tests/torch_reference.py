"""A float64 torch restatement of the forward splat path, for checking the backward with torch autograd.

preprocess() restates lcgs_math.cuh's view_transform / ewa_cov2d / splat_from_cov / sh_color (with the tx/ty and colour
clamps); render() blends, per tile, over the oracle's own ranges and point_list with the oracle's alpha-test and
saturation decisions (computed once, in float32, by decisions()), vectorised over the tile's pixels and entries.
Discrete quantities (radius, tile rect, order, which pairs blend) are fixed by the oracle's frame; everything
continuous is differentiable float64."""
from __future__ import annotations

import numpy as np
import torch

from oracle import oracle as orc

F64 = torch.float64
SH_C0 = 0.28209479177387814
SH_C1 = 0.4886025119029199


def _vp(vp):
    return (torch.tensor(list(vp.view), dtype=F64), torch.tensor(list(vp.proj), dtype=F64), float(vp.tanfovx),
            float(vp.tanfovy), float(vp.focalx), float(vp.focaly), torch.tensor(list(vp.cam_pos), dtype=F64))


def sh_basis(d: torch.Tensor, deg: int) -> torch.Tensor:
    """[P, (deg+1)^2] real SH basis of the unit directions d [P, 3], with sh_color's signs."""
    x, y, z = d[:, 0], d[:, 1], d[:, 2]
    out = [torch.full_like(x, SH_C0)]
    if deg > 0:
        out += [-SH_C1 * y, SH_C1 * z, -SH_C1 * x]
    if deg > 1:
        xx, yy, zz = x * x, y * y, z * z
        out += [1.0925484305920792 * x * y, -1.0925484305920792 * y * z, 0.31539156525252005 * (2 * zz - xx - yy),
                -1.0925484305920792 * z * x, 0.5462742152960396 * (xx - yy)]
    if deg > 2:
        out += [-0.5900435899266435 * y * (3 * xx - yy), 2.890611442640554 * x * y * z,
                -0.4570457994644658 * y * (4 * zz - xx - yy), 0.3731763325901154 * z * (2 * zz - 3 * xx - 3 * yy),
                -0.4570457994644658 * x * (4 * zz - xx - yy), 1.445305721320277 * z * (xx - yy),
                -0.5900435899266435 * x * (xx - 3 * yy)]
    return torch.stack(out, 1)


def preprocess(pos, scale, rotq, sh, vp, deg: int = 3, scale_modifier: float = 1.0):
    """Per-Gaussian forward in float64.  Returns (means [P,2] pixels, conic [P,3], color [P,3], depth [P])."""
    V, proj, tfx, tfy, fx, fy, cam = _vp(vp)
    W, H = vp.width, vp.height
    vx = pos[:, 0] * V[0] + pos[:, 1] * V[4] + pos[:, 2] * V[8] + V[12]
    vy = pos[:, 0] * V[1] + pos[:, 1] * V[5] + pos[:, 2] * V[9] + V[13]
    vz = pos[:, 0] * V[2] + pos[:, 1] * V[6] + pos[:, 2] * V[10] + V[14]
    p_w = 1.0 / (vz + 1e-6)
    ndc_x, ndc_y = vx * proj[0] * p_w, vy * proj[5] * p_w
    mx = ((ndc_x + 1.0) * W - 1.0) * 0.5
    my = ((ndc_y + 1.0) * H - 1.0) * 0.5
    # ewa_cov2d: M[c][r] = s_c R[c][r], Sigma = M^T M
    w, x, y, z = rotq[:, 0], rotq[:, 1], rotq[:, 2], rotq[:, 3]
    R = torch.stack([
        torch.stack([1 - 2 * y * y - 2 * z * z, 2 * x * y + 2 * z * w, 2 * x * z - 2 * y * w], 1),
        torch.stack([2 * x * y - 2 * z * w, 1 - 2 * x * x - 2 * z * z, 2 * y * z + 2 * x * w], 1),
        torch.stack([2 * x * z + 2 * y * w, 2 * y * z - 2 * x * w, 1 - 2 * x * x - 2 * y * y], 1)], 1)  # [P, c, r]
    M = (scale_modifier * scale)[:, :, None] * R
    S = torch.einsum("pkc,pkr->pcr", M, M)
    limx, limy = 1.3 * tfx, 1.3 * tfy
    tx = torch.clamp(vx / vz, -limx, limx) * vz
    ty = torch.clamp(vy / vz, -limy, limy) * vz
    J00, J11 = fx / vz, fy / vz
    J02, J12 = -fx * tx / (vz * vz), -fy * ty / (vz * vz)
    Vm = V.view(4, 4)  # Vm[c][r] = V[c*4 + r]; row r of mat3(view) is (V[r*4+0], V[r*4+1], V[r*4+2])
    T0 = J00[:, None] * Vm[:3, 0][None] + J02[:, None] * Vm[:3, 2][None]
    T1 = J11[:, None] * Vm[:3, 1][None] + J12[:, None] * Vm[:3, 2][None]
    c0 = torch.einsum("pi,pij,pj->p", T0, S, T0)
    c1 = torch.einsum("pi,pij,pj->p", T0, S, T1)
    c2 = torch.einsum("pi,pij,pj->p", T1, S, T1)
    a, b, c = c0 + 0.3, c1, c2 + 0.3
    inv = 1.0 / (a * c - b * b + 1e-6)
    conic = torch.stack([inv * c, -inv * b, inv * a], 1)
    # sh_color
    d = pos - cam[None]
    d = d / torch.sqrt((d * d).sum(1, keepdim=True))
    basis = sh_basis(d, deg)
    res = torch.einsum("pk,pkc->pc", basis, sh[:, :basis.shape[1]]) + 0.5
    color = torch.clamp(res, 0.0, 1.0)
    return torch.stack([mx, my], 1), conic, color, vz


def _f32_power(mx, my, conic, pxs, pys):
    """The oracle's per-pair power in float32 (fma emulated in binary64: the products of two floats are exact)."""
    f = np.float32
    dx = (mx[None, :] - pxs[:, None]).astype(f)
    dy = (my[None, :] - pys[:, None]).astype(f)
    a = (f(-0.5) * conic[:, 0]).astype(f)
    cz = (f(-0.5) * conic[:, 2]).astype(f)
    inner = ((cz[None] * dy).astype(f) * dy).astype(f)
    t = ((a[None] * dx).astype(f)).astype(np.float64) * dx.astype(np.float64) + inner.astype(np.float64)
    inner2 = t.astype(f)
    bdx = (-(conic[:, 1][None] * dx)).astype(f)
    return (bdx.astype(np.float64) * dy.astype(np.float64) + inner2.astype(np.float64)).astype(f)


def decisions(fr, opacity, W, H):
    """Per tile: (pixel x, pixel y, Gaussian ids, blended mask [pixels, entries]) from the oracle's frame, with the
    oracle's alpha test (power <= 0 and power >= alpha_threshold(opacity)) and its float32 saturation stop."""
    gx, gy = orc.grids(W, H)
    opacity = np.ascontiguousarray(opacity, np.float32)
    thr = {}
    out = []
    for t in range(gx * gy):
        s, e = int(fr.ranges[t, 0]), int(fr.ranges[t, 1])
        bx, by = t % gx, t // gx
        ys, xs = np.meshgrid(np.arange(by * 16, by * 16 + 16), np.arange(bx * 16, bx * 16 + 16), indexing="ij")
        inside = (xs < W) & (ys < H)
        xs, ys = xs[inside].ravel(), ys[inside].ravel()
        if xs.size == 0:
            continue
        ids = fr.vals_sorted[s:e].astype(np.int64) if e > s else np.zeros(0, np.int64)
        if ids.size == 0:
            out.append((xs, ys, ids, np.zeros((xs.size, 0), bool)))
            continue
        for i in ids:
            if i not in thr:
                thr[int(i)] = orc.alpha_threshold(float(opacity[i]))
        th = np.array([thr[int(i)] for i in ids], np.float32)
        pw = _f32_power(fr.means_2d[ids, 0], fr.means_2d[ids, 1], fr.conic[ids], xs.astype(np.float32), ys.astype(np.float32))
        ok = ~(pw > 0) & ~(pw < th[None])
        alpha = np.minimum(np.float32(0.99), (opacity[ids][None] * np.exp(pw.astype(np.float64)).astype(np.float32)).astype(np.float32))
        fac = np.where(ok, (np.float32(1.0) - alpha).astype(np.float32), np.float32(1.0)).astype(np.float32)
        T_after = np.multiply.accumulate(fac, axis=1, dtype=np.float32)
        sat = ok & (T_after < np.float32(1e-4))
        stop = np.where(sat.any(1), sat.argmax(1), ids.size)
        blended = ok & (np.arange(ids.size)[None] < stop[:, None])
        out.append((xs, ys, ids, blended))
    return out


def render(means, conic, color, opacity, dec, W, H, bg=(0.0, 0.0, 0.0)):
    """Planar [3, H, W] float64 image from per-Gaussian tensors and the frozen decisions."""
    bgt = torch.tensor(bg, dtype=F64)
    pixs, cols = [], []
    for xs, ys, ids, blended in dec:
        if ids.size == 0 or not blended.any():
            continue
        keep = blended.any(0)
        ids, blended = ids[keep], torch.from_numpy(blended[:, keep])
        idt = torch.from_numpy(ids)
        xt, yt = torch.from_numpy(xs.astype(np.float64)), torch.from_numpy(ys.astype(np.float64))
        dx = means[idt, 0][None] - xt[:, None]
        dy = means[idt, 1][None] - yt[:, None]
        cn = conic[idt]
        power = -0.5 * (cn[:, 0][None] * dx * dx + cn[:, 2][None] * dy * dy) - cn[:, 1][None] * dx * dy
        alpha = torch.clamp(opacity[idt][None] * torch.exp(power), max=0.99)
        alpha = torch.where(blended, alpha, torch.zeros_like(alpha))
        one_m = 1.0 - alpha
        T_excl = torch.cumprod(torch.cat([torch.ones_like(one_m[:, :1]), one_m[:, :-1]], 1), 1)
        wgt = T_excl * alpha
        T_fin = T_excl[:, -1] * one_m[:, -1]
        Cpix = wgt @ color[idt] + T_fin[:, None] * bgt[None]
        pixs.append(torch.from_numpy(xs + W * ys))
        cols.append(Cpix)
    img = bgt[:, None].expand(3, H * W)
    if pixs:
        img = img.index_put((torch.arange(3)[:, None], torch.cat(pixs)[None]), torch.cat(cols).T)
    return img.reshape(3, H, W)


def forward(pos, scale, rotq, sh, opacity, vp, fr, deg=3, bg=(0.0, 0.0, 0.0), scale_modifier=1.0, dec=None,
            keep_2d=False):
    """The whole frame: float64 tensors in, [3, H, W] image out.  keep_2d: also return (means, conic, color) with
    retain_grad() so their gradients can be compared with the optional 2D outputs."""
    if dec is None:
        dec = decisions(fr, opacity.detach().float().numpy(), vp.width, vp.height)
    means, conic, color, _ = preprocess(pos, scale, rotq, sh, vp, deg, scale_modifier)
    if keep_2d:
        for t in (means, conic, color):
            t.retain_grad()
    img = render(means, conic, color, opacity, dec, vp.width, vp.height, bg)
    return (img, (means, conic, color)) if keep_2d else img


def leaf(a):
    return torch.tensor(np.ascontiguousarray(a, np.float64), dtype=F64, requires_grad=True)
