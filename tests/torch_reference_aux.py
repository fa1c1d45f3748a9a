"""The float64 torch reference (tests/torch_reference.py) with the blend's aux planes: render_aux() blends over the
oracle's frozen decisions like torch_reference.render() and also returns the accumulated opacity 1 - T and the depth
plane sum w_i z_i, the view depth z being torch_reference.preprocess()'s fourth output."""
from __future__ import annotations

import numpy as np
import torch

import torch_reference as tr

F64 = tr.F64


def render_aux(means, conic, color, depth, opacity, dec, W, H, bg=(0.0, 0.0, 0.0)):
    """([3, H, W] image, [H, W] alpha, [H, W] depth plane), float64, from per-Gaussian tensors and the decisions."""
    bgt = torch.tensor(bg, dtype=F64)
    pixs, cols, alps, deps = [], [], [], []
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
        cols.append(wgt @ color[idt] + T_fin[:, None] * bgt[None])
        alps.append(1.0 - T_fin)
        deps.append(wgt @ depth[idt])
        pixs.append(torch.from_numpy(xs + W * ys))
    img = bgt[:, None].expand(3, H * W)
    alpha_map = torch.zeros(H * W, dtype=F64)
    depth_map = torch.zeros(H * W, dtype=F64)
    if pixs:
        idx = torch.cat(pixs)
        img = img.index_put((torch.arange(3)[:, None], idx[None]), torch.cat(cols).T)
        alpha_map = alpha_map.index_put((idx,), torch.cat(alps))
        depth_map = depth_map.index_put((idx,), torch.cat(deps))
    return img.reshape(3, H, W), alpha_map.reshape(H, W), depth_map.reshape(H, W)


def forward_aux(pos, scale, rotq, sh, opacity, vp, fr, deg=3, bg=(0.0, 0.0, 0.0), scale_modifier=1.0, dec=None):
    """The whole frame: float64 tensors in, (image [3, H, W], alpha [H, W], depth plane [H, W], (means, conic, color,
    view depth)) out.  The per-Gaussian tensors have retain_grad(), for comparison with the optional 2D outputs and
    grad_depth (dL/d(view depth) through the blend only, as grad_means_2d is through the blend only)."""
    if dec is None:
        dec = tr.decisions(fr, opacity.detach().float().numpy(), vp.width, vp.height)
    means, conic, color, vz = tr.preprocess(pos, scale, rotq, sh, vp, deg, scale_modifier)
    # vz also feeds the means and the conic: the blend's own view-depth input is a node of its own, so that its
    # gradient is the blend's part only, like grad_depth's
    depth = vz.clone()
    for t in (means, conic, color, depth):
        t.retain_grad()
    img, alpha, dmap = render_aux(means, conic, color, depth, opacity, dec, vp.width, vp.height, bg)
    return img, alpha, dmap, (means, conic, color, depth)
