"""The float64 torch reference (tests/torch_reference.py) with the camera pose as differentiable inputs: preprocess() and
forward() take the view matrix (the 16 entries of vp.view, column-major) and the camera position as float64 tensors,
so that torch autograd gives dL/dview and dL/dcam_pos.  The intrinsics (proj, tanfov, focal) and the resolution come
from vp and are held fixed.  With vp's own view and camera position the results equal torch_reference's."""
from __future__ import annotations

import numpy as np
import torch

import torch_reference as tr

F64 = tr.F64


def preprocess(pos, scale, rotq, sh, vp, view, cam_pos, deg: int = 3, scale_modifier: float = 1.0):
    """torch_reference.preprocess with V = view [16] and the SH view origin cam_pos [3] as tensors.  Returns (means
    [P,2] pixels, conic [P,3], color [P,3], depth [P])."""
    _, proj, tfx, tfy, fx, fy, _ = tr._vp(vp)
    V, cam = view, cam_pos
    W, H = vp.width, vp.height
    vx = pos[:, 0] * V[0] + pos[:, 1] * V[4] + pos[:, 2] * V[8] + V[12]
    vy = pos[:, 0] * V[1] + pos[:, 1] * V[5] + pos[:, 2] * V[9] + V[13]
    vz = pos[:, 0] * V[2] + pos[:, 1] * V[6] + pos[:, 2] * V[10] + V[14]
    p_w = 1.0 / (vz + 1e-6)
    ndc_x, ndc_y = vx * proj[0] * p_w, vy * proj[5] * p_w
    mx = ((ndc_x + 1.0) * W - 1.0) * 0.5
    my = ((ndc_y + 1.0) * H - 1.0) * 0.5
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
    Vm = V.view(4, 4)  # Vm[c][r] = V[c*4 + r]
    T0 = J00[:, None] * Vm[:3, 0][None] + J02[:, None] * Vm[:3, 2][None]
    T1 = J11[:, None] * Vm[:3, 1][None] + J12[:, None] * Vm[:3, 2][None]
    c0 = torch.einsum("pi,pij,pj->p", T0, S, T0)
    c1 = torch.einsum("pi,pij,pj->p", T0, S, T1)
    c2 = torch.einsum("pi,pij,pj->p", T1, S, T1)
    a, b, c = c0 + 0.3, c1, c2 + 0.3
    inv = 1.0 / (a * c - b * b + 1e-6)
    conic = torch.stack([inv * c, -inv * b, inv * a], 1)
    d = pos - cam[None]
    d = d / torch.sqrt((d * d).sum(1, keepdim=True))
    basis = tr.sh_basis(d, deg)
    res = torch.einsum("pk,pkc->pc", basis, sh[:, :basis.shape[1]]) + 0.5
    color = torch.clamp(res, 0.0, 1.0)
    return torch.stack([mx, my], 1), conic, color, vz


def forward(pos, scale, rotq, sh, opacity, vp, fr, view, cam_pos, deg=3, bg=(0.0, 0.0, 0.0), scale_modifier=1.0,
            dec=None):
    """torch_reference.forward with the pose tensors: the [3, H, W] float64 image over the oracle's frozen decisions."""
    if dec is None:
        dec = tr.decisions(fr, opacity.detach().float().numpy(), vp.width, vp.height)
    means, conic, color, _ = preprocess(pos, scale, rotq, sh, vp, view, cam_pos, deg, scale_modifier)
    return tr.render(means, conic, color, opacity, dec, vp.width, vp.height, bg)


def vp_pose(vp):
    """vp's own view [16] and camera position [3] as float64 leaf tensors that require grad."""
    return (torch.tensor(np.asarray(list(vp.view), np.float64), requires_grad=True),
            torch.tensor(np.asarray(list(vp.cam_pos), np.float64), requires_grad=True))
