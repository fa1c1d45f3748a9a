"""Cost of the backward through the alpha and depth planes on the C3 frame (run on its own: nothing else on the GPU).

Renders the C3 frame once with the aux planes (Renderer(aux=True)), then times, with CUDA events over alternated blocks
of calls, lcgs_b200_render_backward on that frame without (image only: blend_backward_kernel) and with dl_dalpha and
dl_ddepth (blend_backward_aux_kernel), every scene gradient and grad_depth requested.  The blend kernels alone are
timed with torch.profiler in a separate pass.  Records the card name and power limit.  Writes
profiles/r05_aux_backward_cost_c3.json (or --out)."""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from backward_cost import card  # noqa: E402
from luisacomputegaussiansplatting_b200 import lcgs, scenes  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_aux_backward_cost_c3.json"))
    args = ap.parse_args()
    sc, cfg = scenes.make_config_scene("C3")
    W, H = cfg.W, cfg.H
    dev = lcgs.Device(0)
    r = lcgs.Renderer(dev, sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, W, H, list_capacity=20_000_000, aux=True)
    vp = lcgs.view_params(lcgs.make_camera(scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world), W, H))
    r.render_async(vp)
    n = dev.num_rendered()
    dl = torch.rand(3 * W * H, device="cuda")
    da = torch.rand(W * H, device="cuda")
    dd = torch.rand(W * H, device="cuda")
    outs = {k: torch.empty_like(t) for k, t in zip(("pos", "scale", "rotq", "sh", "opacity"), (r.pos, r.scale, r.rotq, r.sh, r.opacity))}
    outs["depth"] = torch.empty_like(r.opacity)

    def grad(aux):
        g = lcgs._capi.Grad()
        g.dl_dimg = dl.data_ptr()
        for k, t in outs.items():
            setattr(g, "grad_" + k, t.data_ptr())
        if aux:
            g.dl_dalpha, g.dl_ddepth = da.data_ptr(), dd.data_ptr()
        return g

    g_img, g_aux = grad(False), grad(True)

    def bwd(g):
        dev.check(dev.lib.lcgs_b200_render_backward(dev.ctx, C.byref(r.c_scene), C.byref(vp), C.byref(r.c_frame), C.byref(g), None))

    def timed(g):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        for _ in range(args.calls):
            bwd(g)
        ev[1].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1]) / args.calls

    for _ in range(20):
        bwd(g_img); bwd(g_aux)
    torch.cuda.synchronize()
    img_ms, aux_ms = [], []
    for _ in range(args.blocks):  # alternated blocks
        img_ms.append(timed(g_img))
        aux_ms.append(timed(g_aux))

    from torch.profiler import ProfilerActivity, profile
    kern = {}
    for name, g in (("image_only", g_img), ("aux", g_aux)):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(20):
                bwd(g)
            torch.cuda.synchronize()
        for e in prof.key_averages():
            if "blend_backward" in e.key or "preprocess_backward" in e.key:
                t = getattr(e, "device_time_total", None)
                if t is None:
                    t = e.cuda_time_total
                kern["%s: %s" % (name, e.key)] = t / 20.0 / 1000.0
    res = dict(card(), scene="C3", width=W, height=H, num_gaussians=int(r.P), num_rendered=int(n),
               backward_image_only_ms=dict(median=float(np.median(img_ms)), blocks=img_ms),
               backward_aux_ms=dict(median=float(np.median(aux_ms)), blocks=aux_ms),
               aux_over_image_only=float(np.median(aux_ms) / np.median(img_ms)),
               kernels_ms=kern,
               note="lcgs_b200_render_backward on one aux-rendered C3 frame, pos/scale/rotq/sh/opacity/depth gradients; "
                    "image_only = dl_dalpha = dl_ddepth = NULL (blend_backward_kernel), aux = both set "
                    "(blend_backward_aux_kernel); blocks of calls alternated")
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    dev.close()


if __name__ == "__main__":
    main()
