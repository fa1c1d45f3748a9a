"""Cost of the camera-pose gradient on the C3 frame (run on its own: nothing else on the GPU).

Times, with CUDA events over alternated blocks of frames, lcgs_b200_render_backward with the five scene gradients,
without and with grad_view / grad_cam_pos, and splits both into their kernels with torch.profiler in a separate pass
(preprocess_backward_kernel against preprocess_pose_grad_kernel + pose_grad_reduce_kernel).  Also times the tracking
call (pose outputs only).  Records the card name and power limit.  Writes profiles/r06_pose_backward_cost_c3.json (or
--out)."""
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
    ap.add_argument("--frames", type=int, default=100)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_pose_backward_cost_c3.json"))
    args = ap.parse_args()
    sc, cfg = scenes.make_config_scene("C3")
    W, H = cfg.W, cfg.H
    dev = lcgs.Device(0)
    r = lcgs.Renderer(dev, sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, W, H, list_capacity=20_000_000)
    vp = lcgs.view_params(lcgs.make_camera(scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world), W, H))
    r.render_async(vp)
    n = dev.num_rendered()
    dl = torch.rand(3 * W * H, device="cuda")
    outs = {k: torch.empty_like(t) for k, t in zip(("pos", "scale", "rotq", "sh", "opacity"), (r.pos, r.scale, r.rotq, r.sh, r.opacity))}
    gv, gc = torch.empty(16, device="cuda"), torch.empty(3, device="cuda")

    def grad(scene, pose):
        g = lcgs._capi.Grad()
        g.dl_dimg = dl.data_ptr()
        if scene:
            for k, t in outs.items():
                setattr(g, "grad_" + k, t.data_ptr())
        if pose:
            g.grad_view, g.grad_cam_pos = gv.data_ptr(), gc.data_ptr()
        return g

    calls = {"scene": grad(True, False), "scene_and_pose": grad(True, True), "pose_only": grad(False, True)}

    def bwd(g):
        dev.check(dev.lib.lcgs_b200_render_backward(dev.ctx, C.byref(r.c_scene), C.byref(vp), C.byref(r.c_frame), C.byref(g), None))

    def timed(g):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        for _ in range(args.frames):
            bwd(g)
        ev[1].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1]) / args.frames

    for _ in range(10):
        for g in calls.values():
            bwd(g)
    torch.cuda.synchronize()
    ms = {k: [] for k in calls}
    for _ in range(args.blocks):  # alternated blocks
        for k, g in calls.items():
            ms[k].append(timed(g))

    from torch.profiler import ProfilerActivity, profile
    kernels = {}
    for k, g in calls.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(20):
                bwd(g)
            torch.cuda.synchronize()
        per = {}
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            if t > 0:
                per[e.key] = per.get(e.key, 0.0) + t / 20.0 / 1000.0
        kernels[k] = per

    def pick(k, part):
        return sum(v for name, v in kernels[k].items() if part in name)

    base = pick("scene", "preprocess_backward_kernel")
    pose_k = pick("scene_and_pose", "preprocess_pose_grad_kernel")
    res = dict(card(), scene="C3", width=W, height=H, num_gaussians=int(r.P), num_rendered=int(n),
               backward_ms={k: dict(median=float(np.median(v)), blocks=v) for k, v in ms.items()},
               preprocess_backward_kernel_ms=base, preprocess_pose_grad_kernel_ms=pose_k,
               pose_over_preprocess_backward=pose_k / base if base else None,
               pose_grad_reduce_kernel_us=1000.0 * pick("scene_and_pose", "pose_grad_reduce_kernel"),
               kernels_ms=kernels,
               note="lcgs_b200_render_backward on the C3 frame: 'scene' = pos/scale/rotq/sh/opacity gradients, "
                    "'scene_and_pose' = the same plus grad_view and grad_cam_pos, 'pose_only' = grad_view and "
                    "grad_cam_pos alone (tracking against a frozen scene); CUDA events over alternated blocks")
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    dev.close()


if __name__ == "__main__":
    main()
