"""Cost of the backward pass on the C3 frame (run on its own: nothing else on the GPU).

Times, with CUDA events over blocks of frames, the forward with the intermediates the backward needs
(lcgs_b200_render with means_2d / conic / color kept) and the backward (lcgs_b200_render_backward), and splits the
backward into its kernels -- record rebuild (+ tile order and the gradient clear), blend backward, preprocess
backward -- with torch.profiler in a separate pass.  Records the card name and power limit.  Writes
profiles/r04_backward_cost_c3.json (or --out)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from luisacomputegaussiansplatting_b200 import lcgs, scenes  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return dict(gpu=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # noqa: BLE001
        return dict(gpu=torch.cuda.get_device_name(0), power_limit="unknown (%s)" % e)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_backward_cost_c3.json"))
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
    g = lcgs._capi.Grad()
    g.dl_dimg = dl.data_ptr()
    for k, t in outs.items():
        setattr(g, "grad_" + k, t.data_ptr())

    def fwd():
        dev.check(dev.lib.lcgs_b200_render(dev.ctx, C.byref(r.c_scene), C.byref(vp), C.byref(r.c_frame), None))

    def bwd():
        dev.check(dev.lib.lcgs_b200_render_backward(dev.ctx, C.byref(r.c_scene), C.byref(vp), C.byref(r.c_frame), C.byref(g), None))

    def timed(fn):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        for _ in range(args.frames):
            fn()
        ev[1].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1]) / args.frames

    for _ in range(20):
        fwd(); bwd()
    torch.cuda.synchronize()
    f_ms, b_ms = [], []
    for _ in range(args.blocks):  # alternated blocks
        f_ms.append(timed(fwd))
        b_ms.append(timed(bwd))

    from torch.profiler import ProfilerActivity, profile
    fwd()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(20):
            bwd()
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" or getattr(e, "device_time_total", 0) > 0:
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            per[e.key] = per.get(e.key, 0.0) + t / 20.0 / 1000.0
    split = {"record_rebuild": 0.0, "blend_backward": 0.0, "preprocess_backward": 0.0, "other": 0.0}
    for k, v in per.items():
        if "build_records" in k or "tile_order" in k or "Memset" in k or "memset" in k:
            split["record_rebuild"] += v
        elif "blend_backward" in k:
            split["blend_backward"] += v
        elif "preprocess_backward" in k:
            split["preprocess_backward"] += v
        else:
            split["other"] += v
    res = dict(card(), scene="C3", width=W, height=H, num_gaussians=int(r.P), num_rendered=int(n),
               forward_ms=dict(median=float(np.median(f_ms)), blocks=f_ms),
               backward_ms=dict(median=float(np.median(b_ms)), blocks=b_ms),
               backward_split_ms=split, backward_kernels_ms=per,
               note="forward = lcgs_b200_render with means_2d/conic/color kept; backward = lcgs_b200_render_backward with "
                    "pos/scale/rotq/sh/opacity gradients; record_rebuild includes the gradient clear and the tile order")
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    dev.close()


if __name__ == "__main__":
    main()
