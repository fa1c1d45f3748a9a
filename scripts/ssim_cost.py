"""Cost of the SSIM loss (lcgs_b200_ssim) on one B200 (run on its own: nothing else on the GPU).

Times, with CUDA events over warmed-up, alternated blocks of calls:
- lcgs_b200_ssim without and with the gradient at 1920x1080 and 7680x4320 (per-kernel split by torch.profiler in a
  separate pass);
- the float32 torch formulation (five depthwise 11x11 conv2d, tests/torch_reference_ssim.py) forward + backward, with
  TF32 off and on;
- one C3 training step (DifferentiableRenderer forward, loss, backward) with an L1 loss only, with
  0.8 L1 + 0.2 (1 - lcgs.ssim) and with the same loss on the torch SSIM.
Reports the spread of the blocks, the achieved bytes/s of the algorithm's traffic, and the share of the bound computed
from shapes (the larger of bytes over the HBM peak and FMAs over the FP32 peak).  Records the card name and power
limit.  Writes profiles/r07_ssim_cost.json (or --out)."""
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

from backward_cost import card  # noqa: E402
from luisacomputegaussiansplatting_b200 import lcgs, scenes  # noqa: E402
import torch_reference_ssim as rs  # noqa: E402

HBM_GBS = 6552.0  # DESIGN §6's HBM figure (MEASURED_PEAKS.json hbm_gbs where the machine provides it)
TILE, HALO = 32, 42


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return HBM_GBS, "DESIGN §6 figure (6552 GB/s)"


def traffic(W, H, grad):
    """(bytes, FMAs) the kernels need, from shapes: image and reference read once per pass, the partial maps written
    and read once (36 B/px), the gradient written once; FMAs of the taps (the horizontal pass covers the 42 staged rows
    of each 32-row tile) plus the products x^2, y^2, xy per tap."""
    px = W * H
    fwd_b, bwd_b = 24 * px + (36 * px if grad else 0), (36 + 24 + 12) * px
    rows = HALO / TILE
    fwd_f = 3 * px * (rows * 11 * (5 + 3) + 11 * 5)
    bwd_f = 3 * px * (rows * 11 * 3 + 11 * 3 + 2)
    return (fwd_b + (bwd_b if grad else 0)), (fwd_f + (bwd_f if grad else 0))


def timed(fn, n):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(n):
        fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / n


def alternate(calls, n, blocks, warmup=5):
    for _ in range(warmup):
        for fn in calls.values():
            fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in calls}
    for _ in range(blocks):
        for k, fn in calls.items():
            ms[k].append(timed(fn, n))
    return {k: dict(median=float(np.median(v)), min=float(min(v)), max=float(max(v)),
                    spread=float((max(v) - min(v)) / np.median(v)), blocks=v) for k, v in ms.items()}


def kernel_split(fn, n=20):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            per[e.key] = per.get(e.key, 0.0) + t / n / 1000.0
    return per


def torch_ssim_step(x, y):
    xr = x.detach().requires_grad_()
    rs.ssim_torch(xr, y).backward()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_ssim_cost.json"))
    args = ap.parse_args()
    dev = lcgs.Device(0)
    info = card()
    props = torch.cuda.get_device_properties(0)
    peak_gbs, peak_src = hbm_peak()
    try:
        mhz = float(str(info.get("max_sm_clock", "")).split()[0])
    except Exception:  # noqa: BLE001
        mhz = 1965.0
    fp32_tflops = props.multi_processor_count * 128 * 2 * mhz * 1e6 / 1e12
    res = dict(info, hbm_peak_GBps=peak_gbs, hbm_peak_source=peak_src, fp32_peak_TFLOPs=fp32_tflops,
               fp32_peak_source="derived: %d SMs x 128 FP32 lanes x 2 x %.0f MHz (max SM clock)"
                                % (props.multi_processor_count, mhz), sizes={})
    stream = lambda: torch.cuda.current_stream().cuda_stream or None  # noqa: E731
    for W, H in [(1920, 1080), (7680, 4320)]:
        g = torch.Generator(device="cuda").manual_seed(W)
        x = torch.rand(3, H, W, device="cuda", generator=g)
        y = torch.rand(3, H, W, device="cuda", generator=g)
        out, grad = torch.empty((), device="cuda"), torch.empty_like(x)

        def ours(gr):
            return lambda: dev.check(dev.lib.lcgs_b200_ssim(dev.ctx, W, H, x.data_ptr(), y.data_ptr(), out.data_ptr(),
                                                            gr, stream()))

        calls = {"lcgs_value": ours(None), "lcgs_value_and_grad": ours(grad.data_ptr())}
        ms = alternate(calls, args.calls, args.blocks)
        torch_calls = {}
        for tf32 in (False, True):
            def t(tf32=tf32):
                torch.backends.cudnn.allow_tf32 = tf32
                torch_ssim_step(x, y)
            torch_calls["torch_fp32_fwd_bwd_tf32_%s" % ("on" if tf32 else "off")] = t
        ms.update(alternate(torch_calls, max(args.calls // 5, 5), args.blocks, warmup=3))
        torch.backends.cudnn.allow_tf32 = True
        entry = dict(calls_ms=ms)
        for k, gr in (("lcgs_value", False), ("lcgs_value_and_grad", True)):
            b, f = traffic(W, H, gr)
            t = ms[k]["median"] * 1e-3
            t_bytes, t_fma = b / (peak_gbs * 1e9), 2 * f / (fp32_tflops * 1e12)
            entry[k] = dict(alg_bytes=b, alg_fma=f, achieved_GBps=b / t / 1e9, achieved_TFLOPs=2 * f / t / 1e12,
                            bound_us=1e6 * max(t_bytes, t_fma), bound_by="hbm" if t_bytes >= t_fma else "fp32",
                            share_of_bound=max(t_bytes, t_fma) / t)
        entry["kernels_ms"] = kernel_split(calls["lcgs_value_and_grad"])
        res["sizes"]["%dx%d" % (W, H)] = entry
        del x, y, grad
        torch.cuda.empty_cache()

    # one C3 training step: render, loss, backward
    sc, cfg = scenes.make_config_scene("C3")
    W, H = cfg.W, cfg.H
    cam = lcgs.make_camera(scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world), W, H)
    dr = lcgs.DifferentiableRenderer(dev, W, H, list_capacity=20_000_000)
    leaves = [torch.tensor(a, device="cuda", requires_grad=True) for a in (sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity)]
    with torch.no_grad():
        target = (dr(*leaves, cam) + 0.05 * torch.rand(3, H, W, device="cuda")).clamp(0, 1)

    def step(kind):
        def run():
            for t in leaves:
                t.grad = None
            img = dr(*leaves, cam)
            l1 = (img - target).abs().mean()
            if kind == "l1":
                loss = l1
            elif kind == "lcgs_ssim":
                loss = 0.8 * l1 + 0.2 * (1.0 - lcgs.ssim(dev, img, target))
            else:
                loss = 0.8 * l1 + 0.2 * (1.0 - rs.ssim_torch(img, target))
            loss.backward()
        return run

    torch.backends.cudnn.allow_tf32 = False
    res["c3_training_step_ms"] = alternate({k: step(k) for k in ("l1", "lcgs_ssim", "torch_ssim_tf32_off")},
                                           args.steps, args.blocks, warmup=3)
    res["note"] = ("lcgs_b200_ssim on uniform random images (both planes larger than L2 at 7680x4320, not at 1920x1080); "
                   "CUDA events over alternated blocks after warm-up; the torch formulation is tests/torch_reference_ssim.py "
                   "in float32 with cuDNN TF32 off / on; the C3 step is DifferentiableRenderer forward + loss + backward "
                   "(five scene gradients), torch SSIM with TF32 off")
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    dev.close()


if __name__ == "__main__":
    main()
