"""Cost of the per-pixel aux planes (alpha / depth / contributor count) on the C3 frame (5.8 M Gaussians, 1920x1080).

One Device, one Renderer: after a warm-up, alternating blocks of frames with the aux planes off and on (the same
renderer, only the three frame pointers change).  Every frame is profiled with CUDA events (lcgs_b200_stage_times);
the blend stage and the whole frame are reported per block, and as median and spread over the alternations.  Prints one
JSON line with the GPU's name and power limit, read in the same run.

    python scripts/aux_cost.py [--alternations 7] [--frames 20] [--warmup 10] [--out aux_cost.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from luisacomputegaussiansplatting_b200 import lcgs, scenes  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")] if q.returncode == 0 else ("?", "?", "?")
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--alternations", type=int, default=7)
    ap.add_argument("--frames", type=int, default=20, help="frames per block")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.alternations < 5:
        ap.error("at least 5 alternations")

    sc, cfg = scenes.make_config_scene("C3")
    dev = lcgs.Device(0)
    r = lcgs.Renderer(dev, sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, cfg.W, cfg.H, list_capacity=20_000_000, rgb8=True,
                      aux=True)
    vp = lcgs.view_params(lcgs.make_camera(scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world), cfg.W, cfg.H))
    f = r.c_frame
    planes = (r.alpha_map.data_ptr(), r.depth_plane.data_ptr(), r.n_contrib_map.data_ptr())

    def set_aux(on):
        f.target_alpha, f.target_depth, f.target_n_contrib = planes if on else (None, None, None)

    def block(on, n):
        set_aux(on)
        blend, frame = [], []
        for _ in range(n):
            r.render_async(vp)
            st = dev.stage_times()
            blend.append(st["blend"])
            frame.append(sum(st.values()))
        dev.num_rendered()
        return statistics.median(blend), statistics.median(frame)

    dev.set_profiling(True)
    block(False, a.warmup)
    block(True, a.warmup)
    rows = []
    for i in range(a.alternations):
        off = block(False, a.frames)
        on = block(True, a.frames)
        rows.append(dict(blend_off_ms=off[0], blend_on_ms=on[0], frame_off_ms=off[1], frame_on_ms=on[1]))
    dev.set_profiling(False)
    torch.cuda.synchronize()

    def summary(key):
        v = [row[key] for row in rows]
        return dict(median=statistics.median(v), min=min(v), max=max(v))

    blend_cost = [row["blend_on_ms"] / row["blend_off_ms"] - 1.0 for row in rows]
    frame_cost = [row["frame_on_ms"] / row["frame_off_ms"] - 1.0 for row in rows]
    res = dict(metric="aux_planes_cost", config="C3", W=cfg.W, H=cfg.H, gaussians=sc.num_gaussians,
               num_rendered=dev.num_rendered(), alternations=a.alternations, frames_per_block=a.frames,
               blend_off_ms=summary("blend_off_ms"), blend_on_ms=summary("blend_on_ms"),
               frame_off_ms=summary("frame_off_ms"), frame_on_ms=summary("frame_on_ms"),
               blend_cost_rel=dict(median=statistics.median(blend_cost), min=min(blend_cost), max=max(blend_cost)),
               frame_cost_rel=dict(median=statistics.median(frame_cost), min=min(frame_cost), max=max(frame_cost)),
               blocks=rows, **gpu_info())
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    dev.close()


if __name__ == "__main__":
    main()
