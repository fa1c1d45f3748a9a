#!/usr/bin/env python
"""bench.py -- forward splat-render benchmark (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config C1|C2|C3|C4|C5] [--shard views|rows]
                    [--dump-outputs DIR]

Workloads (BASELINE.json:configs; synthetic scenes of SURVEY.md 8d, the release .ply files are not available offline):

  N = 1 (default)  C3: ONE frame per step of the mip360_garden-shaped scene (5.8 M SH3 Gaussians, 1920x1080, the
                   reference's hard-coded camera, list capacity 20 M) -- the configuration the metric is quoted on.
                   The line also carries `orbit_n1`: the C4 workload on this one GPU, so that a scaling file has the
                   single-GPU number of the workload the N > 1 lines measure.
  N > 1 (default)  C4: the 256-view orbit of the mip360_bicycle-shaped scene (6.1 M Gaussians, 1237x822), view-sharded:
                   one step = N views, view f of the run on rank f mod N, Gaussian set replicated.  Every rank blends
                   straight into rank 0's peer-mapped frame ring over NVLink (the gather is the blend's stores),
                   hands each frame over with a device-side sequence flag, and rank 0 CONSUMES every frame inside
                   the timed region (a checksum kernel reads the whole slot) before it releases the slot -- ring flow
                   control entirely in stream order.  Weak scaling.
  --config C5 --shard rows   ONE 7680x4320 frame of the 10 M-Gaussian scene per step, split by tile rows over the N
                   ranks (bands balanced by instance count, preprocess replicated), all bands blended into the same
                   ring slot on rank 0, consumed there.  Strong scaling.

One JSON line on rank 0:
  value      Gaussians/s, whole job, device-timed (CUDA events on the launching streams, max over ranks)
  e2e        the same metric through the public API with the per-frame host traffic inside the timed region: camera
             parameters in from host memory; finished image (the app's uint8 HWC image, written by the blend kernel's
             epilogue) and num_rendered out to pinned host memory, consumed by the host; wall clock, max over ranks.
             N > 1: rank 0 reads every delivered frame of every rank from its ring.
  roofline   the time-dominant kernel (the blend: FP32 issue bound) per SURVEY.md 8d; roofline_sort = the dominant
             HBM kernel (onesweep pass); stages = per-stage ms and achieved GB/s against the measured HBM peak
  cpu_baseline  the CPU oracle (a port of the reference's algorithm; the reference itself cannot be built offline)
             on all host cores of this box, same scene and camera, whole frames

--impl reference times the CPU oracle alone (rank 0 only), whole frames on all host cores.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "gaussians_per_second_forward_render"
UNIT = "Gaussians/s"
ORBIT_VIEWS = 256
FP32_LANES_PER_SM = 128


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default=None, choices=["C1", "C2", "C3", "C4", "C5"],
                    help="default: C3 on one GPU, C4 (view-sharded orbit) on several")
    ap.add_argument("--shard", default=None, choices=["views", "rows"], help="default: rows for C5, views otherwise")
    ap.add_argument("--gaussians", type=int, default=None, help="override P (debugging only; invalidates the number)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-orbit", action="store_true", help="N = 1: skip the orbit_n1 leg")
    ap.add_argument("--capacity", type=int, default=None, help="instance list capacity L per rank")
    ap.add_argument("--deliver", default="rgb8", choices=["rgb8", "float"],
                    help="sharded workloads: what a rank writes into rank 0's ring -- rgb8: the app's final uint8 HWC image (3 B/pixel over "
                         "NVLink, the float image stays local); float: the planar float32 image as well (15 B/pixel)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float32 or float64, %d MB at most in all; "
                         "larger outputs as a seeded sample, see DIR/manifest.json) to compare two builds" % (DUMP_BUDGET_BYTES // 10**6))
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    return args


def resolve_workload(args, world):
    if args.config is None:
        args.config = "C3" if world == 1 else "C4"
    if args.shard is None:
        args.shard = "rows" if args.config == "C5" else "views"
    if args.capacity is None:
        if args.config == "C5":
            # whole frame: 234 M instances; a band of an 8-way split: ~30 M once balanced, but the calibration frame
            # runs on uniform bands
            args.capacity = 260_000_000 if world == 1 else 160_000_000
        elif args.config == "C4":
            args.capacity = 30_000_000
        else:
            args.capacity = 20_000_000   # app/main.cpp:245
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def scene_key(config):
    return "C2" if config == "C4" else config


def orbit_view(frame_index, total_frames):
    """Orbit view rendered as frame `frame_index` of a run of `total_frames`: the run always spans the whole 256-view
    orbit (evenly spaced views when it is shorter, wrapping around when it is longer)."""
    if total_frames >= ORBIT_VIEWS:
        return frame_index % ORBIT_VIEWS
    return (frame_index * ORBIT_VIEWS) // total_frames


def workload_config(args, cfg, P, world, extra=None):
    if args.config == "C4":
        what = ("C4: %d-view orbit of the %s scene (SURVEY.md 8d orbit), view f on rank f mod N" % (ORBIT_VIEWS, cfg.description))
        par = ("view-sharded x%d: scene replicated, frames blended straight into rank 0's peer-mapped ring over NVLink, "
               "device-side ready/consumed flags, rank 0 checksums every frame inside the timed region" % world) if world > 1 \
            else "single GPU (same ring / flag / consume path, all local)"
    elif args.shard == "rows":
        what = "%s: %s, reference camera (app/main.cpp:191-202), one frame split by tile rows" % (cfg.key, cfg.description)
        par = ("tile-row-sharded x%d: preprocess replicated, bands balanced by instance count, all bands blended into one "
               "ring slot on rank 0, consumed there" % world)
    else:
        what = "%s: %s, reference camera (app/main.cpp:191-202)" % (cfg.key, cfg.description)
        par = "single GPU" if world == 1 else "replicas x%d" % world
    c = {"workload": what + ", list capacity %d" % args.capacity,
         "gaussians": P, "width": cfg.W, "height": cfg.H, "sh_degree": 3,
         "l2": "inputs (%.2f GB Gaussian set + instance lists) exceed the 126 MB L2; no explicit flush" % (P * 236 / 1e9)}
    if extra:
        c.update(extra)
    return c, par


# ------------------------------------------------------------------------------------------------
# CPU legs (oracle): cpu_baseline of the b200 arm and the whole --impl reference arm
# ------------------------------------------------------------------------------------------------

def oracle_frames(sc, cfg, poses, warm, capacity):
    """Times the oracle's whole frame (all Gaussians, all host cores) for each pose after `warm` warm-up frames."""
    from oracle import oracle as orc

    orc.set_num_threads(os.cpu_count() or 1)   # torchrun exports OMP_NUM_THREADS=1: the baseline uses the host's cores
    times, stages, n, stats = [], None, 0, None
    for i, pose in enumerate(poses):
        vp = orc.view_params(orc.make_camera(*pose, cfg.W, cfg.H))
        t0 = time.perf_counter()
        fr = orc.forward(sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, vp, capacity=capacity)
        dt = time.perf_counter() - t0
        if i >= warm:
            times.append(dt)
            stages, n, stats = fr.stage_ms, fr.num_rendered, orc.blend_stats()
        del fr
    return times, stages, n, stats, orc.num_threads()


def reference_poses(args, cfg, count):
    from luisacomputegaussiansplatting_b200 import scenes
    if args.config == "C4":
        return [scenes.orbit_pose(orbit_view(f, count)) for f in range(count)]
    return [(scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world))] * count


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return 0
    resolve_workload(args, world)
    from luisacomputegaussiansplatting_b200 import scenes

    sc, cfg = scenes.make_config_scene(scene_key(args.config), P=args.gaussians)
    P = sc.num_gaussians
    cap = max(args.capacity, 40_000_000)
    # whole frames only, never a sub-sample of the Gaussians: if K + W frames would take more than ~4 minutes,
    # time fewer frames
    probe, _, _, _, cores = oracle_frames(sc, cfg, reference_poses(args, cfg, 1), 0, cap)
    steps, warm = args.steps, args.warmup
    budget = 240.0
    if probe[0] * (steps + warm) > budget:
        warm = 1 if warm > 0 else 0
        steps = max(1, min(steps, int(budget / probe[0]) - warm))
    poses = reference_poses(args, cfg, steps + warm)
    times, stages, n, stats, cores = oracle_frames(sc, cfg, poses, warm, cap)
    sec = float(np.sum(times))
    value = P * len(times) / sec
    sample = "%d whole frames (all %d Gaussians, %dx%d) of the same workload, %d OpenMP threads, oracle stages ms %s" % (
        len(times), P, cfg.W, cfg.H, cores, json.dumps({k: round(v, 1) for k, v in stages.items()}))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
        "steps_requested": args.steps, "warmup": warm, "ms_per_step": sec / len(times) * 1e3, "higher_is_better": True,
        "scaling": "strong" if args.shard == "rows" else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, cfg, P, world)[0],
        "note": "CPU oracle port of the reference path on the host cores (rank 0 only); the reference itself cannot be built "
                "offline (LuisaCompute + lcpp are network dependencies)",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "num_rendered": n,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------
# --dump-outputs: what the last timed step computed, so that two builds can be compared output for output
# ------------------------------------------------------------------------------------------------

DUMP_BUDGET_BYTES = 64 * 10**6
DUMP_SEED = 0


def capture_frame(r, n, img=True, rgb8=True):
    """Device copies of the frame `r` has just rendered, as its caller receives it: num_rendered, the planar image, the
    uint8 image and the frame buffers of app/main.cpp:232-254 except the two unsorted instance lists (the sort's
    input).  Returns name -> (array, numpy dtype of its elements)."""
    import torch

    f32, u32 = np.float32, np.uint32
    bufs = {"depth": (r.depth, f32), "radii": (r.radii, np.int32), "tiles_touched": (r.tiles_touched, u32),
            "offsets": (r.point_offsets, u32), "keys_sorted": (r.keys[:n], np.uint64), "vals_sorted": (r.vals[:n], u32),
            "ranges": (r.ranges[:2 * r.num_tiles].view(-1, 2), u32)}
    if img:
        bufs["img"] = (r.img.view(3, r.H, r.W), f32)
    if rgb8 and r.rgb8 is not None:
        bufs["rgb8"] = (r.rgb8.view(r.H, r.W, 3), np.uint8)
    if r.conic is not None:
        bufs.update(means_2d=(r.means_2d.view(-1, 2), f32), conic=(r.conic.view(-1, 3), f32), color=(r.color.view(-1, 3), f32))
    out = {k: (t.clone(), dt) for k, (t, dt) in bufs.items()}
    out["num_rendered"] = (torch.tensor([n], dtype=torch.int64), np.int64)
    return out


def read_device(dev, ptr, shape, dtype):
    """Host copy of device memory at `ptr` (a ring slot, which may live on another GPU)."""
    out = np.empty(shape, dtype)
    dev.check(dev.lib.lcgs_b200_peer_read(dev.ctx, ptr, out.ctypes.data, out.nbytes))
    return out


def write_outputs(out_dir, arrays):
    """out_dir/<name>.npy for each captured array: float32 for float32 and uint8 data, float64 for integers (checked
    exact).  If the set exceeds DUMP_BUDGET_BYTES, the arrays that do not fit an equal share of what is left keep the
    elements at sorted, seeded random flat indices -- the same indices for the same array size on every run.
    out_dir/manifest.json records each array's source shape and dtype and how it was sampled."""
    os.makedirs(out_dir, exist_ok=True)
    host = {}
    for name, (a, dt) in arrays.items():
        host[name] = (a if isinstance(a, np.ndarray) else a.cpu().numpy()).view(dt)
    size_of = lambda a: 4 if a.dtype in (np.float32, np.uint8) else 8  # noqa: E731  stored bytes per element
    budget = DUMP_BUDGET_BYTES - 2**20                                    # headroom for the .npy headers and the manifest
    left = len(host)
    manifest = {}
    for name, a in sorted(host.items(), key=lambda kv: (kv[1].size * size_of(kv[1]), kv[0])):
        share = budget // left
        entry = {"shape": list(a.shape), "dtype": str(a.dtype), "sample": None}
        if a.size * size_of(a) > share:
            k = share // size_of(a)
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(a.size, k, replace=False))
            a = a.reshape(-1)[idx]
            entry["sample"] = {"count": int(k), "seed": DUMP_SEED,
                               "indices": "np.sort(np.random.default_rng(seed).choice(size, count, replace=False)) into the C-order flattened array"}
        if size_of(a) == 4:
            out = a.astype(np.float32)
        else:
            out = a.astype(np.float64)
            if not np.array_equal(out.astype(a.dtype), a):
                raise ValueError("%s: integer values beyond float64's exact range" % name)
        budget -= out.nbytes
        left -= 1
        entry["stored"] = str(out.dtype)
        manifest[name] = entry
        np.save(os.path.join(out_dir, name + ".npy"), out)
    with open(os.path.join(out_dir, "manifest.json"), "w") as fh:
        json.dump(manifest, fh, indent=1, sort_keys=True)


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------

class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
            atexit.register(self.p.kill)   # a run that fails before stop() must not leave the sampler behind
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.f.read().splitlines():
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), samples=len(sm), reasons=sorted(reasons))
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------

# preprocess, scan+compact (+depth histograms), depth sort (4 u32 passes, the last one returns at once), key emission
# (+chained offsets, tile histograms), tile sort (2 u64 passes), ranges, tile order, blend
KERNELS_PER_FRAME = 12


class Bench:
    def __init__(self, args):
        import torch
        import torch.distributed as dist

        from luisacomputegaussiansplatting_b200 import lcgs, scenes

        self.torch, self.dist, self.lcgs, self.scenes = torch, dist, lcgs, scenes
        self.args = args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            torch.cuda.set_device(self.local)
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        if args.gpus != self.world and self.rank == 0:
            sys.stderr.write("warning: --gpus %d but WORLD_SIZE %d; using WORLD_SIZE\n" % (args.gpus, self.world))
        args.gpus = self.world
        resolve_workload(args, self.world)
        self.dev = lcgs.Device(self.local)
        self.launches = 0
        self.outputs = None   # --dump-outputs: capture of the last timed step (rank 0)

    # -- helpers ------------------------------------------------------------------------------
    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def load_scene(self, key):
        t0 = time.perf_counter()
        sc, cfg = self.scenes.make_config_scene(key, P=self.args.gaussians)
        return sc, cfg, time.perf_counter() - t0

    def make_renderer(self, sc, cfg, capacity, tile_rows=(0, -1), rgb8=True):
        t0 = time.perf_counter()
        r = self.lcgs.Renderer(self.dev, sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity, cfg.W, cfg.H, list_capacity=capacity,
                               keep_intermediates=True, rgb8=rgb8, prepare_scene=True, tile_rows=tile_rows)
        self.torch.cuda.synchronize()
        return r, time.perf_counter() - t0

    def stage_profile(self, r, vps, reps):
        """Per-stage CUDA-event times (ms) averaged over `reps` frames + the tile sort's launch breakdown."""
        dev = self.dev
        dev.set_profiling(True)
        acc, sort_acc = {}, {"histogram_ms": 0.0, "passes_ms": 0.0, "num_passes": 0}
        for i in range(reps):
            r.render_async(vps[i % len(vps)])
            st = dev.stage_times()
            sb = dev.sort_breakdown()
            for k, v in st.items():
                acc[k] = acc.get(k, 0.0) + v / reps
            sort_acc["histogram_ms"] += sb["histogram_ms"] / reps
            sort_acc["passes_ms"] += sb["passes_ms"] / reps
            sort_acc["num_passes"] = sb["num_passes"]
        dev.set_profiling(False)
        return acc, sort_acc

    def stage_table(self, r, stage_ms, N, passes, peak):
        """Algorithmic bytes of the data flow that runs (M = Gaussians touching a tile): the Gaussians are depth-sorted
        first (8-byte pairs, three 9-bit passes; a fourth only for depths beyond 13107), so the 12-byte instance pairs
        need `passes` tile-bit passes.  The reference's flow (SURVEY.md 8d) would move N*(8+24*ceil((32+log2 T)/8))."""
        P, W, H, T = r.P, r.W, r.H, r.num_tiles
        V = int((r.depth >= 0.2).sum().item())
        M = int((r.tiles_touched > 0).sum().item())
        # preprocess / ranges / blend: SURVEY.md 8d's formulas; scan, depth sort, emission, tile sort: the bytes of the flow that runs
        alg = {"preprocess": 48.0 * P + 228.0 * V, "scan": 8.0 * P + 12.0 * M, "depth_sort": 16.0 * M * 3,
               "duplicate_keys": 20.0 * M + 12.0 * N, "sort": 24.0 * N * passes, "ranges": 8.0 * N + 16.0 * T,
               "blend": 40.0 * N + 12.0 * W * H}
        tab = {k: {"ms": round(v, 4), "alg_GB": round(alg[k] / 1e9, 4), "GBps": round(alg[k] / (v * 1e-3) / 1e9, 1),
                   "frac_of_hbm_peak": round(alg[k] / (v * 1e-3) / 1e9 / peak, 3)} for k, v in stage_ms.items() if v > 0}
        if "blend" in tab:
            tab["blend"]["bound"] = "fp32 issue + shared memory (not HBM): see roofline"
        return tab, V, M

    # -- N = 1, fixed pose (C1 / C2 / C3 / C5 unsharded): the headline ---------------------------
    def run_single(self):
        torch, lcgs, scenes, args, dev = self.torch, self.lcgs, self.scenes, self.args, self.dev
        sc, cfg, gen_s = self.load_scene(scene_key(args.config))
        P, W, H = sc.num_gaussians, cfg.W, cfg.H
        r, upload_s = self.make_renderer(sc, cfg, args.capacity)
        pose = (scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world))
        vp = lcgs.view_params(lcgs.make_camera(*pose, W, H))
        warm = max(args.warmup, 3)

        for _ in range(warm):
            r.render_async(vp)
        n_rendered = dev.num_rendered()
        clocks = ClockSampler(self.local)
        clocks.start()
        time.sleep(0.3)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(args.steps):
            r.render_async(vp)
        ev1.record()
        torch.cuda.synchronize()
        ms_total = float(ev0.elapsed_time(ev1))
        self.launches += KERNELS_PER_FRAME * args.steps
        if args.dump_outputs:
            self.outputs = capture_frame(r, dev.num_rendered())

        stage_ms, sort_acc = self.stage_profile(r, [vp], max(3, min(args.steps, 10)))
        clock_info = clocks.stop()

        # ---- end to end through the public API ------------------------------------------------
        # Streaming use: frame i+1 is enqueued while frame i's uint8 image travels to pinned host memory on a copy
        # stream (two device images, two host buffers); the host consumes frame i-1 before it enqueues frame i+1.
        def e2e_loop(use_rgb8):
            main_stream, copy_stream = torch.cuda.current_stream(), torch.cuda.Stream()
            if use_rgb8:
                dev_bufs = [r.rgb8, torch.empty_like(r.rgb8)]
                host_bufs = [torch.empty(3 * W * H, dtype=torch.uint8).pin_memory() for _ in range(2)]
            else:
                dev_bufs = [r.img, torch.empty_like(r.img)]
                host_bufs = [torch.empty(3 * W * H, dtype=torch.float32).pin_memory() for _ in range(2)]
            host_counts = torch.zeros(args.steps, dtype=torch.int32).pin_memory()
            ev_render = [torch.cuda.Event() for _ in range(2)]
            ev_copy = [torch.cuda.Event() for _ in range(2)]
            checksum = 0.0
            t0 = 0.0
            for i in range(-warm, args.steps):                  # `warm` untimed iterations of the very same loop first
                if i == 0:
                    for e in ev_copy:
                        e.synchronize()
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                b = i & 1
                if i >= 2 - warm:
                    main_stream.wait_event(ev_copy[b])          # device buffer b has been read out
                cam = lcgs.make_camera(*pose, W, H)             # host-side camera -> kernel parameters
                if use_rgb8:
                    r.set_target_rgb8(dev_bufs[b])
                else:
                    r.set_target(dev_bufs[b])
                r.render_async(lcgs.view_params(cam))
                r.read_num_rendered_async(host_counts[max(i, 0):max(i, 0) + 1])
                ev_render[b].record(main_stream)
                copy_stream.wait_event(ev_render[b])
                (r.read_image_rgb8 if use_rgb8 else r.read_image)(host_bufs[b], stream=copy_stream)
                ev_copy[b].record(copy_stream)
                if i >= 1 - warm and i != 0:
                    ev_copy[b ^ 1].synchronize()                # frame i-1 is on the host: consume it
                    checksum += float(host_bufs[b ^ 1][12345])
            ev_copy[(args.steps - 1) & 1].synchronize()
            torch.cuda.synchronize()
            checksum += float(host_bufs[(args.steps - 1) & 1][12345])
            dt = time.perf_counter() - t0
            assert int(host_counts.min()) == int(host_counts.max()) == n_rendered, (host_counts.tolist(), n_rendered)
            if use_rgb8:
                r.set_target_rgb8(dev_bufs[0])
            else:
                r.set_target(dev_bufs[0])
            return dt
        e2e_s = e2e_loop(True)
        e2e_f32_s = e2e_loop(False)
        self.launches += 2 * KERNELS_PER_FRAME * (args.steps + warm)

        # ---- variant: re-upload the whole Gaussian set from pinned host memory every frame ------------
        pinned = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in (sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity)]
        dsts = [r.pos, r.scale, r.rotq, r.sh, r.opacity]
        host_rgb = torch.empty(3 * W * H, dtype=torch.uint8).pin_memory()
        k = max(2, min(args.steps, 5))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(k):
            for d, s in zip(dsts, pinned):
                d.view(-1).copy_(s.view(-1), non_blocking=True)
            r.scene_changed()
            r.render_async(vp)
            r.read_image_rgb8(host_rgb)
            dev.num_rendered()
        e2e_cold = {"value": P * k / (time.perf_counter() - t0), "unit": UNIT,
                    "h2d_bytes_per_step": int(sum(p.numel() * 4 for p in pinned)), "d2h_bytes_per_step": 3 * W * H + 8, "steps": k,
                    "note": "scene re-uploaded from pinned memory and lcgs_b200_scene_prepare re-run every frame"}
        del pinned
        self.launches += (KERNELS_PER_FRAME + 1) * k

        # ---- assemble -------------------------------------------------------------------------------
        peak, peak_src = peaks()
        N = n_rendered
        passes = sort_acc["num_passes"]
        stages, V, M = self.stage_table(r, stage_ms, N, passes, peak)
        pass_ms = sort_acc["passes_ms"] / max(passes, 1)
        sort_achieved = 24.0 * N / (pass_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": P * args.steps / (ms_total * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, cfg, P, 1)[0], "parallelism": "single GPU",
            "frame_buffers": "all 12 of app/main.cpp:232-254 written every frame (means_2d, conic, color included) + the uint8 image",
            "scene_constants": "alpha-test constants (threshold, log2 opacity) computed once per scene by lcgs_b200_scene_prepare, "
                               "like the activations the loader applies once (app/gaussians.cpp:15-35)",
            "frames_per_second": args.steps / (ms_total * 1e-3),
            "num_rendered": N, "visible": V, "touching": M,
            "e2e": {"value": P * args.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": 164,
                    "d2h_bytes_per_step": 3 * W * H + 4, "ms_per_step": e2e_s / args.steps * 1e3,
                    "note": "camera parameters in from host memory; the app's uint8 HWC image (blend-kernel epilogue, app/main.cpp:"
                            "322-337) + num_rendered out to pinned host memory and read by the host every frame (D2H of frame i "
                            "overlaps the render of frame i+1, <= 2 frames in flight); Gaussian set uploaded once (%.0f ms) as in "
                            "app/main.cpp:216-226" % (upload_s * 1e3)},
            "e2e_float_image": {"value": P * args.steps / e2e_f32_s, "unit": UNIT, "d2h_bytes_per_step": 12 * W * H + 4,
                                "ms_per_step": e2e_f32_s / args.steps * 1e3,
                                "note": "same loop reading back the planar float32 image the reference reads (app/main.cpp:313-315)"},
            "e2e_with_scene_upload": e2e_cold,
            "stages": stages, "sort_breakdown": sort_acc,
            "roofline_sort": {"kernel": "onesweep_pass_kernel<u64> (dominant HBM kernel)", "bound": "hbm", "achieved": sort_achieved,
                              "peak": peak, "unit": "GB/s", "frac": sort_achieved / peak, "peak_source": peak_src,
                              "alg_bytes_per_launch": 24.0 * N, "launch_ms": pass_ms, "launches_per_step": passes,
                              "traffic": self.committed("onesweep_pass_kernel_dram_bytes_per_launch")},
            "clocks": clock_info,
        }
        blend_ms = stage_ms.get("blend", 0.0)

        if not args.no_cpu_baseline:
            # the full C3 frame costs the oracle about a second: 1 warm-up + 3 timed frames
            times, ostages, on, stats, cores = oracle_frames(sc, cfg, [pose] * 4, 1, max(args.capacity, 40_000_000))
            line["cpu_baseline"] = {"value": P * len(times) / float(np.sum(times)), "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": "3 whole frames of the same scene/camera (all %d Gaussians), oracle stage ms %s" % (
                                        P, json.dumps({k: round(v, 1) for k, v in ostages.items()})),
                                    "ms_per_frame": float(np.mean(times)) * 1e3, "num_rendered": on}
            assert on == N, (on, N)
            line["roofline"] = self.blend_roofline(stats, blend_ms, N, W, H, clock_info, peak)
        else:
            line["roofline"] = self.blend_roofline(None, blend_ms, N, W, H, clock_info, peak)

        if not args.no_orbit and args.config == "C3" and args.gaussians is None:
            del r
            torch.cuda.empty_cache()
            line["orbit_n1"] = self.run_views(as_leg=True)
        line["gpu_launches"] = self.launches
        return line

    def committed(self, key):
        """A counter summarised from the committed ncu --set full capture (profiles/roofline_traffic.json), or None."""
        p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        try:
            return json.load(open(p)).get(key)
        except Exception:
            return None

    def blend_roofline(self, stats, blend_ms, N, W, H, clock_info, hbm_peak):
        """SURVEY.md 8d for the blend: E examined (pixel, entry) pairs of the reference's loop (oracle-exact), 12 FP32 ops for
        an examined-but-rejected pair, 22 for a contributing one, against #SM * 128 lanes * 2 * clock."""
        sm = 148
        mhz = (clock_info or {}).get("sm_mhz") or 1965.0
        peak_tf = sm * FP32_LANES_PER_SM * 2 * mhz * 1e6 / 1e12
        out = {"kernel": "blend2_kernel (time-dominant kernel of the frame)", "bound": "fp32",
               "unit": "TFLOP/s", "peak": peak_tf,
               "peak_source": "derived: %d SMs x %d FP32 lanes x 2 x %.0f MHz (median SM clock sampled during the run); "
                              "MEASURED_PEAKS.json has no FP32 figure" % (sm, FP32_LANES_PER_SM, mhz),
               "launch_ms": blend_ms,
               "hbm": {"alg_bytes_per_launch": 40.0 * N + 12.0 * W * H,
                       "achieved_GBps": (40.0 * N + 12.0 * W * H) / (blend_ms * 1e-3) / 1e9 if blend_ms else None,
                       "frac_of_hbm_peak": (40.0 * N + 12.0 * W * H) / (blend_ms * 1e-3) / 1e9 / hbm_peak if blend_ms else None},
               "ncu": self.committed("blend_kernel"), "traffic": self.committed("blend_kernel_dram_bytes_per_launch")}
        if stats and blend_ms:
            E, Ec = stats["E"], stats["E_contrib"]
            flops = 12.0 * (E - Ec) + 22.0 * Ec
            out.update({"E_examined_pairs": E, "E_alpha_pass": stats["E_alpha"], "E_contrib": Ec, "upper_bound_256N": 256 * N,
                        "pairs_per_second": E / (blend_ms * 1e-3), "alg_flops_per_launch": flops,
                        "achieved": flops / (blend_ms * 1e-3) / 1e12, "frac": flops / (blend_ms * 1e-3) / 1e12 / peak_tf,
                        "note": "reference-equivalent work: the kernel culls (Gaussian, tile) and (Gaussian, 8x8 patch) pairs "
                                "conservatively, so it executes far fewer pair evaluations than E; the fraction says how fast the "
                                "reference's E pairs are retired, not how busy the FP32 pipes are (ncu: issue-active)"})
        else:
            out.update({"achieved": None, "frac": None})
        return out

    # -- view sharding (C4 orbit; also the orbit_n1 leg of the headline line) ------------------------
    def run_views(self, as_leg=False):
        torch, dist, lcgs, scenes, args, dev = self.torch, self.dist, self.lcgs, self.scenes, self.args, self.dev
        from luisacomputegaussiansplatting_b200 import distributed as D

        world, rank = self.world, self.rank
        sc, cfg, gen_s = self.load_scene("C2")
        P, W, H = sc.num_gaussians, cfg.W, cfg.H
        capacity = 30_000_000 if as_leg else args.capacity
        r, upload_s = self.make_renderer(sc, cfg, capacity)
        steps, warm = args.steps, max(args.warmup, 3)
        total = steps * world                       # frames of the timed run; the run spans the whole orbit
        SLOTS = 2                                   # ring slots per rank

        def vp_of(f):
            return lcgs.view_params(lcgs.make_camera(*scenes.orbit_pose(orbit_view(f, total)), W, H))

        fl = args.deliver == "float"
        if world > 1:
            ring = D.PeerFrameRing(dev, W, H, slots=SLOTS * world, rgb8=True, float_image=fl)
        else:
            ring = _LocalRing(torch, dev, W, H, SLOTS, rgb8=True, float_image=fl)
        render_stream = torch.cuda.current_stream()
        consume_stream = torch.cuda.Stream()
        # what rank 0 checksums: the delivered payload (32-bit words; the slot's padding behind a uint8 image stays zero)
        n_words = 3 * W * H if fl else (3 * W * H + 3) // 4
        payload = (lambda sl: ring.ptr(sl)) if fl else (lambda sl: ring.rgb8_ptr(sl))
        local_img = r.img.data_ptr()
        sums = torch.zeros(warm + steps + 8, world, dtype=torch.int64, device="cuda") if rank == 0 else None

        gstep = [0]   # global step counter: sequence numbers continue across warm-up and timed region

        def enqueue_step(s_local, host_out=None, evs=None):
            g = gstep[0]
            gstep[0] += 1
            slot_row, seq = g % SLOTS, g // SLOTS + 1
            slot = slot_row * world + rank
            if g >= SLOTS:
                ring.wait_consumed(slot, seq - 1, stream=render_stream)
            r.set_target_ptr(ring.ptr(slot) if fl else local_img, ring.rgb8_ptr(slot))
            r.render_async(vp_of(s_local * world + rank), stream=render_stream)
            ring.signal_ready(slot, seq, stream=render_stream)
            self.launches += KERNELS_PER_FRAME + (2 if g >= SLOTS else 1)
            if rank == 0:                           # consume the step's N frames in view order
                for w in range(world):
                    sl = slot_row * world + w
                    ring.wait_ready(sl, seq, stream=consume_stream)
                    if host_out is None:
                        dev.checksum_u32(payload(sl), n_words, sums[g, w:w + 1], stream=consume_stream)
                    else:                           # end-to-end: the delivered uint8 image goes to the host
                        k = s_local * world + w
                        dev.check(dev.lib.lcgs_b200_peer_read_async(dev.ctx, ring.rgb8_ptr(sl), host_out[k % len(host_out)].data_ptr(),
                                                                    3 * W * H, consume_stream.cuda_stream or None))
                        evs[k].record(consume_stream)
                    ring.signal_consumed(sl, seq, stream=consume_stream)
                    self.launches += 3
            return g

        for s in range(warm):
            enqueue_step(s)
        self.barrier()
        n_rendered = dev.num_rendered()
        clocks = ClockSampler(self.local) if (rank == 0 and not as_leg) else None
        if clocks:
            clocks.start()
            time.sleep(0.3)
        ev0, ev1, evc = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        self.barrier()
        ev0.record(render_stream)
        first_g = gstep[0]
        for s in range(steps):
            enqueue_step(s)
        ev1.record(render_stream)
        evc.record(consume_stream)
        self.barrier()
        if args.dump_outputs and rank == 0 and not as_leg:
            # rank 0's own last view (its float image stays local unless delivered) and every view of the last step as delivered
            self.outputs = capture_frame(r, dev.num_rendered(), img=not fl, rgb8=False)
            for w in range(world):
                sl, f = ((gstep[0] - 1) % SLOTS) * world + w, (steps - 1) * world + w
                self.outputs["rgb8_frame%d" % f] = (read_device(dev, ring.rgb8_ptr(sl), (H, W, 3), np.uint8), np.uint8)
                if fl:
                    self.outputs["img_frame%d" % f] = (read_device(dev, ring.ptr(sl), (3, H, W), np.float32), np.float32)
        ms = float(ev0.elapsed_time(ev1))
        per_rank_render_ms = self.gather_counts(ms / steps)
        consumer_ms = float(ev0.elapsed_time(evc)) / steps if rank == 0 else None
        if rank == 0:
            ms = max(ms, float(ev0.elapsed_time(evc)))
        ms_total = self.max_over_ranks(ms)
        timeouts = self.max_over_ranks(float(dev.peer_timeouts()))

        # delivered frames are the frames: rank 0 re-renders three of them locally and compares the checksums
        verified = None
        if rank == 0:
            local = torch.zeros(3 * W * H, dtype=torch.float32, device="cuda")
            local8 = torch.zeros(4 * n_words + 256, dtype=torch.uint8, device="cuda")
            one = torch.zeros(1, dtype=torch.int64, device="cuda")
            r.set_target_ptr(local.data_ptr(), local8.data_ptr())
            verified = True
            for (s, w) in {(0, 0), (steps // 2, world - 1), (steps - 1, world // 2)}:
                r.render_async(vp_of(s * world + w))
                dev.checksum_u32((local if fl else local8).data_ptr(), n_words, one)
                torch.cuda.synchronize()
                verified &= bool(int(one.item()) == int(sums[first_g + s, w].item()))
            self.launches += 3 * (KERNELS_PER_FRAME + 1)
        r.set_target_ptr(r.img.data_ptr(), r.rgb8.data_ptr())

        stage_ms, sort_acc = self.stage_profile(r, [vp_of(f * world + rank) for f in range(min(steps, 8))], max(3, min(steps, 8)))
        clock_info = clocks.stop() if clocks else None

        # ---- end to end: rank 0 reads every delivered frame's uint8 image into pinned host memory -----------
        host_out, evs = None, None
        if rank == 0:
            host_out = [torch.empty(3 * W * H, dtype=torch.uint8).pin_memory() for _ in range(min(total, 64))]
            evs = [torch.cuda.Event() for _ in range(total)]
        self.barrier()
        t0 = time.perf_counter()
        checksum = 0
        consumed = 0
        for s in range(steps):
            enqueue_step(s, host_out if rank == 0 else None, evs)
            if rank == 0:
                # the host consumes frames as they arrive, at most 48 behind the enqueue (the pool holds 64)
                while consumed < (s + 1) * world - 48:
                    evs[consumed].synchronize()
                    checksum += int(host_out[consumed % len(host_out)][4321])
                    consumed += 1
        if rank == 0:
            while consumed < total:
                evs[consumed].synchronize()
                checksum += int(host_out[consumed % len(host_out)][4321])
                consumed += 1
        torch.cuda.synchronize()
        e2e_s = self.max_over_ranks(time.perf_counter() - t0)
        timeouts = max(timeouts, self.max_over_ranks(float(dev.peer_timeouts())))
        self.barrier()
        ring.close()

        peak, peak_src = peaks()
        res = {
            "frames": total, "orbit_views": ORBIT_VIEWS, "ms_per_step": ms_total / steps,
            "frames_per_second": total / (ms_total * 1e-3), "value": P * total / (ms_total * 1e-3), "unit": UNIT,
            "e2e_value": P * total / e2e_s, "e2e_frames_per_second": total / e2e_s, "e2e_ms_per_step": e2e_s / steps * 1e3,
            "consumed_frames_verified": verified, "flow_control_timeouts": int(timeouts),
            "per_rank_render_stream_ms_per_step": [round(float(x), 4) for x in per_rank_render_ms],
            "rank0_consumer_stream_ms_per_step": consumer_ms,
            "delivered": "planar float32 + uint8 HWC image" if fl else "uint8 HWC image (the app's final product; the float image stays on the rendering rank)",
            "ring": "%d slots x %d ranks, %.1f MB per slot" % (SLOTS, world, ring.frame_bytes / 1e6),
            "num_rendered_last_view": n_rendered, "stages_rank0": {k: round(v, 4) for k, v in stage_ms.items()},
            "gen_s": round(gen_s, 1), "upload_s": round(upload_s, 2),
        }
        if as_leg:
            res["workload"] = "C4 on this GPU alone: same orbit, ring, flags and consumer as the N > 1 default of bench.py"
            del r
            torch.cuda.empty_cache()
            return res
        if rank != 0:
            return None
        N = n_rendered
        passes = sort_acc["num_passes"]
        stages, V, M = self.stage_table(r, stage_ms, N, passes, peak)
        pass_ms = sort_acc["passes_ms"] / max(passes, 1)
        sort_achieved = 24.0 * N / (pass_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warm,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args, cfg, P, world)[0],
            "parallelism": workload_config(args, cfg, P, world)[1], "views_per_step": world, "frames": total,
            "frames_per_second": res["frames_per_second"],
            "e2e": {"value": res["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": 164 * world, "d2h_bytes_per_step": (3 * W * H) * world,
                    "ms_per_step": res["e2e_ms_per_step"], "frames_per_second": res["e2e_frames_per_second"],
                    "note": "camera parameters in from host memory on every rank; every frame of every rank is delivered to rank 0's "
                            "ring (peer stores + device flags) and its uint8 image is copied from there to pinned host memory and read "
                            "by rank 0's host thread inside the timed region"},
            "view_sharding": res, "stages": stages, "sort_breakdown": sort_acc,
            "roofline": self.blend_roofline(None, stage_ms.get("blend", 0.0), N, W, H, clock_info, peak),
            "roofline_sort": {"kernel": "onesweep_pass_kernel<u64>", "bound": "hbm", "achieved": sort_achieved, "peak": peak,
                              "unit": "GB/s", "frac": sort_achieved / peak, "peak_source": peak_src, "launch_ms": pass_ms},
            "clocks": clock_info, "gpu_launches": self.launches,
        }
        return line

    # -- tile-row sharding (C5) -------------------------------------------------------------------------
    def run_rows(self):
        torch, dist, lcgs, scenes, args, dev = self.torch, self.dist, self.lcgs, self.scenes, self.args, self.dev
        from luisacomputegaussiansplatting_b200 import distributed as D

        world, rank = self.world, self.rank
        sc, cfg, gen_s = self.load_scene(scene_key(args.config))
        P, W, H = sc.num_gaussians, cfg.W, cfg.H
        gy = (H + 15) // 16
        pose = (scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world))
        vp = lcgs.view_params(lcgs.make_camera(*pose, W, H))
        bands = D.split_tile_rows(gy, world)
        r, upload_s = self.make_renderer(sc, cfg, args.capacity, tile_rows=bands[rank], rgb8=True)
        steps, warm = args.steps, max(args.warmup, 3)

        cam = lcgs.make_camera(*pose, W, H)

        def measure():
            """(instances, device ms per frame) of this rank's current band: 1 warm-up + 3 timed frames into the local image."""
            n = r.render(cam)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                r.render_async(vp)
            e1.record()
            torch.cuda.synchronize()
            self.launches += 4 * KERNELS_PER_FRAME
            return n, float(e0.elapsed_time(e1)) / 3.0

        # 1. uniform bands -> instances per tile row (SURVEY.md 8e) and a first set of (instances, rows, ms) samples
        n_uniform, t_uniform = measure()
        mine = torch.zeros(gy, dtype=torch.float64, device="cuda")
        w_rows = D.row_weights_from_ranges(r.ranges[: 2 * r.num_tiles], r.gx)
        mine[bands[rank][0]:bands[rank][1]] = torch.tensor(w_rows, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(mine)
        weights = mine.cpu().tolist()
        uniform_counts, uniform_ms = self.gather_counts(n_uniform), self.gather_counts(t_uniform)
        samples = [(n, b1 - b0, t) for n, (b0, b1), t in zip(uniform_counts, bands, uniform_ms)]
        tried = [("uniform rows", bands, uniform_counts, uniform_ms)]
        # 2. bands balanced by instance count
        bands = D.split_tile_rows(gy, world, weights)
        r.set_tile_rows(*bands[rank])
        n_i, t_i = measure()
        counts_i, ms_i = self.gather_counts(n_i), self.gather_counts(t_i)
        samples += [(n, b1 - b0, t) for n, (b0, b1), t in zip(counts_i, bands, ms_i)]
        tried.append(("balanced by instances", bands, counts_i, ms_i))
        # 3. bands balanced by the measured cost model ms ~ a * instances + b * rows + c (two refinement rounds)
        cost_model = None
        if world > 2:
            for it in range(2):
                a, b = D.fit_band_cost(samples)
                cost_model = {"ms_per_million_instances": a * 1e6, "ms_per_tile_row": b, "samples": len(samples)}
                bands = D.split_tile_rows_by_cost(gy, world, weights, a, b)
                r.set_tile_rows(*bands[rank])
                n_c, t_c = measure()
                counts_c, ms_c = self.gather_counts(n_c), self.gather_counts(t_c)
                samples += [(n, b1 - b0, t) for n, (b0, b1), t in zip(counts_c, bands, ms_c)]
                tried.append(("balanced by fitted cost, round %d" % (it + 1), bands, counts_c, ms_c))
        # the split whose slowest band is fastest
        best = min(range(len(tried)), key=lambda k: max(tried[k][3]))
        split_name, bands, band_counts, band_ms = tried[best]
        r.set_tile_rows(*bands[rank])
        n_band = r.render(cam)
        assert n_band == int(band_counts[rank])

        SLOTS = 2
        fl = args.deliver == "float"
        if world > 1:
            ring = D.PeerFrameRing(dev, W, H, slots=SLOTS, rgb8=True, writers=world, float_image=fl)
        else:
            ring = _LocalRing(torch, dev, W, H, SLOTS, rgb8=True, float_image=fl)
        render_stream = torch.cuda.current_stream()
        consume_stream = torch.cuda.Stream()
        n_words = 3 * W * H if fl else (3 * W * H + 3) // 4
        payload = (lambda sl: ring.ptr(sl)) if fl else (lambda sl: ring.rgb8_ptr(sl))
        local_img = r.img.data_ptr()
        sums = torch.zeros(warm + 2 * steps + 8, dtype=torch.int64, device="cuda") if rank == 0 else None
        gstep = [0]

        def enqueue_step(host_out=None, ev=None):
            g = gstep[0]
            gstep[0] += 1
            slot, seq = g % SLOTS, g // SLOTS + 1
            if g >= SLOTS:
                ring.wait_consumed(slot, seq - 1, stream=render_stream)
            r.set_target_ptr(ring.ptr(slot) if fl else local_img, ring.rgb8_ptr(slot))
            r.render_async(vp, stream=render_stream)
            ring.signal_ready(slot, seq, writer=rank, stream=render_stream)
            self.launches += KERNELS_PER_FRAME + (2 if g >= SLOTS else 1)
            if rank == 0:
                for w in range(world):
                    ring.wait_ready(slot, seq, writer=w, stream=consume_stream)
                if host_out is None:
                    dev.checksum_u32(payload(slot), n_words, sums[g:g + 1], stream=consume_stream)
                else:
                    dev.check(dev.lib.lcgs_b200_peer_read_async(dev.ctx, ring.rgb8_ptr(slot), host_out.data_ptr(), 3 * W * H,
                                                                consume_stream.cuda_stream or None))
                    ev.record(consume_stream)
                ring.signal_consumed(slot, seq, stream=consume_stream)
                self.launches += world + 2
            return g

        for _ in range(warm):
            enqueue_step()
        self.barrier()
        clocks = ClockSampler(self.local) if rank == 0 else None
        if clocks:
            clocks.start()
            time.sleep(0.3)
        ev0, ev1, evc = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        self.barrier()
        ev0.record(render_stream)
        first_g = gstep[0]
        for _ in range(steps):
            enqueue_step()
        ev1.record(render_stream)
        evc.record(consume_stream)
        self.barrier()
        if args.dump_outputs and rank == 0:
            # rank 0's band (its float image stays local unless delivered) and the assembled frame of the last step
            self.outputs = capture_frame(r, dev.num_rendered(), img=not fl, rgb8=False)
            sl = (gstep[0] - 1) % SLOTS
            self.outputs["rgb8_frame"] = (read_device(dev, ring.rgb8_ptr(sl), (H, W, 3), np.uint8), np.uint8)
            if fl:
                self.outputs["img_frame"] = (read_device(dev, ring.ptr(sl), (3, H, W), np.float32), np.float32)
        ms = float(ev0.elapsed_time(ev1))
        per_rank_ms = self.gather_counts(ms / steps)
        if rank == 0:
            ms = max(ms, float(ev0.elapsed_time(evc)))
        ms_total = self.max_over_ranks(ms)
        timeouts = self.max_over_ranks(float(dev.peer_timeouts()))

        r.set_target_ptr(r.img.data_ptr(), r.rgb8.data_ptr())
        stage_ms, sort_acc = self.stage_profile(r, [vp], max(3, min(steps, 5)))
        all_stage = [None] * world
        if world > 1:
            dist.all_gather_object(all_stage, {k: round(v, 4) for k, v in stage_ms.items()})
        else:
            all_stage = [{k: round(v, 4) for k, v in stage_ms.items()}]
        clock_info = clocks.stop() if clocks else None

        # ---- end to end: rank 0 copies the assembled uint8 frame to pinned host memory every step ------
        host_out = [torch.empty(3 * W * H, dtype=torch.uint8).pin_memory() for _ in range(2)] if rank == 0 else None
        evs = [torch.cuda.Event() for _ in range(steps)] if rank == 0 else None
        self.barrier()
        t0 = time.perf_counter()
        checksum = 0
        for s in range(steps):
            enqueue_step(host_out[s & 1] if rank == 0 else None, evs[s] if rank == 0 else None)
            if rank == 0 and s >= 1:
                evs[s - 1].synchronize()
                checksum += int(host_out[(s - 1) & 1][4321])
        if rank == 0:
            evs[steps - 1].synchronize()
            checksum += int(host_out[(steps - 1) & 1][4321])
        torch.cuda.synchronize()
        e2e_s = self.max_over_ranks(time.perf_counter() - t0)
        timeouts = max(timeouts, self.max_over_ranks(float(dev.peer_timeouts())))

        # the assembled frame is the single-GPU frame: rank 0 renders the whole frame alone and compares checksums
        verified = None
        if rank == 0:
            assembled = int(sums[first_g + steps - 1].item())
            if world > 1:
                del r
                torch.cuda.empty_cache()
                rf, _ = self.make_renderer(sc, cfg, 260_000_000 if args.config == "C5" else args.capacity, rgb8=True)
                full8 = torch.zeros(4 * n_words + 256, dtype=torch.uint8, device="cuda")
                rf.set_target_ptr(rf.img.data_ptr(), full8.data_ptr())
                n_full = rf.render(lcgs.make_camera(*pose, W, H))
                one = torch.zeros(1, dtype=torch.int64, device="cuda")
                dev.checksum_u32((rf.img if fl else full8).data_ptr(), n_words, one)
                torch.cuda.synchronize()
                verified = bool(int(one.item()) == assembled) and n_full == int(sum(band_counts))
                del rf
                self.launches += KERNELS_PER_FRAME + 1
            else:
                verified = True
        self.barrier()
        ring.close()
        if rank != 0:
            return None

        peak, peak_src = peaks()
        counts = [int(c) for c in band_counts]
        line = {
            "metric": METRIC, "value": P * steps / (ms_total * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warm,
            "ms_per_step": ms_total / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args, cfg, P, world)[0],
            "parallelism": workload_config(args, cfg, P, world)[1],
            "frames_per_second": steps / (ms_total * 1e-3),
            "e2e": {"value": P * steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": 164 * world, "d2h_bytes_per_step": 3 * W * H,
                    "ms_per_step": e2e_s / steps * 1e3,
                    "note": "camera in from host memory on every rank; every band is blended into rank 0's ring slot, whose uint8 image is "
                            "copied to pinned host memory and read by rank 0's host thread every frame"},
            "tile_row_sharding": {
                "split": split_name, "bands": bands, "instances_per_band": counts, "instances_total": int(sum(counts)),
                "band_imbalance_max_over_mean": max(counts) / (sum(counts) / len(counts)) if sum(counts) else None,
                "band_ms_standalone": [round(float(x), 4) for x in band_ms],
                "time_imbalance_max_over_mean": max(band_ms) / (sum(band_ms) / len(band_ms)),
                "cost_model": cost_model,
                "splits_tried": [{"split": nm, "rows": [b1 - b0 for b0, b1 in bd], "instances": [int(c) for c in cn],
                                  "ms": [round(float(x), 4) for x in tm], "max_ms": round(max(tm), 4)} for nm, bd, cn, tm in tried],
                "per_rank_ms_per_frame": [round(float(x), 4) for x in per_rank_ms], "per_rank_stage_ms": all_stage,
                "delivered": "planar float32 + uint8 HWC image" if fl else "uint8 HWC image (the float strips stay on the rendering ranks)",
                "assembled_frame_equals_single_gpu_frame": verified, "flow_control_timeouts": int(timeouts),
                "hbm_floor_ms_per_gpu": "SURVEY.md 8d: 1.13 ms at 8 TB/s for an 8-way split (preprocess replicated)"},
            "stages": {k: {"ms": v} for k, v in all_stage[0].items()}, "sort_breakdown": sort_acc,
            "roofline": self.blend_roofline(None, stage_ms.get("blend", 0.0), counts[0], W, H, clock_info, peak),
            "clocks": clock_info, "gpu_launches": self.launches, "gen_s": round(gen_s, 1), "upload_s": round(upload_s, 2),
        }
        return line

    def gather_counts(self, x):
        if self.world == 1:
            return [x]
        t = self.torch.zeros(self.world, dtype=self.torch.float64, device="cuda")
        t[self.rank] = float(x)
        self.dist.all_reduce(t)
        return t.cpu().tolist()

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


class _LocalRing:
    """The PeerFrameRing interface over plain local device memory (one GPU: nothing to map), so that the N = 1 number of
    a sharded workload runs the very same ring / flag / consumer code path."""

    def __init__(self, torch, dev, W, H, slots, rgb8=True, writers=1, float_image=True):
        self.dev, self.W, self.H, self.slots, self.writers = dev, W, H, slots, writers
        self.img_bytes = 3 * W * H * 4 if float_image else 0
        self.rgb8_bytes = ((3 * W * H + 255) // 256) * 256 if rgb8 else 0
        self.frame_bytes = ((self.img_bytes + self.rgb8_bytes + 255) // 256) * 256
        self.flags_offset = self.frame_bytes * slots
        self.mem = torch.zeros(self.flags_offset + 4 * slots * (writers + 1) + 256, dtype=torch.uint8, device="cuda")
        self.base = self.mem.data_ptr()

    def ptr(self, slot):
        return self.base + slot * self.frame_bytes

    def rgb8_ptr(self, slot):
        return self.ptr(slot) + self.img_bytes

    def signal_ready(self, slot, seq, writer=0, stream=None):
        self.dev.peer_signal(self.base + self.flags_offset + 4 * (slot * self.writers + writer), seq, stream)

    def wait_ready(self, slot, seq, writer=0, stream=None, timeout_ms=5000):
        self.dev.peer_wait(self.base + self.flags_offset + 4 * (slot * self.writers + writer), seq, timeout_ms, stream)

    def signal_consumed(self, slot, seq, stream=None):
        self.dev.peer_signal(self.base + self.flags_offset + 4 * (self.slots * self.writers + slot), seq, stream)

    def wait_consumed(self, slot, seq, stream=None, timeout_ms=5000):
        self.dev.peer_wait(self.base + self.flags_offset + 4 * (self.slots * self.writers + slot), seq, timeout_ms, stream)

    def close(self):
        self.mem = None


def run_b200(args):
    b = Bench(args)
    try:
        if args.shard == "rows":
            line = b.run_rows()
        elif args.config == "C4":
            line = b.run_views()
        elif b.world > 1:
            raise SystemExit("C1 / C2 / C3 are single-GPU workloads: use --config C4 (view sharding) or --config C5 --shard rows")
        else:
            line = b.run_single()
        if b.rank == 0 and line is not None:
            print(json.dumps(line), flush=True)
        if b.outputs is not None:
            write_outputs(args.dump_outputs, b.outputs)
    finally:
        b.close()
    return 0


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
