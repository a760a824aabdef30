#!/usr/bin/env python
"""bench.py -- frames/s of the 3DGS forward hot path (project+SH -> bin -> sort -> blend) on B200.

Contract: `python bench.py --gpus N --steps K --warmup W [--impl reference]` prints ONE JSON line
(rank 0).  A "step" is one frame of the hot path.  Workload at N=1: BASELINE.json's headline config
(garden, 5.8 M Gaussians, 3200x1400) as a SYNTHETIC STAND-IN (the Inria .ply files are not
available offline): 5.8 M seeded Gaussians tuned to M/N ~ 5 (SURVEY 8d).

  value : frames/s with the camera UBO as a kernel argument and the framebuffer left in HBM
          (K frames enqueued back to back on one stream, CUDA events around them, max over ranks).
  e2e   : frames/s through the public C ABI call gsb_render() with HOST buffers: host UBO in,
          B8G8R8A8 framebuffer (the reference's swapchain format) copied device->host inside the
          timed region every step, synchronous per frame.
  N > 1 : the frame is sharded by tile rows over N GPUs (one process per GPU, scene replicated),
          each rank renders its band, one NCCL all-gather reassembles the framebuffer
          (strong scaling: total work fixed).
  --impl reference : the reference has no CPU path and its Vulkan build is unavailable here, so
          the reference arm times the CPU oracle (oracle/, "port") on the box's host cores on a
          bounded sample (a band of tile rows of the same frame) and extrapolates frames/s.
  --dump-outputs DIR : after the timed frames, writes the framebuffer the last timed frame produced
          to DIR/frame_bgra8.npy as float32 (H, W, 4), so that two builds run with the same arguments
          can be compared output for output.  A frame larger than DUMP_BUDGET_BYTES is written as a
          fixed, seeded sample of whole pixels: frame_bgra8.npy (K, 4) and their row-major pixel
          indices in frame_pixel_index.npy (K,) float64.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT / "3dgs.cpp_b200" / "python"))

WORKLOADS = {
    # name: N, W, H, seed, synth params, camera (pos, fov)
    "garden-standin": dict(n=5_800_000, w=3200, h=1400, seed=3, half=(10.0, 4.0, 10.0), ls=(0.003, 0.05),
                           cam=(0.0, 0.0, 14.0), fov=45.0,
                           note="synthetic stand-in for Mip-NeRF360 garden (5.8M Gaussians, 3200x1400), M/N~5"),
    "bicycle-standin": dict(n=6_100_000, w=1920, h=1080, seed=4, half=(10.0, 5.6, 10.0), ls=(0.003, 0.05),
                            cam=(0.0, 0.0, 14.0), fov=45.0, note="synthetic stand-in for bicycle (6.1M, 1920x1080)"),
    "truck-standin": dict(n=2_500_000, w=3840, h=2160, seed=5, half=(10.0, 5.6, 10.0), ls=(0.003, 0.05),
                          cam=(0.0, 0.0, 14.0), fov=45.0, note="synthetic stand-in for truck (2.5M, 3840x2160)"),
    "synthetic-50m": dict(n=50_000_000, w=7680, h=4320, seed=43, half=(10.0, 5.6, 10.0), ls=(0.002, 0.03),
                          cam=(0.0, 0.0, 14.0), fov=45.0, note="BASELINE config 5: synthetic 50M, 7680x4320"),
    "c1": dict(n=10_000, w=640, h=480, seed=42, half=(3.0, 3.0, 3.0), ls=(0.01, 0.15), cam=(0.0, 0.0, 5.0), fov=45.0,
               note="BASELINE config 1: synthetic 10k, 640x480"),
}
NUM_CAMERAS = 8  # small orbit so consecutive frames differ (M varies a few %)
DUMP_BUDGET_BYTES = 60_000_000  # --dump-outputs writes at most this much (plus .npy headers)
DUMP_SEED = 0


def make_scene(g, wl, first=0, count=None):
    """Gaussians [first, first + count) of the workload as GSScene::Vertex rows.  `g` is the product binding (gs_b200:
    C++ host generator + GSScene::load activations) or, for the reference arm, the oracle binding (the same generator
    and activations restated in oracle/gs_oracle.c, bit-identical: tests/test_oracle.py) -- so that the reference arm
    never loads a product library."""
    p = g.synth_params(center=(0, 0, 0), half_extent=wl["half"], log_scale_min=math.log(wl["ls"][0]),
                       log_scale_max=math.log(wl["ls"][1]))
    n = wl["n"] - first if count is None else count
    activate = g.activate_records if hasattr(g, "activate_records") else g.load_records
    vtx = np.empty((n, 60), np.float32)
    chunk = 1 << 20
    for off in range(0, n, chunk):  # PLY-format records -> GSScene::load activations
        cnt = min(chunk, n - off)
        vtx[off:off + cnt] = activate(g.synth_records(wl["seed"], cnt, p, first=first + off))
    return vtx


def camera_poses(wl):
    """(pos, quat wxyz, fov, near, far, W, H) of the NUM_CAMERAS poses: a +-6 degree orbit around the scene centre."""
    poses = []
    for k in range(NUM_CAMERAS):
        a = math.radians(-6.0 + 12.0 * k / max(1, NUM_CAMERAS - 1))
        d = wl["cam"][2]
        pos = (d * math.sin(a), wl["cam"][1], d * math.cos(a))
        quat = (math.cos(a / 2), 0.0, math.sin(a / 2), 0.0)  # yaw so the camera keeps looking at the origin
        poses.append((pos, quat, wl["fov"], 0.1, 1000.0, wl["w"], wl["h"]))
    return poses


def cameras(g, wl):
    return [g.uniforms_from_camera(*c) for c in camera_poses(wl)]


def bench_config(wl_name, wl):
    """The keys both arms share (the driver compares the two lines' config)."""
    return {"workload": wl_name, "note": wl["note"], "n_gaussians": wl["n"], "width": wl["w"], "height": wl["h"],
            "cameras": NUM_CAMERAS}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower() == "active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def measured_peak_gbs():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def dump_frame(out_dir, frame):
    """Writes an (H, W, 4) uint8 framebuffer as float32 .npy files in out_dir (see --dump-outputs in the docstring)."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    px = frame.reshape(-1, frame.shape[-1])
    if px.size * 4 <= DUMP_BUDGET_BYTES:
        np.save(out_dir / "frame_bgra8.npy", frame.astype(np.float32))
        return
    k = DUMP_BUDGET_BYTES // (px.shape[1] * 4 + 8)  # float32 channels + one float64 index per pixel
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(px.shape[0], size=k, replace=False))
    np.save(out_dir / "frame_bgra8.npy", px[idx].astype(np.float32))
    np.save(out_dir / "frame_pixel_index.npy", idx.astype(np.float64))


def use_all_cores(o):
    """torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU baseline should use every core this process may run on."""
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    o.set_num_threads(cores)
    return o.num_threads()


def cpu_oracle_frame(o, vtx, cov, u):
    """One WHOLE frame of the CPU oracle (all stages, all tile rows), wall-clocked."""
    t0 = time.perf_counter()
    f = o.render_frame(vtx, cov, u, light=True)  # light: no numpy copies of the intermediates inside the timed region
    wall = time.perf_counter() - t0
    return {"fps": 1.0 / wall, "t_frame_s": wall, "sample_wall_s": wall, "rows": (0, f["tiles_y"]), "tiles_y": f["tiles_y"],
            "cores": o.num_threads(), "m_band": int(f["m"]), "stages_s": f["t_stage"], "extrapolated": False}


def cpu_oracle_sample(wl, vtx, u, budget_s, cov=None):
    """Times the CPU oracle on a bounded sample: all N Gaussians preprocessed, but only a centred band
    of tile rows sorted + blended; frames/s is extrapolated by rows_total / rows_band for the
    band-proportional stages."""
    sys.path.insert(0, str(ROOT / "oracle"))
    import oracle as o

    if cov is None:
        cov = o.cov3d(vtx)  # GSScene::precomputeCov3D is load-time work, not per frame
    tiles_y = (wl["h"] + 15) // 16
    rows = 1
    mid = tiles_y // 2
    t0 = time.perf_counter()
    f = o.render_frame(vtx, cov, u, rows=(mid, mid + 1), light=True)  # calibration
    t_cal = time.perf_counter() - t0
    t_pre = f["t_stage"]["preprocess"] + f["t_stage"]["prefix_sum"]
    t_row = max(1e-6, t_cal - t_pre)
    rows = int(max(1, min(tiles_y, (budget_s - t_pre) // t_row)))
    rb = max(0, mid - rows // 2)
    re = min(tiles_y, rb + rows)
    t0 = time.perf_counter()
    f = o.render_frame(vtx, cov, u, rows=(rb, re), light=True)
    wall = time.perf_counter() - t0
    st = f["t_stage"]
    full_pre = st["preprocess"] + st["prefix_sum"]
    banded = st["preprocess_sort"] + st["sort"] + st["tile_boundary"] + st["render"]
    t_frame = full_pre + banded * tiles_y / (re - rb)
    return {"fps": 1.0 / t_frame, "t_frame_s": t_frame, "sample_wall_s": wall, "rows": (rb, re), "tiles_y": tiles_y,
            "cores": o.num_threads(), "m_band": int(f["m"]), "stages_s": st, "extrapolated": (re - rb) < tiles_y}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)   # SURVEY 8d: 20 warm-up + 200 timed frames
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None)
    ap.add_argument("--mode", default="exact", choices=["exact", "fast"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sh16", action="store_true", help="gsb_set_sh_storage(1): fp16 SH coefficients -- NOT a parity mode, never the default")
    ap.add_argument("--no-extra", action="store_true", help="skip the C4 / C5 extra workload measured at --gpus 4 / 8")
    ap.add_argument("--tile-cull", type=int, default=2, help="gsb_set_tile_cull level: 0 reference lists, 1 exact per-tile instance culling, 2 coarse bins (image bit-identical in all three)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the framebuffer of the last timed frame to DIR/*.npy (float32; sampled above DUMP_BUDGET_BYTES)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200: the reference arm times frames that keep no image")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE {world}")
    wl_name = args.workload or "garden-standin"
    wl = WORKLOADS[wl_name]

    # ------------------------------------------------------------------ reference arm (CPU oracle)
    if args.impl == "reference":
        if rank != 0:
            return
        # Only oracle/ is loaded here (no product library): scene, cameras and the frame all come from liboracle.so.
        sys.path.insert(0, str(ROOT / "oracle"))
        import oracle as o
        cores = use_all_cores(o)
        vtx = make_scene(o, wl)
        cams = [o.uniforms_from_camera(*c) for c in camera_poses(wl)]
        cov = o.cov3d(vtx)  # GSScene::precomputeCov3D is load-time work, not per frame
        total = max(1, args.steps + args.warmup)
        # Whole frames when `total` of them fit ~150 s of CPU time (garden: ~2 s per frame on a 64-core box); otherwise
        # a band of tile rows per step with the band-proportional stages extrapolated, and the line says so.
        first = cpu_oracle_frame(o, vtx, cov, cams[0])
        whole = first["t_frame_s"] * total <= 150.0
        per_step = max(2.0, min(30.0, 150.0 / total))
        vals, walls = [], []
        for s in range(total):
            t0 = time.perf_counter()
            r = cpu_oracle_frame(o, vtx, cov, cams[s % NUM_CAMERAS]) if whole else cpu_oracle_sample(wl, vtx, cams[s % NUM_CAMERAS], per_step, cov)
            if s >= args.warmup:
                vals.append(r)
                walls.append(time.perf_counter() - t0)
        fps = float(np.mean([r["fps"] for r in vals]))
        if whole:
            sample = (f"per step: one WHOLE frame of the CPU oracle (all {wl['n']} Gaussians, all {vals[-1]['tiles_y']} tile rows, "
                      f"~{vals[-1]['sample_wall_s']:.2f}s wall); nothing extrapolated; preprocess/scan/emit/sort/ranges/blend all OpenMP")
        else:
            sample = (f"per step: all {wl['n']} Gaussians preprocessed, tile rows {vals[-1]['rows']} of {vals[-1]['tiles_y']} "
                      f"sorted+blended (~{vals[-1]['sample_wall_s']:.1f}s wall), frames/s EXTRAPOLATED by rows_total/rows_band")
        print(json.dumps({
            "impl": "reference", "metric": "frames/sec", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 / fps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "extrapolated": not whole,
            "wall_ms_per_step": 1000.0 * float(np.mean(walls)),
            "config": bench_config(wl_name, wl),
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "the reference (Vulkan/GLSL) has no CPU path and cannot be built offline; this is the CPU oracle port",
        }))
        return

    import gs_b200 as g  # raises if the CUDA library is not built: no fallback

    # ------------------------------------------------------------------ B200 arm
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    ctx = None
    if world > 1:
        # torch.distributed only carries the 128-byte group id and the timing reductions; the frame's exchange (survivor
        # routing + framebuffer) is the product's own: gsb_create_sharded / gsb_render_sharded (peer memory over NVLink)
        dist.init_process_group("nccl", device_id=dev)
        box = [g.shard_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        ctx = g.ShardedContext(local_rank, rank, world, box[0])
    else:
        ctx = g.Context(local_rank)
    ctx.set_mode(g.MODE_EXACT if args.mode == "exact" else g.MODE_FAST)
    ctx.set_tile_cull(int(args.tile_cull))
    if args.sh16:
        ctx.set_sh_storage(True)

    env = dict(g=g, torch=torch, dist=dist, dev=dev, rank=rank, world=world, local_rank=local_rank, ctx=ctx, args=args)
    out = measure(env, wl_name, wl, args.steps, max(3, args.warmup), headline=True)
    # BASELINE configs C4 / C5 are quoted on 4 / 8 GPUs: measured here as well and carried on the same JSON line (the headline
    # workload stays the one `value` is quoted on, so the driver's 1 -> 8 scaling curve is over ONE workload)
    extra_name = {4: "truck-standin", 8: "synthetic-50m"}.get(world) if not args.workload and not args.no_extra else None
    if extra_name:
        try:
            ex = measure(env, extra_name, WORKLOADS[extra_name], min(args.steps, 50), 5, headline=False)
            if rank == 0:
                out["extra_workloads"] = [ex]
        except Exception as exc:  # never lose the headline line over the extra workload
            if rank == 0:
                out["extra_workloads"] = [{"workload": extra_name, "error": repr(exc)}]
    if rank == 0:
        print(json.dumps(out))
        if args.dump_outputs:
            dump_frame(args.dump_outputs, env["last_frame"])
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


class _DevFrame:
    """A device pointer dressed as a __cuda_array_interface__ object so torch can copy from it."""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


def measure(env, wl_name, wl, steps, warmup, headline):
    """Uploads the workload and measures it on the context in `env` (single GPU: gsb_render*; N GPUs: gsb_render_sharded*).
    Returns the JSON dict (rank 0) or None."""
    g, torch, dist, dev, rank, world, ctx, args = (env[k] for k in ("g", "torch", "dist", "dev", "rank", "world", "ctx", "args"))
    sharded = world > 1
    W, H = wl["w"], wl["h"]
    tiles_y = (H + 15) // 16
    fmt, bpp = g.FORMAT_BGRA8, 4
    cams = cameras(g, wl)
    t_load = time.perf_counter()
    if sharded:
        first, count = g.shard_slice(wl["n"], rank, world)  # the scene is sharded by Gaussian index: every rank builds its slice
        vtx = make_scene(g, wl, first, count)
        ctx.upload_slice(vtx, wl["n"])
        del vtx
    else:
        vtx = make_scene(g, wl)
        ctx.upload(vtx)
    t_load = time.perf_counter() - t_load
    stream = torch.cuda.Stream(device=dev)  # a real (non-NULL) stream: NULL would mean the context's own stream
    torch.cuda.set_stream(stream)
    dev_fb = [torch.zeros((H, W, bpp), dtype=torch.uint8, device=dev) for _ in range(2)] if not sharded else None

    def frame(i, sync, k=0):
        u = cams[i % NUM_CAMERAS]
        if sharded:
            if sync:
                ctx.render_sharded_into(u, None, fmt, stream=stream)  # blocking, regrows collectively; frame stays in the window
            else:
                ctx.render_sharded_async(u, fmt, stream=stream)
        else:
            ctx.render_into(u, dev_fb[k].data_ptr(), fmt, stream=stream, sync=sync)

    def barrier():
        if sharded:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if sharded:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # first frames size the instance arena (regrow path), then keep headroom for the orbit
    ctx.set_timers(True)
    frame(0, sync=True)
    peak_m = 0
    for i in range(NUM_CAMERAS):
        frame(i, sync=True)
        peak_m = max(peak_m, ctx.stats().num_instances)
    ctx.reserve(int(peak_m * 1.3) + 65536)
    for i in range(warmup):
        frame(i, sync=True)

    # per-stage / per-kernel times (library cudaEvents), sampled on separate untimed frames
    stage_acc, m_acc, cons_acc, vis_acc, pass_acc, aabb_acc, visit_acc, staged_acc = {}, [], [], [], [], [], [], []
    passes = 0
    for i in range(NUM_CAMERAS):
        frame(i, sync=True)
        s = ctx.stats()
        d = s.as_dict()
        for k in ("preprocess_ms", "preprocess_sort_ms", "sort_ms", "sort_depth_ms", "sort_tile_ms", "tile_boundary_ms", "render_ms",
                  "frame_ms", "sort_hist_ms"):
            stage_acc.setdefault(k, []).append(d[k])
        stage_acc.setdefault("sort_pass_ms", []).append(float(np.mean(d["sort_pass_ms"])) if d["sort_pass_ms"] else 0.0)
        m_acc.append(s.num_instances)
        aabb_acc.append(s.num_instances_aabb)
        cons_acc.append(s.blend_consumed)
        visit_acc.append(s.blend_warp_visits)
        staged_acc.append(s.blend_staged)
        vis_acc.append(s.num_visible)
        passes = s.sort_passes
        pass_acc.append(d["sort_pass_ms"])
    lane_util = None
    if not sharded:  # blend_pixel_hits is counted on debug frames only
        ctx.set_debug(True)
        frame(0, sync=True)
        sd = ctx.stats()
        lane_util = sd.blend_pixel_hits / (64.0 * sd.blend_warp_visits) if sd.blend_warp_visits else None
        ctx.set_debug(False)
        frame(0, sync=True)
    stage = {k: float(np.mean(v)) for k, v in stage_acc.items()}
    pass_each = [float(x) for x in np.mean(np.array(pass_acc), axis=0)] if pass_acc and pass_acc[0] else []
    M, NV, CONS, VISITS = float(np.mean(m_acc)), float(np.mean(vis_acc)), float(np.mean(cons_acc)), float(np.mean(visit_acc))
    STAGED = float(np.mean(staged_acc))
    coarse = int(args.tile_cull) == 2

    # ---- value: K frames, device resident, one stream, CUDA events, max over ranks ----
    ctx.set_timers(False)  # from here on the camera-independent middle of the frame replays from a captured CUDA graph
    for i in range(NUM_CAMERAS):
        frame(i, sync=False)  # untimed: graph capture + instantiation happen here
    barrier()
    sampler = ClockSampler(env["local_rank"]) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(steps):
        frame(i, sync=False)
    e1.record(stream)
    barrier()
    ms_step = reduce_max(e0.elapsed_time(e1)) / steps
    ctx.stats()  # raises GSB_ERR_OVERFLOW if any async frame overflowed the arena (sticky flag)
    if headline and args.dump_outputs and rank == 0:  # the last timed frame, before later loops overwrite it
        src = torch.as_tensor(_DevFrame(ctx.frame_ptr(), (H, W, bpp)), device=dev) if sharded else dev_fb[0]
        env["last_frame"] = src.cpu().numpy()

    # ---- per-frame distribution (SURVEY 8d: median / p95): the same frames again with an event after every frame ----
    nd = min(steps, 200)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(nd + 1)]
    barrier()
    evs[0].record(stream)
    for i in range(nd):
        frame(i, sync=False)
        evs[i + 1].record(stream)
    barrier()
    per_frame_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(nd)]

    # ---- e2e: public C-ABI calls with HOST buffers: host UBO in every step, the whole BGRA8 frame in (rank 0's) pinned host
    # memory every step, all inside the timed region.
    #   sync     : one blocking call per frame: gsb_render(host UBO -> pinned host frame) -- the blend stores straight into the
    #              host frame (N = 1); gsb_render_sharded(... -> host) = frame + one D2H copy of rank 0's whole frame (N > 1)
    #   pipelined: enqueue-only render into one of two device frames + cudaMemcpyAsync of every frame to pinned host memory
    #              on a copy stream (events order buffer reuse); the copy overlaps the next frame's kernels
    host_fb = [torch.empty((H, W, bpp), dtype=torch.uint8).pin_memory() for _ in range(2)] if rank == 0 else None
    barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        u = cams[i % NUM_CAMERAS]
        if sharded:
            ctx.render_sharded_into(u, host_fb[0].data_ptr() if rank == 0 else None, fmt, mem=g.MEM_HOST, stream=stream)
        else:
            ctx._ck(g.lib.gsb_render(ctx.h, u, 0, g.ALL_ROWS, host_fb[0].data_ptr(), 0, g.MEM_HOST, fmt, None))
    torch.cuda.synchronize()
    e2e_sync_fps = steps / reduce_max(time.perf_counter() - t0)

    copy_stream = torch.cuda.Stream(device=dev)
    rendered = [torch.cuda.Event() for _ in range(2)]
    copied = [torch.cuda.Event() for _ in range(2)]
    barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        k = i & 1
        if i >= 2:
            stream.wait_event(copied[k])  # frame i - 2 has left the buffer frame i is about to overwrite
        frame(i, sync=False, k=k)
        rendered[k].record(stream)
        if rank == 0:
            src = torch.as_tensor(_DevFrame(ctx.frame_ptr(), (H, W, bpp)), device=dev) if sharded else dev_fb[k]
            copy_stream.wait_event(rendered[k])
            with torch.cuda.stream(copy_stream):
                host_fb[k].copy_(src, non_blocking=True)
        copied[k].record(copy_stream)
    torch.cuda.synchronize()
    e2e_fps = steps / reduce_max(time.perf_counter() - t0)
    ctx.stats()  # raises if an async frame overflowed the arena
    clocks = sampler.stop() if sampler else None

    per_rank = None
    if sharded:  # band imbalance: every rank's instance count and device frame time (library timers) for one pose
        ctx.set_timers(True)
        frame(0, sync=True)
        frame(0, sync=True)
        s = ctx.stats()
        mine = {"rank": rank, "visible": int(s.num_visible), "instances": int(s.num_instances), "frame_ms": float(s.frame_ms),
                "project_exchange_ms": float(s.preprocess_ms), "blend_ms": float(s.shard_blend_ms), "band_wait_ms": float(s.shard_wait_ms),
                "depth_sort_ms": float(s.sort_depth_ms), "emit_ms": float(s.preprocess_sort_ms), "tile_sort_ms": float(s.sort_tile_ms),
                "blend_consumed": int(s.blend_consumed), "blend_warp_visits": int(s.blend_warp_visits)}
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)
        ctx.set_timers(False)
    if rank != 0:
        return None

    peak, peak_src = measured_peak_gbs()
    nv = NV
    n_local = wl["n"] / world
    # algorithmic bytes per launch (SURVEY 8d / DESIGN.md), one launch = one frame's worth of that kernel ON THIS RANK
    T_tiles = ((W + 15) // 16) * tiles_y
    kd = "sort_depth(hist+4 onesweep passes over N_v)"
    alg = {
        "k_project": n_local * 40 + (nv * 192 + nv * (64 + 8)) * (1.0 if not sharded else 1.0),  # scene read + SH of survivors + 64-B record, depth key + payload
        kd: nv * (4 + 16 * 4 - 4),                                 # histogram read + 4 x (8 B read + 8 B written); the last pass writes no keys
        "k_emit": nv * (4 + 32) + 8 * M,                           # sorted ids + one 32-B record sector per survivor in, (tile / block id, payload) out
        "k_sort_hist": 4 * M,
        # per launch, averaged over the passes: 8 B read + 8 B written per (tile id, payload) pair; the last pass
        # writes payloads only (4 B) plus the tile ranges
        # with coarse bins the blend reads the sorted keys (tile masks), so the last pass writes them too
        "k_onesweep_pass": (16 * M * passes - (0 if coarse else 4 * M) + 8 * T_tiles) / max(passes, 1),
        # per tile: list entries scanned (coarse bins: 4-B key + 4-B payload each; otherwise the 4-B payload) + 36 B of record
        # for every entry staged + the tile's pixels
        "k_blend": (CONS * 8 + STAGED * 36 if coarse else CONS * (4 + 36)) + H * W * bpp / world * (world if sharded else 1),
    }
    dur = {"k_project": stage["preprocess_ms"], kd: stage["sort_depth_ms"], "k_emit": stage["preprocess_sort_ms"],
           "k_sort_hist": stage["sort_hist_ms"], "k_onesweep_pass": stage["sort_pass_ms"],
           "k_blend": stage["render_ms"]}
    share = dict(dur)
    share["k_onesweep_pass"] = stage["sort_pass_ms"] * passes
    kern = {k: {"ms_per_launch": dur[k], "launches_per_step": passes if k == "k_onesweep_pass" else (5 if k == kd else 1),
                "alg_bytes_per_launch": alg[k], "achieved_gbs": alg[k] / (dur[k] * 1e-3) / 1e9 if dur[k] > 0 else None,
                "share_of_step": share[k] / stage["frame_ms"] if stage["frame_ms"] > 0 else None} for k in alg}
    dom = max(share, key=share.get)
    traffic = None
    try:  # DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture (headline workload, N = 1)
        tj = json.loads((ROOT / "profiles" / "ncu_traffic.json").read_text())
        traffic = (tj["dram_bytes_per_launch"].get(dom) or tj["dram_bytes_per_launch"].get(dom + "2")) if (headline and not sharded) else None
    except Exception:
        pass
    roof = {"kernel": dom, "bound": "hbm", "achieved": kern[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
            "frac": kern[dom]["achieved_gbs"] / peak if kern[dom]["achieved_gbs"] else None, "traffic": traffic,
            "peak_source": peak_src,
            "note": "k_blend is FP32-issue bound, not HBM bound (SURVEY 8d): its HBM fraction is reported as required; "
                    "blend_warp_visits_per_s x the SASS instructions per visit (profiles/) is its issue-slot utilisation"}
    out = {
        "metric": "frames/sec", "value": 1000.0 / ms_step, "unit": "frames/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {**bench_config(wl_name, wl),
                   "instances_M": M, "instances_aabb": float(np.mean(aabb_acc)), "tile_cull": int(args.tile_cull), "visible": NV,
                   "sort_passes": passes, "blend_mode": args.mode, "sh_storage": "fp16 (NON-PARITY)" if args.sh16 else "fp32", "output": "BGRA8", "scene_load_s": t_load,
                   "l2": "inputs (scene + sort keys, > 1 GB) larger than the 126 MB L2; 8 camera poses alternate; no flush",
                   "parallelism": (f"scene sharded by Gaussian index x{world}, frame by tile-row bands x{world}; survivors and framebuffer "
                                   f"exchanged by stores into peer memory (NVLink), no collective in the frame" if sharded else "single GPU")},
        "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": 160, "d2h_bytes_per_step": int(H * W * bpp) + 64,
                "api": ("gsb_render_sharded_async(host UBO) on every rank + cudaMemcpyAsync of every whole BGRA8 frame from rank 0's copy to its pinned host memory, double buffered"
                        if sharded else "gsb_render_async(host UBO) + cudaMemcpyAsync of every BGRA8 frame to pinned host memory, double buffered"),
                "sync_value": e2e_sync_fps,
                "sync_api": ("gsb_render_sharded(host UBO -> rank 0's pinned host BGRA8 frame), one blocking collective call per frame" if sharded
                             else "gsb_render(host UBO -> pinned host BGRA8 frame: the blend stores straight into host memory), one blocking call per frame")},
        # k_frame_init, k_project, hist + 4 passes (depth), k_emit, hist + P passes (tile; the last one also writes the tile
        # ranges), k_blend -- the sorts and the emission are launched through one captured CUDA graph per frame; sharded
        # frames add k_shard_gather and 2 signal + 2 wait one-warp kernels (the survivor routing is inside k_project)
        "gpu_launches": int((10 + passes + (5 if sharded else 0)) * steps),
        "clocks": clocks,
        "roofline": roof,
        "kernels": kern,
        "stage_ms": stage,
        "sort_pass_ms_each": pass_each,
        # keys the instance sort actually moved (with coarse bins: (Gaussian, 4x4-tile block) entries) per second of both sorts;
        # and the reference's own instance count (AABB tiles, what its 8-pass sort would be given) over the same time
        "sort_keys_per_s": M / (stage["sort_ms"] * 1e-3) if stage["sort_ms"] > 0 else None,
        "reference_instances_per_sort_s": float(np.mean(aabb_acc)) / (stage["sort_ms"] * 1e-3) if stage["sort_ms"] > 0 else None,
        # evaluated work, not the algorithmic pair count: one visit = one (warp, record) iteration of the blend's inner loop = 64
        # pixel x Gaussian pairs evaluated (k_blend2: 2 pixels per lane)
        "blend_warp_visits_per_s": VISITS / (stage["render_ms"] * 1e-3) if stage["render_ms"] > 0 else None,
        "blend_pairs_evaluated_per_s": VISITS * 64 / (stage["render_ms"] * 1e-3) if stage["render_ms"] > 0 else None,
        # of the evaluated pairs, the fraction that passes render.comp:68-80 (the rest is SIMT lanes riding along)
        "blend_lane_utilisation": lane_util,
        "blend_records_consumed": CONS, "blend_records_staged": STAGED, "blend_warp_visits": VISITS,
    }
    if sharded:
        out["per_rank"] = per_rank
        out["stage_ms_note"] = "stage times, instance counts and rooflines are rank 0's (its band, its slice); per_rank has every rank's frame"
    try:  # SURVEY 8d: M for every timed camera, median / p95 of the per-camera frame time (library timers)
        fm = [float(x) for x in stage_acc.get("frame_ms", [])]
        out["per_camera"] = {"frame_ms": fm, "instances": [int(x) for x in m_acc],
                             "frame_ms_median": float(np.median(fm)) if fm else None,
                             "frame_ms_p95": float(np.percentile(fm, 95)) if fm else None}
        out["frame_ms_distribution"] = {"frames": len(per_frame_ms), "median": float(np.median(per_frame_ms)),
                                        "p95": float(np.percentile(per_frame_ms, 95)), "max": float(np.max(per_frame_ms)),
                                        "how": "cudaEvent after every frame of the device-resident loop (this rank)"}
    except Exception as exc:  # reporting only: never lose the bench line over it
        out["per_camera"] = {"error": str(exc)}
    if headline and world == 1 and not args.no_cpu_baseline:
        sys.path.insert(0, str(ROOT / "oracle"))
        import oracle as o
        cores = use_all_cores(o)
        cov = o.cov3d(vtx)
        r = cpu_oracle_frame(o, vtx, cov, cams[0])  # calibration / warm-up
        if r["t_frame_s"] <= 10.0:  # whole frames, nothing extrapolated (garden: ~2-3 s each)
            rs = [cpu_oracle_frame(o, vtx, cov, cams[k % NUM_CAMERAS]) for k in range(max(1, min(8, int(20.0 / r["t_frame_s"]))))]
            fps = float(np.mean([x["fps"] for x in rs]))
            sample = f"{len(rs)} WHOLE frames of the CPU oracle ({np.mean([x['t_frame_s'] for x in rs]):.2f} s each), nothing extrapolated"
        else:
            r = cpu_oracle_sample(wl, vtx, cams[0], 20.0, cov)
            fps = r["fps"]
            sample = (f"all {wl['n']} Gaussians preprocessed, tile rows {r['rows']} of {r['tiles_y']} sorted+blended "
                      f"({r['sample_wall_s']:.1f}s wall), EXTRAPOLATED by rows_total/rows_band")
        out["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample}
    return out


if __name__ == "__main__":
    main()
