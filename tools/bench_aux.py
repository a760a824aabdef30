"""Cost of the aux planes: gsb_render vs gsb_render_aux on bench.py's headline workload (garden stand-in, 5.8 M Gaussians,
3200x1400, BGRA8 into device memory), EXACT mode, gsb_set_tile_cull level 2.

Both calls are synchronous, so a frame is timed on the host around the call (it returns after the device finished).  The two
entry points alternate round by round (which one goes first alternates too) over `--rounds` rounds of `--frames` frames each,
with timers off (the captured middle graph replays, as in bench.py's timed loop); the cameras cycle through bench.py's
8-pose orbit.  The blend-stage times come from separate rounds with the library's cudaEvent timers on.  The GPU name and
power limit are read in the same run.  Prints one JSON object (and writes it to --out).

    python tools/bench_aux.py --out r3_aux.json
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "3dgs.cpp_b200" / "python"))
import bench  # noqa: E402  (workload table + scene / camera generators)


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=60)
        name, power = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as exc:  # the numbers below are still measured; say that the card could not be named
        return {"gpu": None, "power_limit": None, "nvidia_smi_error": str(exc)}


def stats_of(ms):
    a = np.asarray(ms, np.float64)
    return {"median_ms": float(np.median(a)), "p95_ms": float(np.percentile(a, 95)), "mean_ms": float(a.mean()), "frames": int(a.size)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workload", default="garden-standin", choices=list(bench.WORKLOADS))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--tile-cull", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    import gs_b200 as g

    info = gpu_info()
    wl = bench.WORKLOADS[args.workload]
    W, H = wl["w"], wl["h"]
    cams = bench.cameras(g, wl)
    ctx = g.Context(0)
    ctx.set_mode(g.MODE_EXACT)
    ctx.set_tile_cull(args.tile_cull)
    ctx.upload(bench.make_scene(g, wl))
    stream = torch.cuda.Stream()
    img = torch.zeros((H, W, 4), dtype=torch.uint8, device="cuda:0")
    img_aux = torch.zeros((H, W, 4), dtype=torch.uint8, device="cuda:0")
    aux = torch.zeros((H, W, 2), dtype=torch.float32, device="cuda:0")
    fmt = g.FORMAT_BGRA8

    def plain(i):
        ctx.render_into(cams[i % len(cams)], img.data_ptr(), fmt, stream=stream, sync=True)

    def with_aux(i):
        ctx.render_aux_into(cams[i % len(cams)], img_aux.data_ptr(), aux.data_ptr(), fmt, stream=stream)

    variants = {"render": plain, "render_aux": with_aux}
    # size the instance arena over the orbit (regrow path), then headroom as bench.py keeps it
    ctx.set_timers(True)
    peak = 0
    for i in range(len(cams)):
        plain(i)
        peak = max(peak, ctx.stats().num_instances)
    ctx.reserve(int(peak * 1.3) + 65536)

    # blend-stage (and frame) times from the library's timers, separate rounds
    stage = {k: {"render_ms": [], "frame_ms": []} for k in variants}
    for r in range(args.rounds):
        for name in (list(variants) if r % 2 == 0 else list(variants)[::-1]):
            for i in range(len(cams) * 4):
                variants[name](i)
                s = ctx.stats()
                stage[name]["render_ms"].append(s.render_ms)
                stage[name]["frame_ms"].append(s.frame_ms)

    # timed rounds: timers off = graph replay of the middle of the frame
    ctx.set_timers(False)
    for _ in range(args.warmup):
        for i in range(len(cams)):
            plain(i)
            with_aux(i)
    torch.cuda.synchronize()
    per_frame = {k: [] for k in variants}
    round_medians = {k: [] for k in variants}
    for r in range(args.rounds):
        for name in (list(variants) if r % 2 == 0 else list(variants)[::-1]):
            fn, ms = variants[name], []
            for i in range(args.frames):
                t0 = time.perf_counter()
                fn(i)
                ms.append((time.perf_counter() - t0) * 1e3)
            per_frame[name] += ms
            round_medians[name].append(float(np.median(ms)))

    # same camera, both entry points: the colour must not change
    plain(0)
    with_aux(0)
    torch.cuda.synchronize()
    colour_identical = bool(torch.equal(img, img_aux))
    a = aux.cpu().numpy()
    ctx.close()

    out = {
        "what": "gsb_render vs gsb_render_aux, device outputs (BGRA8 + float2 aux plane), synchronous calls timed on the host",
        "workload": args.workload, "width": W, "height": H, "gaussians": wl["n"], "mode": "EXACT", "tile_cull": args.tile_cull,
        "rounds": args.rounds, "frames_per_round": args.frames, "warmup_orbits": args.warmup, **info,
        "per_frame": {k: {**stats_of(v), "round_medians_ms": round_medians[k]} for k, v in per_frame.items()},
        "timers_on": {k: {"render_ms_median": float(np.median(v["render_ms"])), "render_ms_mean": float(np.mean(v["render_ms"])),
                          "frame_ms_median": float(np.median(v["frame_ms"])), "frames": len(v["render_ms"])}
                      for k, v in stage.items()},
        "colour_identical": colour_identical,
        "aux_check": {"opacity_max": float(a[..., 0].max()), "covered_fraction": float((a[..., 0] > 0).mean())},
    }
    pf, tm = out["per_frame"], out["timers_on"]
    out["aux_cost"] = {
        "frame_median_ms": pf["render_aux"]["median_ms"] - pf["render"]["median_ms"],
        "frame_median_rel": pf["render_aux"]["median_ms"] / pf["render"]["median_ms"] - 1.0,
        "blend_median_ms": tm["render_aux"]["render_ms_median"] - tm["render"]["render_ms_median"],
        "blend_median_rel": tm["render_aux"]["render_ms_median"] / tm["render"]["render_ms_median"] - 1.0,
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
