#!/usr/bin/env python
"""The device draw_humans (ekp_draw_humans) against the host path users have today, on one GPU, in one run.

Workloads (NCHW maps already on the device, the reference front-end as infer_humans runs it, random-content frames):
  video    64 frames of 480x640 drawn with the people of synthetic.make_batch(64, 46, 54, (1, 6)) scenes;
  crowd    16 frames of 736x1312 drawn with the people of crowded synthetic.make_batch(16, 92, 164, (30, 40)) scenes.

Per workload:
  draw_us          device time of one ekp_draw_humans call (cover + paint), CUDA events around --iters calls;
  post_us          device time of the post-processing batch the draw follows (PostProcessor.run, a graph replay);
  post_draw_us     the two back to back (run, then draw), per batch;
  draw_kernels_profiled_us   the two kernels of a draw separately (torch.profiler over 20 calls, after the timed legs);
  host             what a caller does today on the CPU: pp.humans() (wait, tables, Human objects) plus the reference's
                   draw_humans restated with cv2 (tests/draw_check.py) on every frame, one core (cv2.setNumThreads(1),
                   torch.set_num_threads(1)), mean over --host-iters batches.
Every drawn device frame is compared with the host path's frame; the script exits non-zero on any difference.  The
card's name and power limit are read in the same run.

    python tools/time_draw.py [--out DIR] [--iters 200] [--rounds 3] [--host-iters 3]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

WORKLOADS = {
    "video_64x480x640": dict(n=64, h=46, w=54, people=(1, 6), H=480, W=640, max_humans=64, max_peaks=1024),
    "crowd_16x736x1312": dict(n=16, h=92, w=164, people=(30, 40), H=736, W=1312, max_humans=128, max_peaks=4096),
}


def card(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,power.max_limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, pl, pmax, sm = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": pl, "power_max_limit": pmax, "sm_max_clock": sm}
    except Exception as e:   # the numbers are still reported, with the reason the card could not be read
        return {"query_error": repr(e)}


def kernel_times(torch, fn, calls):
    """Mean device time per call of every kernel ``fn`` launches (torch.profiler, CUDA activity)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if "draw" in ev.key and t > 0:
            out[ev.key.split("(")[0]] = t / calls
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "time_draw"), help="directory of the JSON record")
    ap.add_argument("--iters", type=int, default=200, help="timed device batches per leg and round")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--host-iters", type=int, default=3, help="timed host batches per workload")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_draw.py: no CUDA device (there is nothing to measure on the CPU)")
    import cv2
    import torch_ekpose_b200 as ek
    from tests import draw_check
    from torch_ekpose_b200 import synthetic

    cv2.setNumThreads(1)
    torch.set_num_threads(1)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)
    failures, results = [], {}

    def timed(fn, iters):
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(iters):
            fn()
        e1.record(stream)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) * 1e3 / iters

    for name, wl in WORKLOADS.items():
        heat, paf = synthetic.make_batch(wl["n"], wl["h"], wl["w"], wl["people"], seed=7)
        heat, paf = torch.from_numpy(heat).to(dev), torch.from_numpy(paf).to(dev)
        pp = ek.PostProcessor(device=0, max_batch=wl["n"], max_h=wl["h"], max_w=wl["w"], max_peaks=wl["max_peaks"],
                              max_humans=wl["max_humans"], max_part=512, max_cand=4096)
        host = np.random.default_rng(1).integers(0, 256, (wl["n"], wl["H"], wl["W"], 3), dtype=np.uint8)
        frames = torch.from_numpy(host).to(dev)
        pp.run(heat, paf)
        pp.run(heat, paf)
        people = [len(h) for h in pp.humans()]
        pp.draw_humans(frames)
        want = draw_check.draw_batch(host, pp.humans())
        if not np.array_equal(frames.cpu().numpy(), want):
            failures.append(f"{name}: the device frames differ from the host path's")

        run = lambda: pp.run(heat, paf)             # noqa: E731
        draw = lambda: pp.draw_humans(frames)       # noqa: E731

        def both():
            run()
            draw()

        for fn in (run, draw, both):                 # warm-up of every leg
            timed(fn, 5)
        legs = {"post_us": run, "draw_us": draw, "post_draw_us": both}
        ent = {k: [] for k in legs}
        for _ in range(args.rounds):
            for k, fn in legs.items():
                ent[k].append(timed(fn, args.iters))
        keys = torch.empty(wl["n"] * wl["H"] * wl["W"], dtype=torch.int32, device=dev)
        memset_us = timed(keys.zero_, args.iters)   # what clearing the keys on every call would add instead
        del keys
        kernels = kernel_times(torch, draw, 20)     # torch.profiler, after the timed legs
        launches0 = pp.kernel_launches()
        draw()
        draw_launches = pp.kernel_launches() - launches0

        # the host path: humans() + restated draw_humans on every frame, one core
        host_t, humans_t = [], []
        for _ in range(args.host_iters):
            pp.run(heat, paf)
            torch.cuda.synchronize(dev)
            img = host.copy()
            t0 = time.perf_counter()
            humans = pp.humans()
            t1 = time.perf_counter()
            for i, hs in enumerate(humans):
                draw_check.draw_humans(img[i], hs)
            t2 = time.perf_counter()
            humans_t.append((t1 - t0) * 1e6)
            host_t.append((t2 - t0) * 1e6)
            if not np.array_equal(img, want):
                failures.append(f"{name}: the host path is not deterministic")
        pp.close()
        med = {k: float(np.median(v)) for k, v in ent.items()}
        results[name] = {
            "workload": f"synthetic.make_batch({wl['n']}, {wl['h']}, {wl['w']}, {wl['people']}, seed=7) drawn onto "
                        f"{wl['n']} random frames of {wl['H']}x{wl['W']}",
            "people_per_frame": {"min": min(people), "max": max(people), "mean": float(np.mean(people))},
            "device_rounds_us": ent,
            "device_median_us": med,
            "draw_per_frame_us": med["draw_us"] / wl["n"],
            "draw_kernel_launches": draw_launches,
            "draw_kernels_profiled_us": kernels,
            "memset_keys_us": memset_us,
            "host_us_per_batch": {"humans": float(np.mean(humans_t)), "humans_plus_draw": float(np.mean(host_t)),
                                  "samples": host_t},
            "host_us_per_frame": float(np.mean(host_t)) / wl["n"],
            "host_over_device_draw": float(np.mean(host_t)) / med["draw_us"],
        }

    out = {
        "what": "ekp_draw_humans vs pp.humans() + cv2 draw_humans (tools/time_draw.py)",
        "card": card(0), "torch_device_name": torch.cuda.get_device_name(0),
        "how": f"device legs: one context, CUDA events around {args.iters} calls per leg, {args.rounds} rounds alternating "
               "post / draw / post+draw, the same frames drawn again every call; reference front-end, maps on the device. "
               "Host leg: one core, mean of the timed batches.",
        "keys": "per-call epoch in the high 16 bits of each key: no clearing pass between draws (memset_keys_us: what a "
                "cudaMemset of the n x H x W uint32 keys per call would cost instead)",
        "workloads": results,
        "checks": {"failures": failures, "ok": not failures},
        "timestamp": time.strftime("%Y-%m-%dT%H:%M:%S"),
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "time_draw.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))
    if failures:
        print("\n".join(failures), file=sys.stderr)
        raise SystemExit(1)


if __name__ == "__main__":
    main()
