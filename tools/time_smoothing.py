#!/usr/bin/env python
"""Device time of the smoother (ekp_smooth_humans / Smoother.update) after the tracker update that gives it its ids, in
one run.

Workloads: the tracker's three of tools/time_tracking.py (reference front-end, max_humans 32 (128 for the crowd),
Tracker and Smoother defaults: max_tracks 256, max_age 30, fps 30, min_cutoff 1, beta 0.007, d_cutoff 1):
    chain_64x46x54     64 consecutive frames as ONE sequence (one block walks 64 frames), 8 clips of 1..8 people;
    cameras_64x46x54   64 sequences of one frame each (64 blocks), 1-8 people;
    crowd_16x92x164    16 consecutive crowded frames (35 people) as one sequence, max_humans 128.
Per workload: the smoother update's device time as CUDA events over --iters updates queued behind a device sleep (so the
host never starves the device), the kernel alone by torch.profiler (a separate pass), and the tracker update it follows
measured the same way.  Before timing, the smoothed keypoints of three consecutive updates are checked bit for bit
against the NumPy restatement of tests/test_smoothing.py on the host tables and the device ids; the script exits
non-zero when they differ.  The card's name and power limit are read in the same run.

    python tools/time_smoothing.py [--out DIR] [--iters 400]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from tools.time_device_results import card   # noqa: E402
from tools.time_tracking import video         # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "time_smoothing"), help="directory of the JSON record")
    ap.add_argument("--iters", type=int, default=400)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_smoothing.py: no CUDA device (there is nothing to measure on the CPU)")
    import torch_ekpose_b200 as ek
    from torch_ekpose_b200 import synthetic
    from tests.test_smoothing import Restatement

    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)
    failures = []

    def events_us(fn, iters):
        for _ in range(5):
            fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(int(2e8))
        e0.record(stream)
        for _ in range(iters):
            fn()
        e1.record(stream)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) * 1e3 / iters

    def kernel_us(fn, calls, key):
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize(dev)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(calls):
                fn()
            torch.cuda.synchronize(dev)
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            if key in ev.key and t > 0:
                return t / calls
        return None

    wls = {
        "chain_64x46x54": dict(maps=video(64, 46, 54, 8, list(range(1, 9)), 11), n_seq=1, max_humans=32, max_peaks=1024),
        "cameras_64x46x54": dict(maps=synthetic.make_batch(64, 46, 54, (1, 8), seed=5), n_seq=64, max_humans=32, max_peaks=1024),
        "crowd_16x92x164": dict(maps=video(16, 92, 164, 1, [35], 21), n_seq=1, max_humans=128, max_peaks=4096),
    }
    results = {}
    for name, wl in wls.items():
        heat, paf = (torch.from_numpy(a).to(dev) for a in wl["maps"])
        n, _, h, w = heat.shape
        pp = ek.PostProcessor(device=0, max_batch=n, max_h=h, max_w=w, max_peaks=wl["max_peaks"], max_humans=wl["max_humans"],
                              max_part=512, max_cand=4096)
        pp.run(heat, paf)
        num, hparts, _ = pp.human_tables()
        host = np.zeros((n, wl["max_humans"], 18, 4), np.int32)
        for f, k in enumerate(("x", "y", "score", "id")):
            host[..., f] = hparts[k].view(np.int32) if k == "score" else hparts[k]
        tabs = pp.result_tensors()
        tr = ek.Tracker(0, n_seq=wl["n_seq"])
        sm = ek.Smoother(0, n_seq=wl["n_seq"])
        R = Restatement(wl["n_seq"])
        for call in range(3):   # consecutive calls carry the tracks and the filters
            ids = tr.update(tabs)
            got = sm.update(tabs, ids).cpu().numpy()
            want = R.update(num, host, ids.cpu().numpy())
            if not np.array_equal(got.view(np.uint32), want.view(np.uint32)):
                failures.append(f"{name}: smoothed keypoints of call {call} differ from the restatement")
        ids = tr.update(tabs)
        xy = sm.update(tabs, ids)
        upd = lambda: sm.update(tabs, ids, out=xy)    # noqa: E731
        trk = lambda: tr.update(tabs, out=ids)        # noqa: E731
        results[name] = {
            "images": int(n), "n_seq": wl["n_seq"], "frames_per_sequence": int(n) // wl["n_seq"],
            "people_per_image": {"min": int(num.min()), "max": int(num.max()), "mean": float(num.mean())},
            "smooth_update_us_events": events_us(upd, args.iters),
            "smooth_kernel_us_profiled": kernel_us(upd, 50, "smooth_kernel"),
            "track_update_us_events": events_us(trk, max(50, args.iters // 4)),
        }
        print(name, json.dumps(results[name]), flush=True)
        pp.close()

    rec = {
        "card": card(0),
        "torch": torch.__version__,
        "device_name": torch.cuda.get_device_name(0),
        "workloads": results,
        "notes": ["smooth_update_us_events: CUDA events over --iters updates queued behind a device sleep (per update, gaps included)",
                  "smooth_kernel_us_profiled: smooth_kernel alone, torch.profiler over 50 updates (a separate pass)",
                  "track_update_us_events: the tracker update the smoother follows (its ids), measured like the smoother",
                  "keypoints of three consecutive updates checked bit for bit against tests/test_smoothing.py's restatement"],
        "failures": failures,
    }
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "r8_smoothing.json")
    with open(path, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({k: v["smooth_update_us_events"] for k, v in results.items()}), "->", path)
    if failures:
        raise SystemExit("time_smoothing.py: " + "; ".join(failures))


if __name__ == "__main__":
    main()
