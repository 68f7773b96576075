#!/usr/bin/env python
"""Device time of the tracker (ekp_track_humans / Tracker.update) next to the post-processing batch it follows, in one run.

Workloads (reference front-end, max_humans 32 (128 for the crowd), Tracker defaults: max_tracks 256, min_oks 0.5,
max_age 30).  Video frames are synthetic scenes sliding right by one stride-8 cell every two frames, so people persist:
    chain_64x46x54     64 consecutive frames as ONE sequence (the longest chain: one block walks 64 frames), 8 clips of
                       8 frames with 1..8 people;
    cameras_64x46x54   64 sequences of one frame each (64 blocks, one frame each), 1-8 people;
    crowd_16x92x164    16 consecutive crowded frames (35 people) as one sequence, max_humans 128.
Per workload: the update's device time as CUDA events over --iters updates queued behind a device sleep (so the host
never starves the device), the kernel alone by torch.profiler (a separate pass), and the post-processing batch's device
time measured the same way.  Before timing, the ids of every update of the first pass are checked against the NumPy
oracle of tests/test_tracking.py on the host tables; the script exits non-zero when they differ.
Pipelined images/s of chain_64x46x54 over 8 contexts on 8 streams: run + result_tensors(out=ring) per batch, with and
without a Tracker.update per batch (one tracker per stream), alternated over --rounds rounds.
The card's name and power limit are read in the same run.

    python tools/time_tracking.py [--out DIR] [--iters 400] [--batches 1000] [--rounds 5]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from tools.time_device_results import card   # noqa: E402


def video(n, h, w, clips, people, seed):
    """n frames NCHW: len(clips) clips, clip c holds people[c] people sliding one stride-8 cell every two frames"""
    from torch_ekpose_b200 import synthetic
    per = n // clips
    heats, pafs = [], []
    for c in range(clips):
        bh, bp = synthetic.make_scene(h, w + per, people[c], seed=seed + c, noise=False)
        for t in range(per):
            heats.append(np.roll(bh, t // 2, axis=1)[:, :w])
            pafs.append(np.roll(bp, t // 2, axis=1)[:, :w])
    return np.ascontiguousarray(np.stack(heats).transpose(0, 3, 1, 2)), np.ascontiguousarray(np.stack(pafs).transpose(0, 3, 1, 2))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "time_tracking"), help="directory of the JSON record")
    ap.add_argument("--iters", type=int, default=400)
    ap.add_argument("--batches", type=int, default=1000)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_tracking.py: no CUDA device (there is nothing to measure on the CPU)")
    import torch_ekpose_b200 as ek
    from torch_ekpose_b200 import synthetic
    from tests.test_tracking import Oracle

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
        o = Oracle(wl["n_seq"], 256, 0.5, 30, check_margin=False)
        for call in range(3):   # consecutive calls carry the tracks
            got = tr.update(tabs).cpu().numpy()
            if not np.array_equal(got, o.update(num, host)):
                failures.append(f"{name}: ids of call {call} differ from the oracle")
        ids = tr.update(tabs)
        upd = lambda: tr.update(tabs, out=ids)   # noqa: E731
        run = lambda: pp.run(heat, paf)          # noqa: E731
        results[name] = {
            "images": int(n), "n_seq": wl["n_seq"], "frames_per_sequence": int(n) // wl["n_seq"],
            "people_per_image": {"min": int(num.min()), "max": int(num.max()), "mean": float(num.mean())},
            "tracks_opened_in_3_calls": int(sum(q["next_id"] for q in o.seq)),
            "update_us_events": events_us(upd, args.iters),
            "update_kernel_us_profiled": kernel_us(upd, 50, "track_kernel"),
            "postprocess_batch_us_events": events_us(run, max(50, args.iters // 4)),
        }
        print(name, json.dumps(results[name]), flush=True)
        pp.close()

    # ---- pipelined images/s over 8 contexts on 8 streams ------------------------------------------------------------------
    heat, paf = (torch.from_numpy(a).to(dev) for a in wls["chain_64x46x54"]["maps"])
    N = 8
    pps = [ek.PostProcessor(device=0, max_batch=64, max_h=46, max_w=54, max_peaks=1024, max_humans=32) for _ in range(N)]
    for p in pps:
        p.set_host_copy(False)
    streams = [torch.cuda.Stream(dev) for _ in range(N)]
    trackers = [ek.Tracker(0) for _ in range(N)]
    for k in range(N):
        pps[k].run(heat, paf, stream=streams[k])
    ring = [pps[k].result_tensors(stream=streams[k]) for k in range(N)]
    idr = [trackers[k].update(ring[k], stream=streams[k]) for k in range(N)]

    def loop(track, batches):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for i in range(batches):
            k = i % N
            pps[k].run(heat, paf, stream=streams[k])
            pps[k].result_tensors(out=ring[k], stream=streams[k])
            if track:
                trackers[k].update(ring[k], stream=streams[k], out=idr[k])
        torch.cuda.synchronize(dev)
        return 64 * batches / (time.perf_counter() - t0)

    loop(False, 100)
    loop(True, 100)
    rates = {"run_export": [], "run_export_track": []}
    for _ in range(args.rounds):
        rates["run_export"].append(loop(False, args.batches))
        rates["run_export_track"].append(loop(True, args.batches))
    pipelined = {k: {"median_images_per_s": float(np.median(v)), "min": float(min(v)), "max": float(max(v))} for k, v in rates.items()}

    rec = {
        "card": card(0),
        "torch": torch.__version__,
        "device_name": torch.cuda.get_device_name(0),
        "workloads": results,
        "pipelined_chain_64x46x54_8ctx": pipelined,
        "notes": ["update_us_events: CUDA events over --iters updates queued behind a device sleep (per update, gaps included)",
                  "update_kernel_us_profiled: track_kernel alone, torch.profiler over 50 updates (a separate pass)",
                  "postprocess_batch_us_events: the batch the update follows (pp.run), measured like the update",
                  "ids checked against tests/test_tracking.py's oracle on the host tables before timing"],
        "failures": failures,
    }
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "r6_tracking.json")
    with open(path, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec["pipelined_chain_64x46x54_8ctx"]), "->", path)
    if failures:
        raise SystemExit("time_tracking.py: " + "; ".join(failures))


if __name__ == "__main__":
    main()
