#!/usr/bin/env python
"""The device export of the result tables (ekp_results_device / PostProcessor.result_tensors) on one GPU, in one run.

1. Device time of one export.  Workloads (NCHW maps on the device, the reference front-end):
     video    64 x 46x54 scenes of synthetic.make_batch(64, 46, 54, (1, 6)) at max_humans 32 and 128;
     crowd    16 crowded 92x164 scenes of synthetic.make_batch(16, 92, 164, (30, 40)) at max_humans 64 and 128;
   each with and without the subset table.  After one run, --iters exports into the same out= tensors are queued behind
   a device sleep that covers their submission, and CUDA events around them give the device time per export (launch
   gaps included, host submission excluded).  torch.profiler gives the kernel's own time in a separate pass.
2. Pipelined images/s: 8 contexts on 8 streams take 64 x 46x54 batches (device inputs, the lean reference front-end) in
   turn, as bench.py's configs legs do.  Three loops, alternated within the run, --batches batches each:
     runs       the runs only;
     device     the runs plus result_tensors(out=ring[i % 8]) on every batch (on the batch's stream);
     host       the runs plus human_tables() of batch i - 8 (the e2e leg's read pattern: the host waits for it).
   images/s = images / wall time of the loop, from a synchronised device to a synchronised device.
The device loop's last 8 exported tables must equal the host loop's last 8 host tables, and every export of part 1 the
host readers' tables; the script exits non-zero otherwise.  The card's name and power limit are read in the same run.

    python tools/time_device_results.py [--out DIR] [--iters 400] [--batches 3000] [--rounds 5]
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

EXPORTS = {
    "video_64x46x54": dict(n=64, h=46, w=54, people=(1, 6), max_peaks=1024, max_humans=(32, 128)),
    "crowd_16x92x164": dict(n=16, h=92, w=164, people=(30, 40), max_peaks=4096, max_humans=(64, 128)),
}
N_CTX = 8


def card(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,power.max_limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, pl, pmax, sm = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": pl, "power_max_limit": pmax, "sm_max_clock": sm}
    except Exception as e:   # the numbers are still reported, with the reason the card could not be read
        return {"query_error": repr(e)}


def host_view(t):
    """The device tables as the host readers lay them out: (num_humans, parts structured, scores, overflow)."""
    from torch_ekpose_b200.paf_to_pose import _PEAK_DT
    return (t["num_humans"].cpu().numpy(), t["parts"].cpu().numpy().view(_PEAK_DT)[..., 0], t["scores"].cpu().numpy(),
            t["overflow"].cpu().numpy().view(np.uint32))


def same_tables(a, b):
    return all(x.shape == y.shape and x.tobytes() == y.tobytes() for x, y in zip(a, b))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "time_device_results"), help="directory of the JSON record")
    ap.add_argument("--iters", type=int, default=400, help="timed exports per configuration (>= 200)")
    ap.add_argument("--batches", type=int, default=3000, help="batches per pipelined loop and round")
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_device_results.py: no CUDA device (there is nothing to measure on the CPU)")
    import torch_ekpose_b200 as ek
    from torch_ekpose_b200 import synthetic

    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)
    failures = []

    # ---- 1. one export -----------------------------------------------------------------------------------------------
    def kernel_us(fn, calls):
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize(dev)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(calls):
                fn()
            torch.cuda.synchronize(dev)
        out = {}
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            if "results_export" in ev.key and t > 0:
                out[ev.key.split("(")[0]] = t / calls
        return out

    exports = {}
    for name, wl in EXPORTS.items():
        heat, paf = synthetic.make_batch(wl["n"], wl["h"], wl["w"], wl["people"], seed=7)
        heat, paf = torch.from_numpy(heat).to(dev), torch.from_numpy(paf).to(dev)
        for mh in wl["max_humans"]:
            pp = ek.PostProcessor(device=0, max_batch=wl["n"], max_h=wl["h"], max_w=wl["w"], max_peaks=wl["max_peaks"],
                                  max_humans=mh, max_part=512, max_cand=4096)
            pp.run(heat, paf)
            res, tabs = pp.results(), pp.human_tables()
            people = res["num_humans"]
            for subset in (False, True):
                out = pp.result_tensors(subset=subset)
                call = lambda: pp.result_tensors(subset=subset, out=out)    # noqa: E731
                for _ in range(5):
                    call()
                torch.cuda.synchronize(dev)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda._sleep(int(2e8))                   # ~0.1 s: the exports below are all queued before it ends
                e0.record(stream)
                for _ in range(args.iters):
                    call()
                e1.record(stream)
                torch.cuda.synchronize(dev)
                us = e0.elapsed_time(e1) * 1e3 / args.iters
                kern = kernel_us(call, 50)
                got = host_view(out)
                if not same_tables(got, (tabs[0], tabs[1], tabs[2], res["overflow"])) or \
                        (subset and out["subset"].cpu().numpy().tobytes() != res["subset"].tobytes()):
                    failures.append(f"{name} max_humans {mh} subset {subset}: the export differs from the host tables")
                rows = wl["n"] * mh * ((20 if subset else 0) + 18 * 4 + 1)
                written = 4 * (rows + 3 * wl["n"])
                exports[f"{name}_mh{mh}{'_subset' if subset else ''}"] = {
                    "workload": f"synthetic.make_batch({wl['n']}, {wl['h']}, {wl['w']}, {wl['people']}, seed=7), reference "
                                f"front-end, max_humans {mh}, subset {subset}",
                    "people_per_image": {"min": int(people.min()), "max": int(people.max()), "mean": float(people.mean())},
                    "export_us": us, "export_kernel_profiled_us": kern, "bytes_written": written,
                    "written_gbs": written / (us * 1e-6) / 1e9}
            pp.close()

    # ---- 2. pipelined images/s ---------------------------------------------------------------------------------------
    n, h, w = 64, 46, 54
    inputs = []
    for s in range(4):
        hh, pf = synthetic.make_batch(n, h, w, (1, 6), seed=7 + s)
        inputs.append((torch.from_numpy(hh).to(dev), torch.from_numpy(pf).to(dev)))
    pps = [ek.PostProcessor(device=0, max_batch=n, max_h=h, max_w=w, max_peaks=1024, max_humans=128) for _ in range(N_CTX)]
    streams = [torch.cuda.Stream(dev) for _ in range(N_CTX)]

    def submit(i):
        k = i % N_CTX
        pps[k].run(*inputs[i % len(inputs)], layout="nchw", frontend="reference", stream=streams[k])
        return k

    for i in range(2 * N_CTX):
        submit(i)
    ring = [pps[k].result_tensors(stream=streams[k]) for k in range(N_CTX)]
    last_host = [None] * N_CTX

    def runs(batches):
        for i in range(batches):
            submit(i)

    def device(batches):
        for i in range(batches):
            k = submit(i)
            pps[k].result_tensors(out=ring[k], stream=streams[k])

    def host(batches):
        for i in range(batches):
            k = i % N_CTX
            if i >= N_CTX:
                pps[k].human_tables()                     # batch i - 8 (waits for it)
            submit(i)
        for i in range(max(batches - N_CTX, 0), batches):
            last_host[i % N_CTX] = pps[i % N_CTX].human_tables()

    loops = {"runs": runs, "device": device, "host": host}

    def timed(fn, batches):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        main = torch.cuda.current_stream(dev)
        for s_ in streams:
            s_.wait_stream(main)
        fn(batches)
        for s_ in streams:
            main.wait_stream(s_)
        torch.cuda.synchronize(dev)
        return n * batches / (time.perf_counter() - t0)

    for fn in loops.values():                              # warm-up of every loop
        timed(fn, 4 * N_CTX)
    rounds = {k: [] for k in loops}
    for _ in range(args.rounds):
        for k, fn in loops.items():
            rounds[k].append(timed(fn, args.batches))
    for k in range(N_CTX):
        num, parts, scores = last_host[k]
        if not same_tables(host_view(ring[k])[:3], (num, parts, scores)):
            failures.append(f"context {k}: the device loop's last export differs from the host loop's last tables")
    for p in pps:
        p.close()
    med = {k: float(np.median(v)) for k, v in rounds.items()}

    out = {
        "what": "ekp_results_device / PostProcessor.result_tensors: one export's device time, and pipelined images/s with "
                "the tables exported to the device vs read on the host (tools/time_device_results.py)",
        "card": card(0), "torch_device_name": torch.cuda.get_device_name(0),
        "exports": exports,
        "exports_how": f"one context; after one run, {args.iters} exports into the same out= tensors queued behind a "
                       "device sleep, CUDA events around them (per export: the kernel plus the launch gap); "
                       "export_kernel_profiled_us: the kernel alone (torch.profiler over 50 calls, a separate pass)",
        "pipelined": {
            "workload": f"synthetic.make_batch({n}, {h}, {w}, (1, 6)), 4 seeded input sets on the device, reference "
                        f"front-end, no materialisation, max_humans 128, {N_CTX} contexts on {N_CTX} streams",
            "images_per_s_rounds": rounds, "images_per_s_median": med,
            "device_over_runs": med["device"] / med["runs"], "host_over_runs": med["host"] / med["runs"],
            "how": f"{args.batches} batches per loop and round, {args.rounds} rounds alternating runs / device / host; "
                   "images over the wall time from a synchronised device to a synchronised device",
        },
        "checks": {"failures": failures, "ok": not failures},
        "timestamp": time.strftime("%Y-%m-%dT%H:%M:%S"),
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r5_device_results.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))
    if failures:
        print("\n".join(failures), file=sys.stderr)
        raise SystemExit(1)


if __name__ == "__main__":
    main()
