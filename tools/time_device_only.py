#!/usr/bin/env python
"""What the per-batch device-to-host copy of the result records costs in the pipelined loop: ekp_set_host_copy /
PostProcessor.set_host_copy on one GPU, in one run.

Workloads (NCHW maps on the device, nothing materialised), each on 8 contexts driven on 8 streams in turn, as bench.py's
configs legs drive them:
    64 x 46x54 scenes of synthetic.make_batch(64, 46, 54, (1, 6)), reference and dense front-ends, max_humans 32 and 128;
    16 crowded 92x164 scenes of synthetic.make_batch(16, 92, 164, (30, 40)), reference front-end, max_humans 128.
Four loops per workload, alternated within each round, --batches batches each:
    runs_copy        the runs only, host copy on (the default);
    runs_device      the runs only, host copy off;
    export_copy      the runs plus result_tensors(out=ring[k]) on every batch (on its stream), host copy on;
    export_device    the same, host copy off.
images/s = images / wall time of the loop, from a synchronised device to a synchronised device.  The spread over rounds
is reported next to each median.  d2h_bytes_per_batch is the copy the host-copy mode adds to every batch (ResultLayout
stride x batch).  The card's name and power limit are read in the same run.
After the last round (export_device), every context's last exported tables, and one more export with subset and peaks,
must equal the host readers' tables of the same run (which download the records of that device-only run); the script
exits non-zero otherwise.

    python tools/time_device_only.py [--out DIR] [--batches 2000] [--rounds 5]
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

WORKLOADS = {
    "video_64x46x54_reference_mh32": dict(n=64, h=46, w=54, people=(1, 6), frontend="reference", max_peaks=1024, max_humans=32),
    "video_64x46x54_reference_mh128": dict(n=64, h=46, w=54, people=(1, 6), frontend="reference", max_peaks=1024, max_humans=128),
    "video_64x46x54_dense_mh32": dict(n=64, h=46, w=54, people=(1, 6), frontend="dense", max_peaks=1024, max_humans=32),
    "video_64x46x54_dense_mh128": dict(n=64, h=46, w=54, people=(1, 6), frontend="dense", max_peaks=1024, max_humans=128),
    "crowd_16x92x164_reference_mh128": dict(n=16, h=92, w=164, people=(30, 40), frontend="reference", max_peaks=4096,
                                            max_humans=128, max_part=512, max_cand=4096),
}
N_CTX = 8
LOOPS = ("runs_copy", "runs_device", "export_copy", "export_device")


def record_stride(max_humans):
    """ResultLayout::stride (capi.cu ekp_create_ex): header, subset rows, part table, human scores, 16-byte aligned."""
    return (16 + 4 * 20 * max_humans + 16 * 18 * max_humans + 4 * max_humans + 15) & ~15


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "time_device_only"), help="directory of the JSON record")
    ap.add_argument("--batches", type=int, default=2000, help="batches per loop and round")
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_device_only.py: no CUDA device (there is nothing to measure on the CPU)")
    import torch_ekpose_b200 as ek
    from torch_ekpose_b200 import synthetic
    from torch_ekpose_b200.paf_to_pose import _PEAK_DT

    dev = torch.device("cuda", 0)
    failures = []
    results = {}

    def same(a, b):
        return a.shape == b.shape and np.ascontiguousarray(a).tobytes() == np.ascontiguousarray(b).tobytes()

    for name, wl in WORKLOADS.items():
        n, h, w = wl["n"], wl["h"], wl["w"]
        inputs = []
        for s in range(4):
            hh, pf = synthetic.make_batch(n, h, w, wl["people"], seed=7 + s)
            inputs.append((torch.from_numpy(hh).to(dev), torch.from_numpy(pf).to(dev)))
        pps = [ek.PostProcessor(device=0, max_batch=n, max_h=h, max_w=w, max_peaks=wl["max_peaks"], max_humans=wl["max_humans"],
                                max_part=wl.get("max_part", 0), max_cand=wl.get("max_cand", 0)) for _ in range(N_CTX)]
        streams = [torch.cuda.Stream(dev) for _ in range(N_CTX)]

        def submit(i):
            k = i % N_CTX
            pps[k].run(*inputs[i % len(inputs)], layout="nchw", frontend=wl["frontend"], stream=streams[k])
            return k

        for i in range(N_CTX):
            submit(i)
        ring = [pps[k].result_tensors(stream=streams[k]) for k in range(N_CTX)]

        def loop(copy, export):
            def fn(batches):
                for p in pps:
                    p.set_host_copy(copy)
                for i in range(batches):
                    k = submit(i)
                    if export:
                        pps[k].result_tensors(out=ring[k], stream=streams[k])
            return fn

        loops = {"runs_copy": loop(True, False), "runs_device": loop(False, False), "export_copy": loop(True, True),
                 "export_device": loop(False, True)}

        def timed(fn, batches):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            main_st = torch.cuda.current_stream(dev)
            for s_ in streams:
                s_.wait_stream(main_st)
            fn(batches)
            for s_ in streams:
                main_st.wait_stream(s_)
            torch.cuda.synchronize(dev)
            return n * batches / (time.perf_counter() - t0)

        for fn in loops.values():                          # warm-up: tables, each mode's graphs, the out= buffers
            timed(fn, 4 * N_CTX)
        rounds = {k: [] for k in LOOPS}
        for _ in range(args.rounds):
            for k in LOOPS:
                rounds[k].append(timed(loops[k], args.batches))

        for k, p in enumerate(pps):                        # the last loop ran device-only: the host readers download
            t = ring[k]
            num, parts, scores = p.human_tables()
            res = p.results(with_peaks=True, raise_on_overflow=False)
            full = p.result_tensors(subset=True, peaks=True, stream=streams[k])
            torch.cuda.synchronize(dev)
            ok = (same(t["num_humans"].cpu().numpy(), num) and same(t["parts"].cpu().numpy().view(_PEAK_DT)[..., 0], parts) and
                  same(t["scores"].cpu().numpy(), scores) and same(t["n_peaks"].cpu().numpy(), res["n_peaks"]) and
                  same(t["overflow"].cpu().numpy().view(np.uint32), res["overflow"]) and
                  same(full["subset"].cpu().numpy(), res["subset"]) and
                  same(full["peaks"].cpu().numpy().view(_PEAK_DT)[..., 0], res["peaks"]) and
                  same(full["part_off"].cpu().numpy(), res["part_off"]))
            if not ok:
                failures.append(f"{name} context {k}: the device tables differ from the host tables")
        people = [int(x) for x in pps[0].results(raise_on_overflow=False)["num_humans"]]
        for p in pps:
            p.close()

        med = {k: float(np.median(v)) for k, v in rounds.items()}
        results[name] = {
            "workload": f"synthetic.make_batch({n}, {h}, {w}, {wl['people']}), 4 seeded input sets on the device, "
                        f"{wl['frontend']} front-end, no materialisation, max_peaks {wl['max_peaks']}, max_humans {wl['max_humans']}, "
                        f"{N_CTX} contexts on {N_CTX} streams",
            "people_per_image_context0": {"min": min(people), "max": max(people), "mean": float(np.mean(people))},
            "d2h_bytes_per_batch": record_stride(wl["max_humans"]) * n,
            "images_per_s_rounds": rounds,
            "images_per_s_median": med,
            "spread_over_median": {k: (max(v) - min(v)) / med[k] for k, v in rounds.items()},
            "device_over_copy": {"runs": med["runs_device"] / med["runs_copy"], "export": med["export_device"] / med["export_copy"]},
        }

    out = {
        "what": "ekp_set_host_copy: pipelined images/s with and without the per-batch device-to-host copy of the result "
                "records, runs only and runs plus the device export (tools/time_device_only.py)",
        "card": card(0), "torch_device_name": torch.cuda.get_device_name(0),
        "how": f"{args.batches} batches per loop and round, {args.rounds} rounds alternating {' / '.join(LOOPS)}; images over "
               "the wall time from a synchronised device to a synchronised device",
        "workloads": results,
        "checks": {"failures": failures, "ok": not failures},
        "timestamp": time.strftime("%Y-%m-%dT%H:%M:%S"),
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r5_device_only.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))
    if failures:
        print("\n".join(failures), file=sys.stderr)
        raise SystemExit(1)


if __name__ == "__main__":
    main()
