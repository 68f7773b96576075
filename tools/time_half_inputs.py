#!/usr/bin/env python
"""bf16 / fp16 heat and PAF maps against float32 on one GPU, in one run:

  e2e          bench.py's e2e leg (configs[1]: 64 x 368x432 per batch, dense front-end materialising, 8 contexts
               rotating over 8 streams, one pinned host block per batch, H2D copies and the result tables read back
               inside the timed window) with PinnedBatch blocks of each dtype, next to the in-run pinned H2D ceiling
               for each block size (36 MB float32, 18 MB 16-bit);
  device       per-batch device time (CUDA events over the timed batches of one context) for maps already in HBM:
               float32 / bf16 through .float() + run (what infer_humans did) / bf16 through the native typed entry,
               for the lean reference front-end (the infer_humans default) and the lean dense front-end.

Legs alternate fp32 / bf16 / fp16 (resp. the three device cases) for three rounds on the same seeded
synthetic.make_batch inputs.  Every 16-bit leg's results are checked against the float32 path on x16.float() and the
script exits non-zero on any difference.  The card's name and power limit are read in the same run.

    python tools/time_half_inputs.py [--out DIR] [--batches 160] [--device-batches 48] [--rounds 3]
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

BATCH, H_LO, W_LO, PEOPLE = 64, 46, 54, (1, 6)   # bench.py configs[1]
N_CTX, INPUT_SETS = 8, 4
PIN_DTYPES = {"fp32": "float32", "bf16": "bfloat16", "fp16": "float16"}


def card(index):
    info = {}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,power.max_limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, pl, pmax, sm = [x.strip() for x in out.split(",")]
        info = {"name": name, "power_limit": pl, "power_max_limit": pmax, "sm_max_clock": sm}
    except Exception as e:   # the numbers are still reported, with the reason the card could not be read
        info = {"query_error": repr(e)}
    return info


def tables_equal(a, b):
    return all(np.array_equal(np.ascontiguousarray(x).view(np.uint8), np.ascontiguousarray(y).view(np.uint8)) for x, y in zip(a, b))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "time_half_inputs"), help="directory of the JSON record")
    ap.add_argument("--batches", type=int, default=160, help="timed batches per e2e leg")
    ap.add_argument("--device-batches", type=int, default=48, help="timed batches per device leg (>= 32)")
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_half_inputs.py: no CUDA device (there is nothing to measure on the CPU)")
    import torch_ekpose_b200 as ek
    from torch_ekpose_b200 import synthetic

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    main_stream = torch.cuda.current_stream(dev)
    host = [synthetic.make_batch(BATCH, H_LO, W_LO, PEOPLE, seed=100 + s) for s in range(INPUT_SETS)]
    tdt = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}
    failures = []

    # float32 results of every input set in every dtype's values (x16.float()): what each leg must reproduce
    ref_pp = ek.PostProcessor(device=0, max_batch=BATCH, max_h=H_LO, max_w=W_LO, max_peaks=1024, max_humans=32, max_part=64, max_cand=512)

    def reference(dt, s, frontend, materialize):
        h, p = (torch.from_numpy(x).to(dev).to(tdt[dt]).float() for x in host[s])
        ref_pp.run(h, p, frontend=frontend, materialize=materialize)
        return ref_pp.human_tables()

    # ---- e2e -------------------------------------------------------------------------------------------------------
    pps = [ek.PostProcessor(device=0, max_batch=BATCH, max_h=H_LO, max_w=W_LO, max_peaks=1024, max_humans=32, max_part=64, max_cand=512)
           for _ in range(N_CTX)]
    streams = [torch.cuda.Stream(dev) for _ in range(N_CTX)]
    pinned = {}
    for dt, name in PIN_DTYPES.items():
        blocks = []
        for s in range(INPUT_SETS):
            pb = ek.PinnedBatch(BATCH, H_LO, W_LO, "nchw", dtype=name)
            h, p = (torch.from_numpy(x).to(tdt[dt]) for x in host[s])   # rounded by torch, as the reference runs are
            if dt == "bf16":
                pb.heat.copy_(h); pb.paf.copy_(p)
            else:
                np.copyto(pb.heat, h.numpy()); np.copyto(pb.paf, p.numpy())
            blocks.append(pb)
        pinned[dt] = blocks

    def e2e_loop(dt, batches):
        last = {}
        for i in range(batches + N_CTX):
            if i >= N_CTX:   # results of batch i - N_CTX (waits for it)
                j = i - N_CTX
                last[j % INPUT_SETS] = pps[j % N_CTX].human_tables()
            if i < batches:
                k = i % N_CTX
                pb = pinned[dt][i % INPUT_SETS]
                pps[k].run(pb.heat, pb.paf, layout="nchw", frontend="dense", materialize=True, stream=streams[k])
        return last

    def fork():
        for s_ in streams:
            s_.wait_stream(main_stream)

    def join():
        for s_ in streams:
            main_stream.wait_stream(s_)

    e2e = {dt: [] for dt in PIN_DTYPES}
    for dt in PIN_DTYPES:
        e2e_loop(dt, 2 * N_CTX)   # warm-up: graphs captured, materialised tensors allocated
    for rnd in range(args.rounds):
        for dt in PIN_DTYPES:
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(main_stream)
            fork()
            last = e2e_loop(dt, args.batches)
            join()
            e1.record(main_stream)
            torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1)
            e2e[dt].append(BATCH * args.batches / (ms / 1e3))
            if rnd == 0:
                for s, got in last.items():
                    if not tables_equal(reference(dt, s, "dense", True), got):
                        failures.append(f"e2e {dt} input set {s}: results differ from the float32 path on x.float()")

    # in-run pinned H2D ceiling per block size: N_CTX streams x 8 copies of one block each, best of 3 (as bench.py)
    ceiling = {}
    for label, nbytes in (("fp32_block", pinned["fp32"][0].nbytes), ("16bit_block", pinned["bf16"][0].nbytes)):
        dst = [torch.empty(nbytes, dtype=torch.uint8, device=dev) for _ in range(N_CTX)]
        src = [torch.empty(nbytes, dtype=torch.uint8).pin_memory() for _ in range(N_CTX)]

        def h2d_round(reps):
            for _ in range(reps):
                for k in range(N_CTX):
                    with torch.cuda.stream(streams[k]):
                        dst[k].copy_(src[k], non_blocking=True)
        h2d_round(2)
        best = 0.0
        for _ in range(3):
            torch.cuda.synchronize(dev)
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record(main_stream)
            fork()
            h2d_round(8)
            join()
            c1.record(main_stream)
            torch.cuda.synchronize(dev)
            best = max(best, nbytes * 8 * N_CTX / (c0.elapsed_time(c1) / 1e3) / 1e9)
        ceiling[label] = {"block_bytes": nbytes, "gbs": best, "images_per_s_if_copy_bound": best * 1e9 / (nbytes / BATCH)}
        del dst, src
    for pp in pps:
        pp.close()
    for blocks in pinned.values():
        for pb in blocks:
            pb.close()
    torch.cuda.empty_cache()

    # ---- device path -----------------------------------------------------------------------------------------------
    dev16 = [tuple(torch.from_numpy(x).to(dev).to(torch.bfloat16) for x in host[s]) for s in range(INPUT_SETS)]
    dev32 = [tuple(x.float() for x in pair) for pair in dev16]     # the same values, float32, already in HBM
    cases = {
        "fp32_in_hbm": lambda pp, s, fe: pp.run(*dev32[s], frontend=fe),
        "bf16_float_then_run": lambda pp, s, fe: pp.run(dev16[s][0].float(), dev16[s][1].float(), frontend=fe),
        "bf16_native": lambda pp, s, fe: pp.run(*dev16[s], frontend=fe),
    }
    device = {}
    for fe in ("reference", "dense"):
        pps = {c: ek.PostProcessor(device=0, max_batch=BATCH, max_h=H_LO, max_w=W_LO, max_peaks=1024, max_humans=32, max_part=64,
                                   max_cand=512) for c in cases}
        want = [reference("bf16", s, fe, False) for s in range(INPUT_SETS)]
        ent = {c: {"ms_per_batch": [], "graph_launches": 0, "batches": 0} for c in cases}
        for c, fn in cases.items():   # warm-up, and every case's results against the float32 path
            for s in range(INPUT_SETS):
                fn(pps[c], s, fe)
                if not tables_equal(want[s], pps[c].human_tables()):
                    failures.append(f"device {fe} {c} input set {s}: results differ from the float32 path")
                fn(pps[c], s, fe)
        torch.cuda.synchronize(dev)
        for _ in range(args.rounds):
            for c, fn in cases.items():
                g0 = pps[c].graph_launches()
                torch.cuda.synchronize(dev)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(main_stream)
                for i in range(args.device_batches):
                    fn(pps[c], i % INPUT_SETS, fe)
                e1.record(main_stream)
                torch.cuda.synchronize(dev)
                ent[c]["ms_per_batch"].append(e0.elapsed_time(e1) / args.device_batches)
                ent[c]["graph_launches"] += pps[c].graph_launches() - g0
                ent[c]["batches"] += args.device_batches
        for c in cases:
            v = ent[c]["ms_per_batch"]
            ent[c]["median_ms_per_batch"] = float(np.median(v))
            ent[c]["images_per_s"] = BATCH / (float(np.median(v)) / 1e3)
            pps[c].close()
        device[fe + "_lean"] = ent

    out = {
        "what": "bf16 / fp16 heat+PAF inputs vs float32 (tools/time_half_inputs.py)",
        "card": card(0), "torch_device_name": torch.cuda.get_device_name(0),
        "workload": f"synthetic.make_batch({BATCH}, {H_LO}, {W_LO}, {PEOPLE}, seed=100..{100 + INPUT_SETS - 1}), NCHW",
        "rounds": args.rounds, "order": "legs alternate fp32 / bf16 / fp16 within every round",
        "e2e": {
            "how": f"{N_CTX} contexts on {N_CTX} streams, one PinnedBatch per batch ({INPUT_SETS} rotating), PostProcessor.run "
                   "(ekp_postprocess_host_typed) dense materialising + human_tables(), copies inside the timed window; "
                   f"{args.batches} batches per leg",
            "images_per_s": {dt: {"rounds": v, "median": float(np.median(v))} for dt, v in e2e.items()},
            "h2d_ceiling": ceiling,
        },
        "device": {"how": f"one context, {args.device_batches} batches per leg timed with CUDA events on its stream, "
                          "inputs already on the device; lean (non-materialising)", **device},
        "checks": {"failures": failures, "ok": not failures},
        "timestamp": time.strftime("%Y-%m-%dT%H:%M:%S"),
    }
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "time_half_inputs.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))
    ref_pp.close()
    if failures:
        print("\n".join(failures), file=sys.stderr)
        raise SystemExit(1)


if __name__ == "__main__":
    main()
