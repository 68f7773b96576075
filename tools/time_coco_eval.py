#!/usr/bin/env python
"""Device time of one COCO keypoint evaluation (ekp_coco_eval_kpts / coco_eval.evaluate_keypoints), in one run.

Sets are COCO-val-like synthetic tables (tests/test_coco_eval.py `_big_set`): up to 20 ground-truth people and up to 20
detections per image, 3% crowds, pycocotools' keypoint defaults (10 OKS thresholds, 101 recall thresholds, 3 areas,
max_det 20).  Per set size (5,000 and 100,000 images): the device time of one evaluation as CUDA events around --iters
evaluations on one stream after --warmup warm ones, the workspace reused, the stream synchronised at the end; the
device's precision / recall / scores are checked bit for bit against ekp_debug_coco_eval_host on the 5,000-image set.
Next to these, the NumPy restatement of pycocotools in tests/test_coco_eval.py (not pycocotools, which is not installed)
timed on one core on the first --restated images of the 5,000-image set.  The card's name and power limit are read in
the same run.

    python tools/time_coco_eval.py [--out DIR] [--iters 50] [--warmup 5] [--restated 200]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "time_coco_eval"), help="directory of the JSON record")
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--restated", type=int, default=200)
    args = ap.parse_args()

    import torch
    from torch_ekpose_b200 import coco_eval
    from tests.test_coco_eval import COCOevalKps, _big_set, _dev_tables, _tables_to_coco, host_eval

    assert torch.cuda.is_available(), "this tool measures the device: it needs a CUDA device"
    rec = dict(card=card(0), workload="COCO-val-like synthetic sets: 0-20 gts and 0-20 dts per image, pycocotools keypoint "
                                     "defaults (T=10, R=101, A=3, max_det=20)", sets={})
    for n_img in (5000, 100000):
        rng = np.random.default_rng(n_img)
        gtn, dtn = _big_set(rng, n_img)
        gt, dt = _dev_tables(torch, gtn, dtn)
        ws = None
        for _ in range(args.warmup):
            ev = coco_eval.evaluate_keypoints(gt, dt, workspace=ws)
            ws = ev._keep[2]
        torch.cuda.synchronize()
        if n_img == 5000:
            host = host_eval(gtn, dtn)
            for k in ("precision", "recall", "scores"):
                assert np.array_equal(getattr(ev, k).cpu().numpy().view(np.uint64), host[k].view(np.uint64)), k
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(args.iters):
            ev = coco_eval.evaluate_keypoints(gt, dt, workspace=ws)
        t1.record()
        torch.cuda.synchronize()
        ms = t0.elapsed_time(t1) / args.iters
        stats = ev.stats()
        rec["sets"][str(n_img)] = dict(images=n_img, sorted_detections=int(np.minimum(dtn["count"], 20).sum()),
                                       gts=int(gtn["count"].sum()), device_ms_per_evaluation=round(ms, 4),
                                       workspace_bytes=int(ws.numel()), ap=float(stats[0]), checked_against_host_hook=n_img == 5000)
        print(n_img, "images:", f"{ms:.3f} ms per evaluation", flush=True)
    # the NumPy restatement on one core, on the first images of the 5,000-image set
    rng = np.random.default_rng(5000)
    gtn, dtn = _big_set(rng, 5000)
    k = args.restated
    ds, res = _tables_to_coco({f: v[:k] for f, v in gtn.items()}, {f: v[:k] for f, v in dtn.items()})
    t = time.perf_counter()
    COCOevalKps(ds, res, check_margin=False).run().summarize()
    sec = time.perf_counter() - t
    rec["numpy_restatement_one_core"] = dict(images=k, seconds=round(sec, 3), ms_per_image=round(1e3 * sec / k, 3),
                                             note="the NumPy restatement of pycocotools in tests/test_coco_eval.py, not "
                                                  "pycocotools itself; evaluate + accumulate + summarize")
    print("restatement:", f"{sec:.2f} s for {k} images", flush=True)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "r7_coco_eval.json")
    with open(path, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
