"""COCO keypoint evaluation on the device (``ekp_coco_eval_kpts``): pycocotools' ``COCOeval(..., 'keypoints')`` for one
category, with its ``precision``, ``recall`` and ``scores`` arrays equal bit for bit and ``stats`` computed from them by
``_summarizeKps``' rules.

    gt = gt_tables(dataset)                         # a person_keypoints_*.json dict, packed once and uploaded
    dt = dt_tables(results, gt["img_ids"])          # a COCO result list (what eval.py hands to loadRes), or
    dt = dt_tables_from_results(pp.result_tensors(), map_hw, upsample_keypoints)   # the people, never leaving the GPU
    ev = evaluate_keypoints(gt, dt)                 # asynchronous: ev.precision / ev.recall / ev.scores CUDA tensors
    ev.stats()                                      # waits; the 10 numbers of COCOeval.summarize() for keypoints

Tables are dicts of arrays with the image on axis 0 (``concat_tables`` joins batches).  The packers work in NumPy
(``pack_gt`` / ``pack_dt``) and upload once; the full rule text is in include/ekpose_b200.h.  The package imports
without torch; the device entry points need it.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _lib
from .coco import ORDER_COCO

try:  # as in paf_to_pose: the host surface imports without torch
    import torch
except Exception:  # pragma: no cover
    torch = None

# pycocotools' Params(iouType='keypoints'), computed exactly as it computes them
IOU_THRS = np.linspace(.5, 0.95, int(np.round((0.95 - .5) / .05)) + 1, endpoint=True)
REC_THRS = np.linspace(.0, 1.00, int(np.round((1.00 - .0) / .01)) + 1, endpoint=True)
AREA_RNG = np.array([[0 ** 2, 1e5 ** 2], [32 ** 2, 96 ** 2], [96 ** 2, 1e5 ** 2]], np.float64)
AREA_LBL = ("all", "medium", "large")
MAX_DET = 20
PERSON = 1

GT_FIELDS = ("count", "keypoints", "bbox", "area", "iscrowd", "ignore")
DT_FIELDS = ("count", "keypoints", "score")


def _img_ids(img_ids) -> np.ndarray:
    return np.unique(np.asarray(list(img_ids), np.int64))   # p.imgIds = list(np.unique(p.imgIds))


def pack_gt(dataset: dict, img_ids=None, cat_id: int = PERSON) -> dict:
    """The ground-truth tables of ``dataset`` (a COCO person-keypoints annotation dict) as NumPy arrays: ``count`` int32
    [n], ``keypoints`` float64 [n, max_gt, 17, 3], ``bbox`` float64 [n, max_gt, 4], ``area`` float64 [n, max_gt],
    ``iscrowd`` / ``ignore`` int32 [n, max_gt] (``ignore`` = iscrowd or num_keypoints == 0, as ``_prepare`` sets it),
    and ``img_ids`` int64 [n].  Images are the sorted unique ``img_ids`` (default: every image of the dataset); rows
    are the image's annotations of ``cat_id`` in annotation order."""
    ids = _img_ids([im["id"] for im in dataset.get("images", [])] if img_ids is None else img_ids)
    row = {int(i): k for k, i in enumerate(ids)}
    per = [[] for _ in ids]
    for ann in dataset.get("annotations", []):
        k = row.get(int(ann["image_id"]))
        if k is not None and ann.get("category_id", cat_id) == cat_id:
            per[k].append(ann)
    n, mg = len(ids), max([1] + [len(p) for p in per])
    out = dict(count=np.array([len(p) for p in per], np.int32), keypoints=np.zeros((n, mg, 17, 3)),
               bbox=np.zeros((n, mg, 4)), area=np.zeros((n, mg)), iscrowd=np.zeros((n, mg), np.int32),
               ignore=np.zeros((n, mg), np.int32), img_ids=ids)
    for k, anns in enumerate(per):
        for g, a in enumerate(anns):
            out["keypoints"][k, g] = np.asarray(a["keypoints"], np.float64).reshape(17, 3)
            out["bbox"][k, g] = a["bbox"]
            out["area"][k, g] = a["area"]
            out["iscrowd"][k, g] = int(a["iscrowd"])
            out["ignore"][k, g] = int(bool(a["iscrowd"]) or a["num_keypoints"] == 0)
    return out


def pack_dt(results: Sequence[dict], img_ids) -> dict:
    """The detection tables of a COCO keypoint result list as NumPy arrays: ``count`` int32 [n], ``keypoints`` float64
    [n, max_dt, 17, 3], ``score`` float64 [n, max_dt], ``img_ids``.  Image k is the k-th of the sorted unique
    ``img_ids``; its rows are its results in list order.  Results for other images are dropped, as COCOeval drops
    them."""
    ids = _img_ids(img_ids)
    row = {int(i): k for k, i in enumerate(ids)}
    per = [[] for _ in ids]
    for r in results:
        k = row.get(int(r["image_id"]))
        if k is not None:
            per[k].append(r)
    n, md = len(ids), max([1] + [len(p) for p in per])
    out = dict(count=np.array([len(p) for p in per], np.int32), keypoints=np.zeros((n, md, 17, 3)),
               score=np.zeros((n, md)), img_ids=ids)
    for k, rs in enumerate(per):
        for d, r in enumerate(rs):
            out["keypoints"][k, d] = np.asarray(r["keypoints"], np.float64).reshape(17, 3)
            out["score"][k, d] = r["score"]
    return out


def _upload(tables: dict, device) -> dict:
    dev = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
    return {k: (torch.from_numpy(np.ascontiguousarray(v)).to(dev) if k != "img_ids" else v) for k, v in tables.items()}


def gt_tables(dataset: dict, img_ids=None, device=0, cat_id: int = PERSON) -> dict:
    """``pack_gt`` uploaded to ``device`` (``img_ids`` stays a NumPy array)."""
    return _upload(pack_gt(dataset, img_ids, cat_id), device)


def dt_tables(results: Sequence[dict], img_ids, device=0) -> dict:
    """``pack_dt`` uploaded to ``device``."""
    return _upload(pack_dt(results, img_ids), device)


def dt_tables_from_results(tensors: dict, map_hw, upsample_keypoints, scores=None) -> dict:
    """The detection tables of the people of ``result_tensors()`` (``num_humans`` and ``parts`` are read), built on their
    device with ``coco.coco_keypoints``' float64 arithmetic: keypoint j = part ``ORDER_COCO[j]``, ``x / W *
    upsample_keypoints[1] + 0.5`` and ``y / H * upsample_keypoints[0] + 0.5`` for present parts, (0, 0, 0) for absent
    ones; ``map_hw`` = (H, W) of the full-resolution map, ``upsample_keypoints`` one (up_h, up_w) pair or one per
    image.  The score is eval.py's 1.0, or ``scores`` [n, max_humans] (e.g. ``tensors["scores"]``).  Bit-identical to
    ``coco_keypoints`` on the same tables; no host wait."""
    num, parts = tensors["num_humans"], tensors["parts"]
    if not (torch is not None and isinstance(parts, torch.Tensor) and parts.dim() == 4 and tuple(parts.shape[2:]) == (_lib.NUM_PART, 4)):
        raise ValueError("tensors['parts'] must be an int32 tensor [n, max_humans, 18, 4]")
    n, mh = int(parts.shape[0]), int(parts.shape[1])
    dev = parts.device
    H, W = map_hw
    ups = np.broadcast_to(np.asarray(upsample_keypoints, np.float64).reshape(-1, 2), (n, 2)).copy()
    ups = torch.from_numpy(ups).pin_memory().to(dev, non_blocking=True)   # pinned: the copy does not wait
    p = parts[:, :, ORDER_COCO]
    present = p[..., 3] >= 0
    zero = torch.zeros((), dtype=torch.float64, device=dev)
    # elementwise divisions by full tensors: a CPU scalar divisor would become a multiplication by its reciprocal
    x = p[..., 0].double() / torch.full((n, mh, 17), float(W), dtype=torch.float64, device=dev)
    y = p[..., 1].double() / torch.full((n, mh, 17), float(H), dtype=torch.float64, device=dev)
    kp = torch.stack([torch.where(present, x * ups[:, 1, None, None] + 0.5, zero),
                      torch.where(present, y * ups[:, 0, None, None] + 0.5, zero), present.double()], dim=-1)
    score = torch.ones((n, mh), dtype=torch.float64, device=dev) if scores is None else scores.to(dev, torch.float64).reshape(n, mh)
    count = num.to(dev, torch.int32).clamp(0, mh)
    return dict(count=count.contiguous(), keypoints=kp.contiguous(), score=score.contiguous())


def concat_tables(tables: Sequence[dict]) -> dict:
    """Tables of several batches (NumPy or torch, all of one kind) joined along the image axis, rows padded to the
    largest ``max_gt`` / ``max_dt``."""
    out = {}
    for k in tables[0]:
        parts = [t[k] for t in tables]
        if k in ("count", "img_ids"):
            out[k] = torch.cat(parts) if torch is not None and isinstance(parts[0], torch.Tensor) else np.concatenate(parts)
            continue
        m = max(int(p.shape[1]) for p in parts)
        if torch is not None and isinstance(parts[0], torch.Tensor):
            out[k] = torch.cat([torch.nn.functional.pad(p, [0, 0] * (p.dim() - 2) + [0, m - p.shape[1]]) for p in parts])
        else:
            out[k] = np.concatenate([np.pad(p, [(0, 0), (0, m - p.shape[1])] + [(0, 0)] * (p.ndim - 2)) for p in parts])
    return out


def summarize(precision: np.ndarray, recall: np.ndarray, iou_thrs=IOU_THRS, area_lbl=AREA_LBL, max_det: int = MAX_DET) -> np.ndarray:
    """The 10 numbers of ``COCOeval._summarizeKps`` from precision [T, R, A] and recall [T, A]: means over the entries
    > -1 (or -1 when there are none) for all thresholds, t = .5, t = .75 (found by exact equality in ``iou_thrs``), and
    the medium and large areas.  ``_summarizeKps`` asks for maxDets=20, so every number is -1 for another max_det."""
    def one(ap, iou_thr=None, area="all"):
        if max_det != 20:
            return -1.0
        aind = [i for i, lbl in enumerate(area_lbl) if lbl == area]
        s = precision if ap else recall
        if iou_thr is not None:
            s = s[np.where(iou_thr == np.asarray(iou_thrs))[0]]
        s = s[:, :, aind] if ap else s[:, aind]
        return -1.0 if len(s[s > -1]) == 0 else np.mean(s[s > -1])
    return np.array([one(1), one(1, .5), one(1, .75), one(1, area="medium"), one(1, area="large"),
                     one(0), one(0, .5), one(0, .75), one(0, area="medium"), one(0, area="large")], np.float64)


class KeypointEval:
    """One evaluation in flight: ``precision`` [T, R, A], ``recall`` [T, A] and ``scores`` [T, R, A] float64 CUDA tensors
    (pycocotools' arrays with the category and max-detection axes dropped), complete once ``event`` has fired."""

    def __init__(self, precision, recall, scores, event, keep, iou_thrs, area_lbl, max_det):
        self.precision, self.recall, self.scores, self.event = precision, recall, scores, event
        self._keep, self.iou_thrs, self.area_lbl, self.max_det = keep, iou_thrs, area_lbl, max_det

    def synchronize(self) -> None:
        self.event.synchronize()
        self._keep = None

    def stats(self) -> np.ndarray:
        """Waits for the evaluation and returns COCOeval's ``stats`` for keypoints (float64 [10])."""
        self.synchronize()
        return summarize(self.precision.cpu().numpy(), self.recall.cpu().numpy(), self.iou_thrs, self.area_lbl, self.max_det)


_CTX = {}      # device -> PostProcessor: the context supplies the device, the error reporting and the launch count
_THRS = {}     # (device, bytes) -> the thresholds uploaded once


def _context(device: int):
    from .paf_to_pose import PostProcessor
    if device not in _CTX:
        _CTX[device] = PostProcessor(device=device, max_batch=1, max_h=5, max_w=5, max_peaks=16, max_humans=4)
    return _CTX[device]


def _thresholds(dev, arr) -> "torch.Tensor":
    a = np.ascontiguousarray(arr, np.float64)
    key = (dev.index, a.shape, a.tobytes())
    if key not in _THRS:
        _THRS[key] = torch.from_numpy(a.copy()).to(dev)
        torch.cuda.current_stream(dev).synchronize()   # once per set: later calls never wait
    return _THRS[key]


def kernel_launches(device: int = 0) -> int:
    """Kernels launched by the evaluation context of ``device`` so far."""
    return _context(device).kernel_launches()


def evaluate_keypoints(gt: dict, dt: dict, stream=None, max_det: int = MAX_DET, iou_thrs=IOU_THRS, rec_thrs=REC_THRS,
                       area_rng=AREA_RNG, area_lbl=AREA_LBL, workspace: Optional["torch.Tensor"] = None) -> KeypointEval:
    """COCOeval(iouType='keypoints') of the detection tables ``dt`` against the ground-truth tables ``gt`` (CUDA
    tensors on one device, the same images in the same order), with pycocotools' keypoint defaults.  One call of
    ``ekp_coco_eval_kpts`` on ``stream`` (default: the current stream), after whatever wrote the tables there; no host
    wait (the thresholds are uploaded on the first use of each set).  ``workspace``: a CUDA uint8 tensor of at least
    ``ekp_coco_eval_workspace_bytes`` to use instead of a new one."""
    if torch is None:
        raise ImportError("evaluate_keypoints needs torch (its tables and outputs are CUDA tensors)")
    from .paf_to_pose import _torch_stream
    kp = gt["keypoints"]
    dev = kp.device
    if dev.type != "cuda":
        raise ValueError(f"the evaluation runs on a CUDA device, got {dev} (there is no CPU path)")
    for name, t, fields in (("gt", gt, GT_FIELDS), ("dt", dt, DT_FIELDS)):
        for f in fields:
            v = t[f]
            want = torch.int32 if f in ("count", "iscrowd", "ignore") else torch.float64
            if not (isinstance(v, torch.Tensor) and v.device == dev and v.dtype == want and v.is_contiguous()):
                raise ValueError(f"{name}[{f!r}] must be a contiguous {want} tensor on {dev}")
    n, mg, md = int(gt["count"].shape[0]), int(kp.shape[1]), int(dt["keypoints"].shape[1])
    if int(dt["count"].shape[0]) != n:
        raise ValueError(f"gt holds {n} images and dt {int(dt['count'].shape[0])}")
    rng = np.asarray(area_rng, np.float64).reshape(-1, 2)
    T, R, A = len(iou_thrs), len(rec_thrs), len(rng)
    nbytes = int(_lib.lib.ekp_coco_eval_workspace_bytes(n, mg, md, max_det, A, T))
    if not nbytes:
        raise ValueError(f"{n} images, max_gt {mg}, max_dt {md}, max_det {max_det}, {T} thresholds x {A} areas: outside the "
                         "EKP_COCO_LIMIT_* limits")
    ctx = _context(dev.index)
    st = _torch_stream(dev, stream)
    iou_d, rec_d, rng_d = _thresholds(dev, iou_thrs), _thresholds(dev, rec_thrs), _thresholds(dev, rng)
    with torch.cuda.device(dev), torch.cuda.stream(st):
        if workspace is None or workspace.numel() < nbytes or workspace.device != dev:
            workspace = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        prec = torch.empty((T, R, A), dtype=torch.float64, device=dev)
        rec = torch.empty((T, A), dtype=torch.float64, device=dev)
        scores = torch.empty((T, R, A), dtype=torch.float64, device=dev)
    g = _lib.CocoGt(*(gt[f].data_ptr() for f in GT_FIELDS))
    d = _lib.CocoDt(*(dt[f].data_ptr() for f in DT_FIELDS))
    out = _lib.CocoEvalOut(prec.data_ptr(), rec.data_ptr(), scores.data_ptr(), None, None, None)
    _lib.check(_lib.lib.ekp_coco_eval_kpts(ctx._ctx, C.byref(g), mg, C.byref(d), md, n, max_det, iou_d.data_ptr(), T,
                                           rec_d.data_ptr(), R, rng_d.data_ptr(), A, workspace.data_ptr(), C.byref(out),
                                           int(st.cuda_stream)))
    ev = torch.cuda.Event()
    ev.record(st)
    return KeypointEval(prec, rec, scores, ev, (gt, dt, workspace), iou_thrs, area_lbl, max_det)
