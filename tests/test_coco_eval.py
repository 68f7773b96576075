"""COCO keypoint evaluation (ekp_coco_eval_kpts / coco_eval.evaluate_keypoints) against a NumPy restatement of
pycocotools' COCOeval(iouType='keypoints'), structured like pycocotools itself (loadRes' area, _prepare, computeOks,
evaluateImg, accumulate, _summarizeKps), since the package is not installed here.  The restatement is pinned by hand-worked
answers; on the CPU, ekp_debug_coco_eval_host (the kernels' own code run serially) must equal it on thousands of random
image sets; on the GPU, the device."""
import copy
import ctypes as C

import numpy as np
import pytest

from torch_ekpose_b200 import _lib, coco_eval
from torch_ekpose_b200.coco import ORDER_COCO

SIGMAS = np.array([.26, .25, .25, .35, .35, .79, .79, .72, .72, .62, .62, 1.07, 1.07, .87, .87, .89, .89]) / 10.0
MARGIN = 1e-9


class MarginError(AssertionError):
    """An OKS within MARGIN of a threshold, or two competing OKS values that close without being equal: the device's exp
    and NumPy's may differ by an ulp, so such a set does not pin the result."""


# ---- the restatement ----------------------------------------------------------------------------------------------------
def load_res(results):
    """COCO.loadRes for keypoint results: area over all 17 keypoints (absent triples included), ids from 1."""
    anns = copy.deepcopy(list(results))
    for id, ann in enumerate(anns):
        s = ann["keypoints"]
        x = s[0::3]
        y = s[1::3]
        x0, x1, y0, y1 = np.min(x), np.max(x), np.min(y), np.max(y)
        ann["area"] = (x1 - x0) * (y1 - y0)
        ann["id"] = id + 1
        ann["bbox"] = [x0, y0, x1 - x0, y1 - y0]
    return anns


class COCOevalKps:
    def __init__(self, dataset, results, img_ids=None, max_det=20, iou_thrs=coco_eval.IOU_THRS,
                 rec_thrs=coco_eval.REC_THRS, area_rng=coco_eval.AREA_RNG, check_margin=True):
        self.dataset, self.results = dataset, results
        ids = [im["id"] for im in dataset["images"]] if img_ids is None else img_ids
        self.imgIds = list(np.unique(ids))
        self.maxDets = [max_det]
        self.iouThrs, self.recThrs = np.asarray(iou_thrs), np.asarray(rec_thrs)
        self.areaRng = [list(a) for a in np.asarray(area_rng).reshape(-1, 2)]
        self.check_margin = check_margin

    def _prepare(self):
        self._gts = {i: [] for i in self.imgIds}
        self._dts = {i: [] for i in self.imgIds}
        for gt in copy.deepcopy(self.dataset["annotations"]):
            if gt["image_id"] in self._gts and gt["category_id"] == 1:
                gt["ignore"] = gt["ignore"] if "ignore" in gt else 0
                gt["ignore"] = "iscrowd" in gt and gt["iscrowd"]
                gt["ignore"] = (gt["num_keypoints"] == 0) or gt["ignore"]
                self._gts[gt["image_id"]].append(gt)
        for dt in load_res(self.results):
            if dt["image_id"] in self._dts:
                self._dts[dt["image_id"]].append(dt)

    def computeOks(self, imgId):
        gts, dts = self._gts[imgId], self._dts[imgId]
        inds = np.argsort([-d["score"] for d in dts], kind="mergesort")
        dts = [dts[i] for i in inds]
        if len(dts) > self.maxDets[-1]:
            dts = dts[0:self.maxDets[-1]]
        if len(gts) == 0 or len(dts) == 0:
            return []
        ious = np.zeros((len(dts), len(gts)))
        vars = (SIGMAS * 2) ** 2
        k = len(SIGMAS)
        for j, gt in enumerate(gts):
            g = np.array(gt["keypoints"])
            xg, yg, vg = g[0::3], g[1::3], g[2::3]
            k1 = np.count_nonzero(vg > 0)
            bb = gt["bbox"]
            x0, x1 = bb[0] - bb[2], bb[0] + bb[2] * 2
            y0, y1 = bb[1] - bb[3], bb[1] + bb[3] * 2
            for i, dt in enumerate(dts):
                d = np.array(dt["keypoints"])
                xd, yd = d[0::3], d[1::3]
                if k1 > 0:
                    dx, dy = xd - xg, yd - yg
                else:
                    z = np.zeros((k))
                    dx = np.max((z, x0 - xd), axis=0) + np.max((z, xd - x1), axis=0)
                    dy = np.max((z, y0 - yd), axis=0) + np.max((z, yd - y1), axis=0)
                e = (dx ** 2 + dy ** 2) / vars / (gt["area"] + np.spacing(1)) / 2
                if k1 > 0:
                    e = e[vg > 0]
                ious[i, j] = np.sum(np.exp(-e)) / e.shape[0]
        if self.check_margin:
            thr = np.minimum(self.iouThrs, 1 - 1e-10)
            near = np.abs(ious[..., None] - thr)
            if ((near < MARGIN) & (near > 0)).any():
                raise MarginError("an OKS within 1e-9 of a threshold")
            for row in ious:   # only values that can match compete
                v = np.unique(row[row >= thr.min() - MARGIN])
                if len(v) > 1 and (np.diff(v) < MARGIN).any():
                    raise MarginError("two OKS of one detection within 1e-9")
        return ious

    def evaluateImg(self, imgId, aRng, maxDet):
        gt, dt = self._gts[imgId], self._dts[imgId]
        if len(gt) == 0 and len(dt) == 0:
            return None
        for g in gt:
            g["_ignore"] = 1 if (g["ignore"] or (g["area"] < aRng[0] or g["area"] > aRng[1])) else 0
        gtind = np.argsort([g["_ignore"] for g in gt], kind="mergesort")
        gt = [gt[i] for i in gtind]
        dtind = np.argsort([-d["score"] for d in dt], kind="mergesort")
        dt = [dt[i] for i in dtind[0:maxDet]]
        iscrowd = [int(o["iscrowd"]) for o in gt]
        ious = self.ious[imgId][:, gtind] if len(self.ious[imgId]) > 0 else self.ious[imgId]
        T, G, D = len(self.iouThrs), len(gt), len(dt)
        gtm = np.zeros((T, G))
        dtm = np.zeros((T, D))
        gtIg = np.array([g["_ignore"] for g in gt])
        dtIg = np.zeros((T, D))
        if not len(ious) == 0:
            for tind, t in enumerate(self.iouThrs):
                for dind, d in enumerate(dt):
                    iou = min([t, 1 - 1e-10])
                    m = -1
                    for gind, g in enumerate(gt):
                        if gtm[tind, gind] > 0 and not iscrowd[gind]:
                            continue
                        if m > -1 and gtIg[m] == 0 and gtIg[gind] == 1:
                            break
                        if ious[dind, gind] < iou:
                            continue
                        iou = ious[dind, gind]
                        m = gind
                    if m == -1:
                        continue
                    dtIg[tind, dind] = gtIg[m]
                    dtm[tind, dind] = gt[m]["id"]
                    gtm[tind, m] = d["id"]
        a = np.array([d["area"] < aRng[0] or d["area"] > aRng[1] for d in dt]).reshape((1, len(dt)))
        dtIg = np.logical_or(dtIg, np.logical_and(dtm == 0, np.repeat(a, T, 0)))
        return {"image_id": imgId, "aRng": aRng, "maxDet": maxDet, "dtIds": [d["id"] for d in dt],
                "gtIds": [g["id"] for g in gt], "dtMatches": dtm, "gtMatches": gtm,
                "dtScores": [d["score"] for d in dt], "gtIgnore": gtIg, "dtIgnore": dtIg}

    def evaluate(self):
        self._prepare()
        self.ious = {i: self.computeOks(i) for i in self.imgIds}
        maxDet = self.maxDets[-1]
        self.evalImgs = [self.evaluateImg(i, a, maxDet) for a in self.areaRng for i in self.imgIds]

    def accumulate(self):
        T, R, K, A, M = len(self.iouThrs), len(self.recThrs), 1, len(self.areaRng), len(self.maxDets)
        precision = -np.ones((T, R, K, A, M))
        recall = -np.ones((T, K, A, M))
        scores = -np.ones((T, R, K, A, M))
        I0 = len(self.imgIds)
        for k in range(K):
            for a in range(A):
                for m, maxDet in enumerate(self.maxDets):
                    E = [self.evalImgs[a * I0 + i] for i in range(I0)]
                    E = [e for e in E if e is not None]
                    if len(E) == 0:
                        continue
                    dtScores = np.concatenate([e["dtScores"][0:maxDet] for e in E])
                    inds = np.argsort(-dtScores, kind="mergesort")
                    dtScoresSorted = dtScores[inds]
                    dtm = np.concatenate([e["dtMatches"][:, 0:maxDet] for e in E], axis=1)[:, inds]
                    dtIg = np.concatenate([e["dtIgnore"][:, 0:maxDet] for e in E], axis=1)[:, inds]
                    gtIg = np.concatenate([e["gtIgnore"] for e in E])
                    npig = np.count_nonzero(gtIg == 0)
                    if npig == 0:
                        continue
                    tps = np.logical_and(dtm, np.logical_not(dtIg))
                    fps = np.logical_and(np.logical_not(dtm), np.logical_not(dtIg))
                    tp_sum = np.cumsum(tps, axis=1).astype(dtype=np.float64)
                    fp_sum = np.cumsum(fps, axis=1).astype(dtype=np.float64)
                    for t, (tp, fp) in enumerate(zip(tp_sum, fp_sum)):
                        tp, fp = np.array(tp), np.array(fp)
                        nd = len(tp)
                        rc = tp / npig
                        pr = tp / (fp + tp + np.spacing(1))
                        q = np.zeros((R,))
                        ss = np.zeros((R,))
                        recall[t, k, a, m] = rc[-1] if nd else 0
                        pr, q = pr.tolist(), q.tolist()
                        for i in range(nd - 1, 0, -1):
                            if pr[i] > pr[i - 1]:
                                pr[i - 1] = pr[i]
                        inds = np.searchsorted(rc, self.recThrs, side="left")
                        try:
                            for ri, pi in enumerate(inds):
                                q[ri] = pr[pi]
                                ss[ri] = dtScoresSorted[pi]
                        except IndexError:
                            pass
                        precision[t, :, k, a, m] = np.array(q)
                        scores[t, :, k, a, m] = np.array(ss)
        self.eval = dict(precision=precision, recall=recall, scores=scores)

    def summarize(self):
        """_summarizeKps"""
        p = self.eval

        def _summarize(ap=1, iouThr=None, areaRng="all", maxDets=20):
            aind = [i for i, aRng in enumerate(["all", "medium", "large"]) if aRng == areaRng]
            mind = [i for i, mDet in enumerate(self.maxDets) if mDet == maxDets]
            if ap == 1:
                s = p["precision"]
                if iouThr is not None:
                    s = s[np.where(iouThr == self.iouThrs)[0]]
                s = s[:, :, :, aind, mind]
            else:
                s = p["recall"]
                if iouThr is not None:
                    s = s[np.where(iouThr == self.iouThrs)[0]]
                s = s[:, :, aind, mind]
            return -1 if len(s[s > -1]) == 0 else np.mean(s[s > -1])
        return np.array([_summarize(1), _summarize(1, iouThr=.5), _summarize(1, iouThr=.75),
                         _summarize(1, areaRng="medium"), _summarize(1, areaRng="large"), _summarize(0),
                         _summarize(0, iouThr=.5), _summarize(0, iouThr=.75), _summarize(0, areaRng="medium"),
                         _summarize(0, areaRng="large")])

    def run(self):
        self.evaluate()
        self.accumulate()
        return self

    def arrays(self):
        e = self.eval
        return e["precision"][:, :, 0, :, 0], e["recall"][:, 0, :, 0], e["scores"][:, :, 0, :, 0]

    def dt_rows(self):
        """per image [A, T, kept]: the matched gt row (in annotation order) or -1, and dtIgnore"""
        I0, out = len(self.imgIds), {}
        for ii, img in enumerate(self.imgIds):
            row = {g["id"]: r for r, g in enumerate(self._gts[img])}
            ms, igs = [], []
            for a in range(len(self.areaRng)):
                e = self.evalImgs[a * I0 + ii]
                if e is None:
                    ms.append(np.zeros((len(self.iouThrs), 0), np.int64))
                    igs.append(np.zeros((len(self.iouThrs), 0), np.int64))
                    continue
                ms.append(np.vectorize(lambda v: row.get(int(v), -1), otypes=[np.int64])(e["dtMatches"]) if e["dtMatches"].size
                          else e["dtMatches"].astype(np.int64))
                igs.append(e["dtIgnore"].astype(np.int64))
            out[img] = (np.stack(ms), np.stack(igs))
        return out


# ---- the library ----------------------------------------------------------------------------------------------------
def host_eval(gtn, dtn, max_det=20, iou=coco_eval.IOU_THRS, rec=coco_eval.REC_THRS, area=coco_eval.AREA_RNG):
    """ekp_debug_coco_eval_host on packed NumPy tables; every output starts dirty"""
    g = {k: np.ascontiguousarray(gtn[k], np.int32 if k in ("count", "iscrowd", "ignore") else np.float64) for k in coco_eval.GT_FIELDS}
    d = {k: np.ascontiguousarray(dtn[k], np.int32 if k == "count" else np.float64) for k in coco_eval.DT_FIELDS}
    iou, rec = np.ascontiguousarray(iou, np.float64), np.ascontiguousarray(rec, np.float64)
    area = np.ascontiguousarray(np.asarray(area, np.float64).reshape(-1, 2))
    n, mg, md = len(g["count"]), g["keypoints"].shape[1], d["keypoints"].shape[1]
    T, R, A = len(iou), len(rec), len(area)
    out = dict(precision=np.full((T, R, A), np.nan), recall=np.full((T, A), np.nan), scores=np.full((T, R, A), np.nan),
               dt_match=np.full((n, A, T, max_det), 77, np.int32), dt_ignore=np.full((n, A, T, max_det), 77, np.int32),
               oks=np.full((n, max_det, mg), np.nan))
    rc = _lib.lib.ekp_debug_coco_eval_host(C.byref(_lib.CocoGt(*(g[k].ctypes.data for k in coco_eval.GT_FIELDS))), mg,
                                           C.byref(_lib.CocoDt(*(d[k].ctypes.data for k in coco_eval.DT_FIELDS))), md, n,
                                           max_det, iou.ctypes.data, T, rec.ctypes.data, R, area.ctypes.data, A,
                                           C.byref(_lib.CocoEvalOut(*(out[k].ctypes.data for k in ("precision", "recall", "scores", "dt_match", "dt_ignore", "oks")))))
    _lib.check(rc)
    return out


def check_against(E, got, gtn, dtn, max_det, details=True):
    """bit-identical arrays; identical matches and ignores; OKS to 1e-12"""
    p, r, s = E.arrays()
    for name, want in (("precision", p), ("recall", r), ("scores", s)):
        assert np.array_equal(got[name].view(np.uint64), np.ascontiguousarray(want).view(np.uint64)), (name, got[name], want)
    if not details:
        return
    rows = E.dt_rows()
    for ii, img in enumerate(E.imgIds):
        m, ig = rows[img]
        kept = m.shape[2]
        assert np.array_equal(got["dt_match"][ii, :, :, :kept], m), (img, got["dt_match"][ii], m)
        assert np.array_equal(got["dt_ignore"][ii, :, :, :kept], ig), img
        assert (got["dt_match"][ii, :, :, kept:] == -1).all() and (got["dt_ignore"][ii, :, :, kept:] == 0).all()
        o = E.ious[img]
        if len(o):
            assert np.allclose(got["oks"][ii, :o.shape[0], :o.shape[1]], o, rtol=0, atol=1e-12)


# ---- scene generators -----------------------------------------------------------------------------------------------
def _person(rng, cx, cy, s, absent=0.2):
    kp = np.zeros((17, 3))
    kp[:, 0] = np.round(cx + rng.uniform(-0.5, 0.5, 17) * s, 1)
    kp[:, 1] = np.round(cy + rng.uniform(-0.5, 0.5, 17) * s, 1)
    kp[:, 2] = 2
    off = rng.random(17) < absent
    kp[off] = 0
    return kp


def random_set(rng, n_img, max_gt=6, max_dt=8, first_id=1):
    """a dataset dict and a result list: empty images, crowd and num_keypoints == 0 gts, duplicated people, absent
    keypoints, tied scores (+-0 among them), and more detections than max_det on some images"""
    images, anns, results = [], [], []
    aid = first_id
    ids = rng.permutation(np.arange(1, 4 * n_img + 1))[:n_img]
    score_pool = np.array([0.0, -0.0, 0.25, 0.5, 0.5, 0.75, 1.0])
    for img in ids:
        img = int(img)
        images.append({"id": img})
        people = []
        for _ in range(int(rng.integers(0, max_gt + 1)) if rng.random() > 0.1 else 0):
            s = rng.uniform(10, 160)
            kp = _person(rng, rng.uniform(0, 400), rng.uniform(0, 300), s)
            nk = int((kp[:, 2] > 0).sum())
            crowd = int(rng.random() < 0.08)
            if rng.random() < 0.08:
                kp[:] = 0
                nk = 0
            vis = kp[kp[:, 2] > 0]
            if len(vis):
                bx, by = vis[:, 0].min(), vis[:, 1].min()
                bw, bh = vis[:, 0].max() - bx, vis[:, 1].max() - by
            else:
                bx, by, bw, bh = rng.uniform(0, 300), rng.uniform(0, 200), s * 0.6, s
            area = float(np.round(bw * bh * rng.uniform(0.5, 1.5), 2)) if rng.random() > 0.05 else 0.0
            people.append(kp)
            anns.append({"id": aid, "image_id": img, "category_id": 1, "keypoints": kp.reshape(-1).tolist(),
                         "num_keypoints": nk, "bbox": [float(bx), float(by), float(bw), float(bh)], "area": area,
                         "iscrowd": crowd})
            aid += 1
            if rng.random() < 0.1:   # a duplicated gt: equal OKS for every detection
                anns.append(dict(anns[-1], id=aid))
                aid += 1
        for _ in range(int(rng.integers(0, max_dt + 1)) if rng.random() > 0.1 else 0):
            if people and rng.random() < 0.8:
                kp = people[rng.integers(len(people))].copy()
                if not kp[:, 2].any():
                    kp = _person(rng, rng.uniform(0, 400), rng.uniform(0, 300), 60)
                kp[:, :2] += np.round(rng.normal(0, rng.uniform(0.5, 12), (17, 2)), 1)
                kp[:, 2] = 1
                kp[rng.random(17) < 0.1] = 0
            else:
                kp = _person(rng, rng.uniform(0, 400), rng.uniform(0, 300), rng.uniform(10, 160))
                kp[kp[:, 2] > 0, 2] = 1
            sc = float(score_pool[rng.integers(len(score_pool))]) if rng.random() < 0.5 else float(rng.random())
            results.append({"image_id": img, "category_id": 1, "keypoints": kp.reshape(-1).tolist(), "score": sc})
            if rng.random() < 0.1:
                results.append(dict(results[-1]))   # a duplicated detection
    rng.shuffle(results)
    return {"images": images, "annotations": anns, "categories": [{"id": 1}]}, results


def _thresholds(rng):
    if rng.random() < 0.6:
        return coco_eval.IOU_THRS, coco_eval.REC_THRS, coco_eval.AREA_RNG
    T = int(rng.integers(1, 11))
    A = int(rng.integers(1, max(2, 32 // T) + 1))
    A = min(A, 32 // T)
    iou = np.sort(rng.uniform(0.05, 1.0, T))
    rec = np.linspace(0, 1, int(rng.integers(1, 150)))
    lo = rng.uniform(0, 3e4, A)
    area = np.stack([lo, lo + rng.uniform(0, 6e4, A)], 1)
    area[0] = (0, 1e10)
    return iou, rec, area


# ---- hand-worked answers (the restatement itself) -----------------------------------------------------------------------
def _gt(id, img, kp, area=10000.0, crowd=0, nk=None, bbox=(0, 0, 100, 100)):
    kp = np.asarray(kp, np.float64).reshape(17, 3)
    return {"id": id, "image_id": img, "category_id": 1, "keypoints": kp.reshape(-1).tolist(), "area": area,
            "iscrowd": crowd, "num_keypoints": int((kp[:, 2] > 0).sum()) if nk is None else nk, "bbox": list(bbox)}


def _dt(img, kp, score):
    kp = np.asarray(kp, np.float64).reshape(17, 3)
    return {"image_id": img, "category_id": 1, "keypoints": kp.reshape(-1).tolist(), "score": score}


def _pose(x0, y0, v=2):
    kp = np.zeros((17, 3))
    kp[:, 0] = x0 + 5 * np.arange(17)
    kp[:, 1] = y0 + 3 * np.arange(17)
    kp[:, 2] = v
    return kp


def _run(gts, dts, imgs, **kw):
    return COCOevalKps({"images": [{"id": i} for i in imgs], "annotations": gts}, dts, **kw).run()


def test_restatement_all_perfect():
    E = _run([_gt(1, 1, _pose(0, 0)), _gt(2, 2, _pose(50, 50))], [_dt(1, _pose(0, 0), .9), _dt(2, _pose(50, 50), .8)], [1, 2])
    p, r, s = E.arrays()
    top = 2 / (2 + np.spacing(1))   # pr = [1 / (1 + eps), 2 / (2 + eps)]: the envelope is the second everywhere
    assert (p[:, :, 0] == top).all() and (r[:, 0] == 1).all() and (s[:, :, 0] == np.where(coco_eval.REC_THRS <= .5, .9, .8)).all()
    # the gts' area 10000 is 'large' (> 96^2): no non-ignored gt in 'medium', whose entries stay -1
    assert (p[:, :, 1] == -1).all() and (r[:, 1] == -1).all() and (p[:, :, 2] == top).all()
    st = E.summarize()
    assert abs(st[0] - 1) < 1e-15 and st[5] == 1 and st[3] == -1


def test_restatement_false_positive_ranked_first():
    E = _run([_gt(1, 1, _pose(0, 0))], [_dt(1, _pose(300, 300), .9), _dt(1, _pose(0, 0), .5)], [1])
    p, r, s = E.arrays()
    # sorted: fp (tp 0, fp 1), tp (tp 1, fp 1): pr = [0, 1/2(+eps)], envelope [0.5, 0.5]; rc = [0, 1]
    half = 1 / (2 + np.spacing(1))
    assert p[0, 0, 0] == half and (p[0, 1:, 0] == half).all() and r[0, 0] == 1
    assert s[0, 0, 0] == .9 and (s[0, 1:, 0] == .5).all()   # recThr 0 -> position 0


def test_restatement_equal_oks_last_gt_wins_and_crowd_matched_twice():
    gts = [_gt(1, 1, _pose(0, 0)), _gt(2, 1, _pose(0, 0))]   # identical people: equal OKS
    E = _run(gts, [_dt(1, _pose(0, 0), .9)], [1])
    assert E.dt_rows()[1][0][0, 0, 0] == 1                   # the last of the equal gts
    gts = [_gt(1, 1, _pose(0, 0), crowd=1)]
    E = _run(gts, [_dt(1, _pose(0, 0), .9), _dt(1, _pose(0, 0), .8)], [1])
    m, ig = E.dt_rows()[1]
    assert (m[0, :, :] == 0).all() and ig.all()              # both matched to the crowd gt, both ignored
    p, r, _ = E.arrays()
    assert (p == -1).all() and (r == -1).all()               # npig == 0


def test_restatement_non_ignored_first_break():
    # gt 1 crowd (ignored, OKS 1), gt 2 non-ignored with a lower OKS: the dt takes gt 2 and stops at the ignored one
    near = _pose(0, 0)
    near[:, 0] += 2
    gts = [_gt(1, 1, _pose(0, 0), crowd=1), _gt(2, 1, near)]
    E = _run(gts, [_dt(1, _pose(0, 0), .9)], [1])
    assert E.ious[1][0, 0] == 1 and .5 < E.ious[1][0, 1] < 1
    m, ig = E.dt_rows()[1]
    t_ok = E.ious[1][0, 1] >= np.minimum(E.iouThrs, 1 - 1e-10)
    assert (m[0, t_ok, 0] == 1).all() and (m[0, ~t_ok, 0] == 0).all()   # below its OKS: the crowd gt instead
    assert (ig[0, t_ok, 0] == 0).all() and (ig[0, ~t_ok, 0] == 1).all()


def test_restatement_zero_keypoint_gt_uses_the_bbox():
    gts = [_gt(1, 1, np.zeros((17, 3)), bbox=(100, 100, 50, 80), area=4000.0)]
    inside = _pose(100, 100, v=1)
    inside[:, 0] = 120
    inside[:, 1] = 150
    E = _run(gts, [_dt(1, inside, .9)], [1])
    assert E.ious[1][0, 0] == 1.0                         # every keypoint inside [x - w, x + 2w] x [y - h, y + 2h]
    out = inside.copy()
    out[0, 0] = 100 + 100 + 10                            # 10 px right of x1 = x + 2w
    E = _run(gts, [_dt(1, out, .9)], [1])
    e0 = 100.0 / ((SIGMAS[0] * 2) ** 2) / (4000.0 + np.spacing(1)) / 2
    assert E.ious[1][0, 0] == np.sum(np.exp(-np.array([e0] + [0.0] * 16))) / 17
    p, r, _ = E.arrays()
    assert (p == -1).all()                                # num_keypoints == 0: ignored, npig == 0


def test_restatement_no_detections_and_truncation_and_image_order():
    E = _run([_gt(1, 1, _pose(0, 0))], [], [1])
    p, r, s = E.arrays()
    assert (p[:, :, 0] == 0).all() and (r[:, 0] == 0).all() and (s[:, :, 0] == 0).all()
    dts = [_dt(1, _pose(300, 300), 1.0 - k / 100) for k in range(25)] + [_dt(1, _pose(0, 0), .1)]
    E = _run([_gt(1, 1, _pose(0, 0))], dts, [1])
    assert len(E.evalImgs[0]["dtIds"]) == 20 and E.arrays()[1][0, 0] == 0   # the true positive was cut at max_det
    # equal scores across images: image order decides; +-0 scores are equal
    for s0, s1 in ((.5, .5), (0.0, -0.0), (-0.0, 0.0)):
        E = _run([_gt(1, 1, _pose(0, 0)), _gt(2, 2, _pose(0, 0))], [_dt(2, _pose(300, 300), s1), _dt(1, _pose(0, 0), s0)], [1, 2])
        p, r, s = E.arrays()
        # image 1's tp first, then image 2's fp: rc = [.5, .5], pr = [1 / (1 + eps), 1 / (2 + eps)] (the other order
        # would give rc = [0, .5] and precision .5 at recall 0)
        assert (p[0, :51, 0] == 1 / (1 + np.spacing(1))).all() and (p[0, 51:, 0] == 0).all()
        assert s[0, 0, 0] == s0 and np.signbit(s[0, 0, 0]) == np.signbit(s0)


@pytest.mark.parametrize("case", ["perfect", "fp_first", "last_gt", "break", "crowd", "bbox", "trunc", "ties"])
def test_host_hook_equals_restatement_on_the_hand_worked_sets(case):
    near = _pose(0, 0)
    near[:, 0] += 2
    inside = np.zeros((17, 3))
    inside[:, 0], inside[:, 1], inside[:, 2] = 120, 150, 1
    sets = {
        "perfect": ([_gt(1, 1, _pose(0, 0)), _gt(2, 2, _pose(50, 50))], [_dt(1, _pose(0, 0), .9), _dt(2, _pose(50, 50), .8)]),
        "fp_first": ([_gt(1, 1, _pose(0, 0))], [_dt(1, _pose(300, 300), .9), _dt(1, _pose(0, 0), .5)]),
        "last_gt": ([_gt(1, 1, _pose(0, 0)), _gt(2, 1, _pose(0, 0))], [_dt(1, _pose(0, 0), .9)]),
        "break": ([_gt(1, 1, _pose(0, 0), crowd=1), _gt(2, 1, near)], [_dt(1, _pose(0, 0), .9)]),
        "crowd": ([_gt(1, 1, _pose(0, 0), crowd=1), _gt(2, 2, _pose(0, 0))], [_dt(1, _pose(0, 0), .9), _dt(1, _pose(0, 0), .8), _dt(2, _pose(0, 0), .7)]),
        "bbox": ([_gt(1, 1, np.zeros((17, 3)), bbox=(100, 100, 50, 80), area=4000.0), _gt(2, 1, _pose(0, 0))], [_dt(1, inside, .9), _dt(1, _pose(0, 0), .3)]),
        "trunc": ([_gt(1, 1, _pose(0, 0))], [_dt(1, _pose(300, 300), 1.0 - k / 100) for k in range(25)] + [_dt(1, _pose(0, 0), .1)]),
        "ties": ([_gt(1, 1, _pose(0, 0)), _gt(2, 2, _pose(0, 0))], [_dt(2, _pose(300, 300), -0.0), _dt(1, _pose(0, 0), 0.0), _dt(2, _pose(0, 0), 0.0)]),
    }
    gts, dts = sets[case]
    ds = {"images": [{"id": 1}, {"id": 2}], "annotations": gts}
    E = COCOevalKps(ds, dts).run()
    gtn, dtn = coco_eval.pack_gt(ds), coco_eval.pack_dt(dts, [1, 2])
    check_against(E, host_eval(gtn, dtn), gtn, dtn, 20)


def test_host_hook_equals_restatement_on_random_sets():
    rng = np.random.default_rng(17)
    done = skipped = dets = 0
    while done < 2000:
        n = int(rng.integers(1, 7))
        ds, res = random_set(rng, n)
        iou, rec, area = _thresholds(rng)
        max_det = int(rng.choice([1, 3, 5, 20]))
        try:
            E = COCOevalKps(ds, res, max_det=max_det, iou_thrs=iou, rec_thrs=rec, area_rng=area).run()
        except MarginError:
            skipped += 1
            continue
        gtn, dtn = coco_eval.pack_gt(ds), coco_eval.pack_dt(res, [im["id"] for im in ds["images"]])
        got = host_eval(gtn, dtn, max_det, iou, rec, area)
        check_against(E, got, gtn, dtn, max_det)
        if iou is coco_eval.IOU_THRS:
            assert np.array_equal(coco_eval.summarize(got["precision"], got["recall"], max_det=max_det), E.summarize())
        done += 1
        dets += len(res)
    assert skipped < done / 10
    assert dets > 5000


def test_packers_against_hand_built_dicts():
    ds = {"images": [{"id": 7}, {"id": 3}, {"id": 5}],
          "annotations": [_gt(10, 7, _pose(0, 0), crowd=1), _gt(11, 3, _pose(1, 1), area=5.5), _gt(12, 7, np.zeros((17, 3)), nk=0),
                          _gt(13, 7, _pose(2, 2), nk=0), dict(_gt(14, 7, _pose(0, 0)), category_id=2)]}
    g = coco_eval.pack_gt(ds)
    assert g["img_ids"].tolist() == [3, 5, 7] and g["count"].tolist() == [1, 0, 3]
    assert g["keypoints"].shape == (3, 3, 17, 3) and g["keypoints"][0, 0, 1, 0] == 6.0
    assert g["area"][0, 0] == 5.5 and g["iscrowd"][2].tolist() == [1, 0, 0] and g["ignore"][2].tolist() == [1, 1, 1]
    assert g["ignore"][0].tolist() == [0, 0, 0] and g["bbox"][2, 0].tolist() == [0, 0, 100, 100]
    res = [_dt(5, _pose(0, 0), .3), _dt(9, _pose(0, 0), .9), _dt(5, _pose(1, 0), .4), _dt(3, _pose(0, 0), -0.0)]
    d = coco_eval.pack_dt(res, [5, 3, 3])
    assert d["img_ids"].tolist() == [3, 5] and d["count"].tolist() == [1, 2]       # image 9 is dropped
    assert d["score"][1].tolist() == [.3, .4] and np.signbit(d["score"][0, 0]) and d["keypoints"][1, 1, 0, 0] == 1.0
    both = coco_eval.concat_tables([coco_eval.pack_gt(ds, [3]), coco_eval.pack_gt(ds, [7])])
    assert both["count"].tolist() == [1, 3] and both["keypoints"].shape == (2, 3, 17, 3)
    assert np.array_equal(both["keypoints"][1], g["keypoints"][2]) and (both["keypoints"][0, 1:] == 0).all()


def test_stats_equal_the_restatement():
    rng = np.random.default_rng(3)
    for _ in range(20):
        ds, res = random_set(rng, 12)
        try:
            E = COCOevalKps(ds, res).run()
        except MarginError:
            continue
        p, r, _ = E.arrays()
        assert np.array_equal(coco_eval.summarize(p, r), E.summarize())


def test_argument_errors():
    ds, res = random_set(np.random.default_rng(1), 3)
    gtn, dtn = coco_eval.pack_gt(ds), coco_eval.pack_dt(res, [im["id"] for im in ds["images"]])
    assert host_eval(gtn, dtn)["recall"].shape == (10, 3)
    bad_sets = [dict(max_det=0), dict(max_det=_lib.COCO_LIMIT_DET + 1), dict(iou=np.linspace(.5, .95, 11)),
                dict(rec=np.zeros(0)), dict(rec=np.zeros(_lib.COCO_LIMIT_REC + 1)), dict(area=np.zeros((0, 2)))]
    for bad in bad_sets:
        with pytest.raises(_lib.EkpError) as e:
            host_eval(gtn, dtn, **bad)
        assert e.value.code == _lib.ERR_ARG, bad
    big = dict(gtn, keypoints=np.zeros((3, _lib.COCO_LIMIT_GT + 1, 17, 3)))
    with pytest.raises(_lib.EkpError):
        host_eval(big, dtn)
    assert _lib.lib.ekp_coco_eval_workspace_bytes(0, 1, 1, 20, 3, 10) == 0
    assert _lib.lib.ekp_coco_eval_workspace_bytes(10, 1, 1, 20, 3, 11) == 0
    assert _lib.lib.ekp_coco_eval_workspace_bytes(10, 1, 1, 20, 3, 10) > 0
    g = _lib.CocoGt(*([None] * 6))
    d = _lib.CocoDt(*([None] * 3))
    o = _lib.CocoEvalOut(*([None] * 6))
    assert _lib.lib.ekp_debug_coco_eval_host(C.byref(g), 1, C.byref(d), 1, 1, 20, None, 10, None, 101, None, 3, C.byref(o)) == _lib.ERR_ARG
    assert _lib.lib.ekp_debug_coco_eval_host(None, 1, None, 1, 1, 20, None, 10, None, 101, None, 3, None) == _lib.ERR_ARG
    arr = np.zeros(64)
    misaligned = _lib.CocoEvalOut(arr.ctypes.data + 4, arr.ctypes.data, arr.ctypes.data, None, None, None)
    assert _lib.lib.ekp_coco_eval_kpts(None, C.byref(g), 1, C.byref(d), 1, 1, 20, None, 10, None, 101, None, 3, None,
                                       C.byref(misaligned), None) == _lib.ERR_ARG


# ---- GPU ----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


def _dev_tables(torch, gtn, dtn):
    return coco_eval._upload({k: gtn[k] for k in coco_eval.GT_FIELDS}, 0), coco_eval._upload({k: dtn[k] for k in coco_eval.DT_FIELDS}, 0)


def device_eval(torch, gt, dt, max_det=20, iou=coco_eval.IOU_THRS, rec=coco_eval.REC_THRS, area=coco_eval.AREA_RNG,
                ws=None, stream=None, details=True):
    """ekp_coco_eval_kpts with every output (the optional ones too), starting dirty"""
    n, mg, md = int(gt["count"].shape[0]), int(gt["keypoints"].shape[1]), int(dt["keypoints"].shape[1])
    area = np.asarray(area, np.float64).reshape(-1, 2)
    T, R, A = len(iou), len(rec), len(area)
    dev = torch.device("cuda", 0)
    th = [coco_eval._thresholds(dev, x) for x in (iou, rec, area)]   # uploaded once per set
    nb = _lib.lib.ekp_coco_eval_workspace_bytes(n, mg, md, max_det, A, T)
    if ws is None:
        ws = torch.full((nb,), 0xA5, dtype=torch.uint8, device=dev)
    out = dict(precision=torch.full((T, R, A), float("nan"), dtype=torch.float64, device=dev),
               recall=torch.full((T, A), float("nan"), dtype=torch.float64, device=dev),
               scores=torch.full((T, R, A), float("nan"), dtype=torch.float64, device=dev))
    if details:
        out.update(dt_match=torch.full((n, A, T, max_det), 77, dtype=torch.int32, device=dev),
                   dt_ignore=torch.full((n, A, T, max_det), 77, dtype=torch.int32, device=dev),
                   oks=torch.full((n, max_det, mg), float("nan"), dtype=torch.float64, device=dev))
    names = ("precision", "recall", "scores", "dt_match", "dt_ignore", "oks")
    o = _lib.CocoEvalOut(*(out[k].data_ptr() if k in out else None for k in names))
    ctx = coco_eval._context(0)
    st = stream.cuda_stream if stream is not None else torch.cuda.current_stream().cuda_stream
    _lib.check(_lib.lib.ekp_coco_eval_kpts(ctx._ctx, C.byref(_lib.CocoGt(*(gt[k].data_ptr() for k in coco_eval.GT_FIELDS))), mg,
                                           C.byref(_lib.CocoDt(*(dt[k].data_ptr() for k in coco_eval.DT_FIELDS))), md, n, max_det,
                                           th[0].data_ptr(), T, th[1].data_ptr(), R, th[2].data_ptr(), A, ws.data_ptr(), C.byref(o), st))
    return out, ws


def _np(out, torch):
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


@pytest.mark.gpu
def test_device_equals_restatement_on_random_sets(torch):
    rng = np.random.default_rng(23)
    done = 0
    while done < 300:
        ds, res = random_set(rng, int(rng.integers(1, 12)))
        iou, rec, area = _thresholds(rng)
        max_det = int(rng.choice([1, 3, 5, 20]))
        try:
            E = COCOevalKps(ds, res, max_det=max_det, iou_thrs=iou, rec_thrs=rec, area_rng=area).run()
        except MarginError:
            continue
        gtn, dtn = coco_eval.pack_gt(ds), coco_eval.pack_dt(res, [im["id"] for im in ds["images"]])
        out, _ = device_eval(torch, *_dev_tables(torch, gtn, dtn), max_det, iou, rec, area)
        check_against(E, _np(out, torch), gtn, dtn, max_det)
        done += 1


def _big_set(rng, n_img, max_people=20):
    """COCO-val-like: up to 20 gts and 20 dts per image, integer-free coordinates (ties only from equal scores)"""
    gtn = dict(count=rng.integers(0, max_people + 1, n_img).astype(np.int32), keypoints=np.zeros((n_img, max_people, 17, 3)),
               bbox=np.zeros((n_img, max_people, 4)), area=rng.uniform(100, 40000, (n_img, max_people)),
               iscrowd=(rng.random((n_img, max_people)) < 0.03).astype(np.int32))
    cx, cy = rng.uniform(0, 600, (n_img, max_people, 1)), rng.uniform(0, 400, (n_img, max_people, 1))
    s = np.sqrt(gtn["area"])[..., None]
    gtn["keypoints"][..., 0] = cx + rng.uniform(-.5, .5, (n_img, max_people, 17)) * s
    gtn["keypoints"][..., 1] = cy + rng.uniform(-.5, .5, (n_img, max_people, 17)) * s
    gtn["keypoints"][..., 2] = np.where(rng.random((n_img, max_people, 17)) < 0.8, 2, 0)
    gtn["bbox"][..., 0], gtn["bbox"][..., 1] = cx[..., 0] - s[..., 0] / 2, cy[..., 0] - s[..., 0] / 2
    gtn["bbox"][..., 2] = gtn["bbox"][..., 3] = s[..., 0]
    gtn["ignore"] = (gtn["iscrowd"] | ((gtn["keypoints"][..., 2] > 0).sum(-1) == 0)).astype(np.int32)
    dtn = dict(count=rng.integers(0, max_people + 1, n_img).astype(np.int32),
               keypoints=gtn["keypoints"] + rng.normal(0, 1, (n_img, max_people, 17, 3)) * rng.uniform(0.5, 30, (n_img, max_people, 1, 1)),
               score=np.round(rng.random((n_img, max_people)), 3))
    dtn["keypoints"][..., 2] = 1
    return gtn, dtn


def _tables_to_coco(gtn, dtn):
    ds = {"images": [{"id": i + 1} for i in range(len(gtn["count"]))], "annotations": []}
    res, aid = [], 1
    for i in range(len(gtn["count"])):
        for g in range(gtn["count"][i]):
            ds["annotations"].append({"id": aid, "image_id": i + 1, "category_id": 1, "keypoints": gtn["keypoints"][i, g].reshape(-1).tolist(),
                                      "num_keypoints": int((gtn["keypoints"][i, g, :, 2] > 0).sum()), "bbox": gtn["bbox"][i, g].tolist(),
                                      "area": float(gtn["area"][i, g]), "iscrowd": int(gtn["iscrowd"][i, g])})
            aid += 1
        for d in range(dtn["count"][i]):
            res.append({"image_id": i + 1, "category_id": 1, "keypoints": dtn["keypoints"][i, d].reshape(-1).tolist(),
                        "score": float(dtn["score"][i, d])})
    return ds, res


@pytest.mark.gpu
@pytest.mark.parametrize("n_img,max_det", [(5000, 20), (102, 20), (103, 20), (26, 20), (25, 20), (2048, 1), (2049, 1),
                                           (4097, 1), (512, 1), (513, 1)])
def test_device_coco_val_sized_and_boundaries(torch, n_img, max_det):
    """5,000 images of up to 20 people (about 100k sorted detections), and slot counts n_img x max_det on both sides of a
    2048-key sort tile and a 512-position accumulate chunk; checked against the host hook (itself pinned to the
    restatement above) and, on the small sets, against the restatement"""
    rng = np.random.default_rng(n_img)
    gtn, dtn = _big_set(rng, n_img)
    out, _ = device_eval(torch, *_dev_tables(torch, gtn, dtn), max_det, details=n_img <= 1000)
    got = _np(out, torch)
    host = host_eval(gtn, dtn, max_det)
    for k in ("precision", "recall", "scores"):
        assert np.array_equal(got[k].view(np.uint64), host[k].view(np.uint64)), k
    if n_img <= 1000:
        assert np.array_equal(got["dt_match"], host["dt_match"]) and np.array_equal(got["dt_ignore"], host["dt_ignore"])
        assert np.allclose(got["oks"], host["oks"], rtol=0, atol=1e-12)
    if n_img <= 200:
        ds, res = _tables_to_coco(gtn, dtn)
        try:
            E = COCOevalKps(ds, res, max_det=max_det).run()
        except MarginError:
            return
        p, r, s = E.arrays()
        assert np.array_equal(got["precision"], p) and np.array_equal(got["recall"], r) and np.array_equal(got["scores"], s)


@pytest.mark.gpu
def test_workspace_reuse_dirty_outputs_streams_no_wait_launches(torch):
    rng = np.random.default_rng(5)
    gtn, dtn = _big_set(rng, 300)
    gt, dt = _dev_tables(torch, gtn, dtn)
    want = host_eval(gtn, dtn)
    gtn2, dtn2 = _big_set(rng, 300)
    gt2, dt2 = _dev_tables(torch, gtn2, dtn2)
    want2 = host_eval(gtn2, dtn2)
    ctx = coco_eval._context(0)
    out, ws = device_eval(torch, gt, dt, details=False)
    got = _np(out, torch)
    assert np.array_equal(got["precision"], want["precision"])
    # the same workspace for another set, on a side stream behind a device sleep: no host wait, ordered on that stream
    side = torch.cuda.Stream()
    k0 = ctx.kernel_launches()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)
        out2, _ = device_eval(torch, gt2, dt2, ws=ws, stream=side, details=False)
        ev = torch.cuda.Event()
        ev.record(side)
    assert not ev.query(), "the evaluation waited for the device"
    assert ctx.kernel_launches() == k0 + 29
    side.synchronize()
    got2 = {k: v.cpu().numpy() for k, v in out2.items()}
    for k in ("precision", "recall", "scores"):
        assert np.array_equal(got2[k].view(np.uint64), want2[k].view(np.uint64)), k
    # evaluate_keypoints: no wait after the thresholds' first upload
    e1 = coco_eval.evaluate_keypoints(gt, dt)
    e1.synchronize()
    torch.cuda._sleep(200_000_000)
    e2 = coco_eval.evaluate_keypoints(gt, dt)
    assert not e2.event.query()
    assert np.array_equal(e2.precision.cpu().numpy(), want["precision"])
    assert np.array_equal(e2.stats(), coco_eval.summarize(want["precision"], want["recall"]))


@pytest.mark.gpu
def test_dt_tables_from_results_equal_coco_keypoints(torch):
    import torch_ekpose_b200 as ek
    from torch_ekpose_b200 import coco, synthetic
    heat, paf = synthetic.make_batch(6, 46, 54, (1, 6), seed=4)
    pp = ek.PostProcessor(device=0, max_batch=6, max_h=46, max_w=54, max_peaks=512, max_humans=16)
    pp.run(torch.from_numpy(heat).cuda(), torch.from_numpy(paf).cuda())
    tabs = pp.result_tensors()
    num, parts, scores = pp.human_tables()
    ups = np.array([[480, 640], [427, 640], [500, 375], [640, 480], [333, 500], [612, 612]], np.float64)
    want = coco.coco_keypoints(num, parts, (368, 432), ups)
    for sc in (None, tabs["scores"]):
        dt = coco_eval.dt_tables_from_results(tabs, (368, 432), ups, scores=sc)
        kp, s, cnt = dt["keypoints"].cpu().numpy(), dt["score"].cpu().numpy(), dt["count"].cpu().numpy()
        assert cnt.tolist() == num.tolist()
        for i in range(6):
            assert np.array_equal(kp[i, :num[i]].reshape(num[i], 51).view(np.uint64), want[i].view(np.uint64)), i
            assert (s[i, :num[i]] == (1.0 if sc is None else scores[i, :num[i]].astype(np.float64))).all()


def _truth_gt(truths, img_ids, map_hw, ups):
    """COCO ground truth of synthetic people: keypoint j = the joint ORDER_COCO[j], mapped like coco_keypoints maps a
    found part (x / W * up_w + 0.5 in the full-resolution map's pixels, x 8 of the stride-8 map), visibility 2 when it
    lies inside the map, else 0; bbox = the visible keypoints' box; area = bbox area x 0.8 (a person's segment covers
    about that share of its box)"""
    H, W = map_hw
    ds = {"images": [{"id": int(i)} for i in img_ids], "annotations": []}
    aid = 1
    for img, tr, up in zip(img_ids, truths, ups):
        for person in tr:
            xy = person[ORDER_COCO] * 8.0
            kp = np.zeros((17, 3))
            kp[:, 0] = xy[:, 0] / W * up[1] + 0.5
            kp[:, 1] = xy[:, 1] / H * up[0] + 0.5
            vis = (xy[:, 0] >= 0) & (xy[:, 0] < W) & (xy[:, 1] >= 0) & (xy[:, 1] < H)
            kp[:, 2] = np.where(vis, 2, 0)
            kp[~vis, :2] = 0
            v = kp[vis]
            bb = [v[:, 0].min(), v[:, 1].min(), v[:, 0].max() - v[:, 0].min(), v[:, 1].max() - v[:, 1].min()] if len(v) else [0, 0, 0, 0]
            ds["annotations"].append({"id": aid, "image_id": int(img), "category_id": 1, "keypoints": kp.reshape(-1).tolist(),
                                      "num_keypoints": int(vis.sum()), "bbox": bb, "area": bb[2] * bb[3] * 0.8, "iscrowd": 0})
            aid += 1
    return ds


@pytest.mark.gpu
@pytest.mark.parametrize("frontend", ["reference", "dense"])
def test_end_to_end_synthetic_ap(torch, frontend):
    """Seeded 368x432 scenes through run -> result_tensors -> dt_tables_from_results -> evaluate_keypoints (two batches
    concatenated): stats() equal the restatement's on the host results, and the pipeline finds the synthetic people"""
    import torch_ekpose_b200 as ek
    from torch_ekpose_b200 import coco
    from torch_ekpose_b200 import synthetic
    ups = [np.array([480, 640], np.float64), np.array([368, 432], np.float64)]
    pp = ek.PostProcessor(device=0, max_batch=16, max_h=46, max_w=54, max_peaks=512, max_humans=32)
    pp.set_host_copy(False)
    dts, results, truths, ids, upl = [], [], [], [], []
    for b in range(2):
        heat, paf, tr = synthetic.make_batch(16, 46, 54, (1, 6), seed=40 + b, return_truth=True)
        pp.run(torch.from_numpy(heat).cuda(), torch.from_numpy(paf).cuda(), frontend=frontend)
        tabs = pp.result_tensors()
        dts.append(coco_eval.dt_tables_from_results(tabs, (368, 432), ups[b], scores=tabs["scores"]))
        num, parts, scores = pp.human_tables()
        img = list(range(100 * b + 1, 100 * b + 17))
        for i, kps in enumerate(coco.coco_keypoints(num, parts, (368, 432), ups[b])):
            for k, row in enumerate(kps):
                results.append({"image_id": img[i], "category_id": 1, "keypoints": list(row), "score": float(scores[i, k])})
        truths += tr
        ids += img
        upl += [ups[b]] * 16
    ds = _truth_gt(truths, ids, (368, 432), upl)
    gt = coco_eval.gt_tables(ds)
    dt = coco_eval.concat_tables(dts)
    ev = coco_eval.evaluate_keypoints(gt, dt)
    st = ev.stats()
    E = COCOevalKps(ds, results, check_margin=False).run()
    assert np.array_equal(ev.precision.cpu().numpy(), E.arrays()[0])
    assert np.array_equal(st, E.summarize()), (st, E.summarize())
    # and through the result-list front-end
    ev2 = coco_eval.evaluate_keypoints(gt, coco_eval.dt_tables(results, gt["img_ids"]))
    assert np.array_equal(ev2.stats(), st)
    assert st[1] > 0.5, st    # AP at OKS 0.5: the pipeline finds the people it was given
