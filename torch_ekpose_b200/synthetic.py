"""Seeded synthetic stride-8 heat / PAF tensors (the bench and parity-test workload).

There is no dataset or checkpoint available offline, so the benchmark and the parity
tests run on synthetic network outputs of the shapes BASELINE.json names.  The recipe is
SURVEY.md Appendix F: people are placed from an 18-joint template, heat-maps are Gaussian
blobs (sigma 7 px at stride 8, as the reference's ground-truth synthesis does in
lib/datasets/heatmap.py:11-33), PAFs are unit limb vectors inside a 1-cell-wide band
around each limb (lib/datasets/paf.py:11-63) in the channel order of
lib/pafprocess/pafprocess.h:16-24, plus Gaussian noise.

Everything here is NumPy on the host: it only produces INPUTS.
"""
from __future__ import annotations

import numpy as np

# lib/pafprocess/pafprocess.h:16-24
COCOPAIRS_NET = ((12, 13), (20, 21), (14, 15), (16, 17), (22, 23), (24, 25), (0, 1), (2, 3), (4, 5), (6, 7),
                 (8, 9), (10, 11), (28, 29), (30, 31), (34, 35), (32, 33), (36, 37), (18, 19), (26, 27))
COCOPAIRS = ((1, 2), (1, 5), (2, 3), (3, 4), (5, 6), (6, 7), (1, 8), (8, 9), (9, 10), (1, 11),
             (11, 12), (12, 13), (1, 0), (0, 14), (14, 16), (0, 15), (15, 17), (2, 16), (5, 17))

# unit-box joint template in the reference part order (lib/utils/common.py:6-25)
_TPL = np.array([(.50, .08), (.50, .20), (.35, .20), (.30, .38), (.28, .55), (.65, .20), (.70, .38), (.72, .55),
                 (.42, .55), (.41, .75), (.40, .95), (.58, .55), (.59, .75), (.60, .95), (.46, .05), (.54, .05),
                 (.41, .07), (.59, .07)], dtype=np.float64)

# named shapes of BASELINE.json configs: stride-8 (h, w)
SHAPES = {"368x432": (46, 54), "656x368": (46, 82), "1312x736": (92, 164)}


def make_scene(h: int, w: int, people: int, seed: int, noise: bool = True, return_truth: bool = False):
    """One image: returns (heat[h,w,19], paf[h,w,38]) float32, HWC like estimator.get_outputs.  return_truth=True adds
    a third item, truth float64 [people, 18, 2]: every person's 18 joints (x, y) in reference part order, in the
    stride-8 map's pixels (the centres of the heat blobs)."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)
    heat = np.zeros((h, w, 19), np.float64)
    paf = np.zeros((h, w, 38), np.float64)
    truth = np.zeros((people, 18, 2), np.float64)
    for person in range(people):
        s = rng.uniform(0.35, 0.7) * h
        cx = rng.uniform(0.1, 0.9) * w
        cy = rng.uniform(0.05, 0.4) * h
        kp = _TPL * np.array([0.6 * s, s]) + np.array([cx - 0.3 * s, cy]) + rng.normal(0, 0.3, (18, 2))
        truth[person] = kp
        amp = rng.uniform(0.6, 1.0, 18)
        for k in range(18):
            d2 = (xx - kp[k, 0]) ** 2 + (yy - kp[k, 1]) ** 2
            heat[:, :, k] = np.maximum(heat[:, :, k], amp[k] * np.exp(-d2 / (2 * 0.875 ** 2)))
        for limb, (a, b) in enumerate(COCOPAIRS):
            v = kp[b] - kp[a]
            n = np.hypot(v[0], v[1])
            if n < 1e-6:
                continue
            u = v / n
            rx, ry = xx - kp[a, 0], yy - kp[a, 1]
            t = rx * u[0] + ry * u[1]
            d = np.abs(rx * u[1] - ry * u[0])
            m = (t >= -1) & (t <= n + 1) & (d < 1)
            c1, c2 = COCOPAIRS_NET[limb]
            paf[:, :, c1][m] = u[0]
            paf[:, :, c2][m] = u[1]
    if noise:
        heat[:, :, :18] += rng.normal(0, 0.005, (h, w, 18))
        paf += rng.normal(0, 0.01, (h, w, 38))
    heat[:, :, 18] = np.maximum(1 - heat[:, :, :18].max(axis=2), 0)
    if return_truth:
        return heat.astype(np.float32), paf.astype(np.float32), truth
    return heat.astype(np.float32), paf.astype(np.float32)


def make_batch(batch: int, h: int, w: int, people_range=(1, 6), seed: int = 0, layout: str = "nchw",
               return_truth: bool = False):
    """A batch of scenes.  layout 'nchw' (what the network emits, vgg2016.py:105) or 'nhwc'.

    Scene i uses seed `1000*seed + i` and people count cycling through people_range inclusive.
    Returns (heat, paf) float32 arrays; return_truth=True adds the list of the scenes' truth arrays (make_scene).
    """
    lo, hi = people_range
    heats, pafs, truths = [], [], []
    for i in range(batch):
        p = lo + (i % (hi - lo + 1))
        scene = make_scene(h, w, p, 1000 * seed + i, return_truth=return_truth)
        heats.append(scene[0])
        pafs.append(scene[1])
        truths.append(scene[2] if return_truth else None)
    heat = np.stack(heats)
    paf = np.stack(pafs)
    if layout == "nchw":
        heat = np.ascontiguousarray(heat.transpose(0, 3, 1, 2))
        paf = np.ascontiguousarray(paf.transpose(0, 3, 1, 2))
    elif layout != "nhwc":
        raise ValueError("layout must be 'nchw' or 'nhwc'")
    if return_truth:
        return heat, paf, truths
    return heat, paf
