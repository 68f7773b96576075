"""Every context capacity and every stage 4-5 size threshold, run at its exact edge and one past it, against the oracle.

A scene that does not fit a context is reported (an EKP_OVF_* bit on that image, EkpCapacityError from results()), never
silently cut, and a scene that fits exactly is computed in full.  Off-by-one errors live exactly at the edge, so every
capacity gets two runs here: the count equal to the capacity (no overflow, peaks / people bit for bit equal to the oracle)
and the count one past it (the right bit on that image only, results() raises).  The image at the edge sits in a batch
between clean images, and each batch runs in two orders: a write one slot past an image's slice of the context's tables
lands in its neighbour, whose results must still equal the oracle.  Branches that depend on a count (connections per limb,
tied candidates, staged vs unstaged connection records, process_paf's three upload routes) are run on either side of
their threshold; every case asserts its own precondition (peak, candidate, connection or sample count) from the oracle or
from the construction, so a changed scene fails instead of quietly leaving the edge.

Shared-memory limits are raised per context and kernel attributes are process-wide, so the cases run in fresh worker
processes (one per group; contexts within a group are created in increasing size), as in test_launch_variants.py.  The
worker writes its results to an .npz; the oracle runs here, on the CPU.  test_thresholds_are_the_ones_the_cases_sit_on
(no GPU) reads the thresholds from the sources, so that a changed constant fails loudly instead of dropping coverage."""
import functools
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import oracle
from tests import util
from tests.util import assert_bits_equal

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# the thresholds the cases are built around (pinned to the sources by test_thresholds_are_the_ones_the_cases_sit_on)
LIMITS = dict(max_peaks=16384, max_humans=1024, max_part=1024, max_cand=8192)   # EKP_LIMIT_*
SMALL_PEAKS, SMALL_MAX_SAMPLES, LISTED_MAX_SAMPLES = 512, 16384, 64 * 1024      # process_paf.cu
CONN_CAP_MIN, CONN_CAP_MAX = 64, 1536                                           # assemble_conn_cap's clamp
ONE_MAX_PEAKS = 4096                                                            # peaks_sort.cu kOneMaxPeaks
SORT_SLICE = 256                                                                # peaks_sort.cu kSortThreads
OVF_PEAKS, OVF_PART, OVF_CAND, OVF_HUMANS = 1, 2, 4, 8

# pafprocess.h:16-24: the parts of each limb and its x channel (y = x + 1)
LIMB_PARTS = [(1, 2), (1, 5), (2, 3), (3, 4), (5, 6), (6, 7), (1, 8), (8, 9), (9, 10), (1, 11), (11, 12), (12, 13), (1, 0),
              (0, 14), (14, 16), (0, 15), (15, 17), (2, 16), (5, 17)]
LIMB_CH = [12, 20, 14, 16, 22, 24, 0, 2, 4, 6, 8, 10, 28, 30, 34, 32, 36, 18, 26]
CHAIN_H1 = 16     # heat height for chain scenes: a pair 8 px apart has no penalty, a longer one a large one
TIED_H1 = 4096    # ... and for tied scenes: no pair is penalised, so every horizontal pair scores exactly 1.0


def conn_cap(max_humans, max_part):
    """assemble_conn_cap: connections of one image staged in shared memory"""
    return int(min(max(min(24 * max_humans, 19 * max_part), CONN_CAP_MIN), CONN_CAP_MAX))


def _cdiv(a, b):
    return -(-a // b)


# ---- scenes ------------------------------------------------------------------------------------------------------------
# A scene is (rows, bands): peak rows (x, y, score, 0, part) and PAF bands (channel, y0, y1, x0, x1, value) to paint.
def _chain(n, cols, y_top, seed):
    """n four-part people (neck, RShoulder, RElbow, RWrist in a row, 8 px apart) on a grid of `cols` columns of 40 x 6 px
    cells; limbs 0, 2, 3 run along x-channel bands 3 px tall.  With h1 = CHAIN_H1 every person's three pairs score exactly
    1.0 and any other passing pair less, so the people are the rows, one connection per limb each."""
    rng = np.random.default_rng(seed)
    rows, bands = [], []
    for k in range(n):
        x0, y = 8 + 40 * (k % cols), y_top + 6 * (k // cols)
        for j, part in enumerate((1, 2, 3, 4)):
            rows.append((x0 + 8 * j, y, 0.5 + 0.4 * rng.random(), 0, part))
        bands += [(c, y - 1, y + 2, x0 - 1, x0 + 26, 1.0) for c in (12, 14, 16)]
    return rows, bands


def _chain_size(n, cols):
    return 6 * _cdiv(n, cols) + 4, 40 * cols + 16


def _tied(n_a, n_b, y, limb=0, arms=True, x_start=2):
    """n_a peaks of the limb's first part left of n_b of its second on ONE row under an x-channel of 1: all n_a x n_b pairs
    pass and (h1 = TIED_H1) all score exactly 1.0, so the sort replays libstdc++'s introsort on ties only.  arms: every
    second-part peak (RShoulder) gets its own RElbow and RWrist below it, so each accepted pair becomes a four-part person
    and the subset shows which pairs the greedy step took."""
    pa, pb = LIMB_PARTS[limb]
    xa = [x_start + 2 * i for i in range(n_a)]
    xb = [x_start + 2 * n_a + 6 + 2 * j for j in range(n_b)]
    rows = [(x, y, 0.6 + 0.01 * (i % 7), 0, pa) for i, x in enumerate(xa)]
    rows += [(x, y, 0.7 + 0.01 * (j % 5), 0, pb) for j, x in enumerate(xb)]
    bands = [(LIMB_CH[limb], y - 1, y + 2, 0, xb[-1] + 2, 1.0)]
    if arms:
        for j, x in enumerate(xb):
            rows += [(x, y + 8, 0.8, 0, 3), (x, y + 16, 0.9, 0, 4)]
            bands += [(15, y, y + 9, x, x + 1, 1.0), (17, y + 8, y + 17, x, x + 1, 1.0)]
    return rows, bands


def _clutter(counts, y0, y1, W, seed):
    """counts {part: n} peaks at random positions in rows [y0, y1) (where no band is painted)"""
    rng = np.random.default_rng(seed)
    return [(int(rng.integers(0, W)), int(rng.integers(y0, y1)), 0.25 + 0.5 * rng.random(), 0, p)
            for p, n in sorted(counts.items()) for _ in range(n)]


def _paint(H, W, bands):
    paf = np.zeros((H, W, 38), np.float32)
    for c, y0, y1, x0, x1, v in bands:
        paf[max(y0, 0):y1, max(x0, 0):x1, c] = v
    return paf


def _peak_batch(scenes, H, W, shared_paf=None):
    """run_peaks inputs: scenes [(rows, bands)] on H x W maps (or one PAF shared by all images)"""
    counts = np.array([len(r) for r, _ in scenes], np.int32)
    peaks = np.zeros((len(scenes), max(counts.max(), 1), 5), np.float32)
    rng = np.random.default_rng(int(counts.sum()))
    for i, (r, _) in enumerate(scenes):
        a = np.array(r, np.float32).reshape(-1, 5)
        peaks[i, :len(a)] = a[rng.permutation(len(a))]   # unsorted input on purpose
    paf = shared_paf[None] if shared_paf is not None else np.stack([_paint(H, W, b) for _, b in scenes])
    return dict(peaks=peaks, counts=counts, paf=paf)


def _spikes(h, w, n, seed):
    """a heat map with exactly n peaks for every front-end: isolated asymmetric spikes (one maximum each after the dense
    smoothing, the reference NMS and its refinement) on a 4-cell grid of all 18 parts"""
    rng = np.random.default_rng(seed)
    heat = np.zeros((h, w, 19), np.float32)
    cells = [(y, x, p) for p in range(18) for y in range(1, h - 2, 4) for x in range(1, w - 2, 4)]
    assert n <= len(cells)
    for i in rng.permutation(len(cells))[:n]:
        y, x, p = cells[i]
        v = np.float32(rng.uniform(0.5, 1.0))
        heat[y, x, p], heat[y, x + 1, p], heat[y + 1, x, p] = v, 0.7 * v, 0.6 * v
    return heat


# ---- the cases -------------------------------------------------------------------------------------------------------
# front-end kernels that append peaks: (name, layout, frontend, materialize, h, w, peaks of the edge image, kernel)
FRONTENDS = [("dense_plane", "nchw", "dense", False, 46, 54, 256, r"dense_plane_kernel\("),
             ("dense_plane_sliced", "nchw", "dense", False, 46, 54, 257, r"dense_plane_kernel\("),
             ("dense_tiled_nhwc", "nhwc", "dense", False, 46, 54, 512, r"dense_frontend_kernel<false, false"),
             ("dense_materialize", "nchw", "dense", True, 46, 54, 513, r"dense_frontend_kernel<true, false"),
             ("ref_scan_plane", "nchw", "reference", False, 46, 54, 256, r"ref_scan_kernel<true>"),
             ("ref_scan_generic", "nchw", "reference", False, 40, 300, 513, r"ref_scan_kernel<false>"),
             ("reference_gauss", "nchw", "reference_gauss", False, 46, 54, 512, r"ref_refine_kernel<true>")]


def _frontend_batch(name):
    """image 0: the edge image (exactly N peaks); the others: clean images with N / 2 peaks"""
    _, layout, _, _, h, w, npk, _ = next(f for f in FRONTENDS if f[0] == name)
    n = _unsliced_batch() if name == "dense_plane" else 3
    rng = np.random.default_rng(npk + h)
    heat = np.stack([_spikes(h, w, npk if i == 0 else npk // 2, 10 * i + npk) for i in range(n)])
    paf = rng.normal(0, 0.5, (n, h, w, 38)).astype(np.float32)
    if layout == "nchw":
        heat, paf = heat.transpose(0, 3, 1, 2), paf.transpose(0, 3, 1, 2)
    return dict(heat=np.ascontiguousarray(heat), paf=np.ascontiguousarray(paf))


def _unsliced_batch():
    """the smallest batch the dense plane kernel runs unsliced (18 n >= SMs), at least 8 images"""
    import torch
    return max(8, _cdiv(torch.cuda.get_device_properties(0).multi_processor_count, 18))


def _orders(n):
    """the edge image (0) second, then second to last; the clean images around it in forward, then reverse order"""
    clean = list(range(1, n))
    rev = clean[::-1]
    return [[clean[0], 0] + clean[1:], rev[:-1] + [0] + rev[-1:]]


# stage 4-5 cases: name -> (ctx, h1, scene builder, flag of the edge image); built on demand
def _stage45_cases():
    C = {}
    # run_peaks with exactly max_peaks input rows (peaks_ingest_kernel, one and two 256-peak sort slices) and one more
    for cap in (256, 513):
        def ingest(total, cap=cap):
            people, bands = _chain(20, 8, 4, cap)
            H, W = _chain_size(20, 8)
            rows = people + _clutter({7: (total - 80) // 2, 10: total - 80 - (total - 80) // 2}, H, H + 20, W, total)
            return [(rows, bands), _chain(10, 8, 4, 1), _chain(12, 8, 4, 2)], H + 20, W
        C[f"ingest_{cap}_at"] = (dict(max_peaks=cap, max_humans=64), CHAIN_H1, functools.partial(ingest, cap), 0, dict(peaks=cap))
        C[f"ingest_{cap}_over"] = (dict(max_peaks=cap - 1, max_humans=64), CHAIN_H1, functools.partial(ingest, cap), OVF_PEAKS,
                                   dict(peaks=cap))
    # max_part: part 2 (RShoulder) is B of limb 0 and A of limb 2
    for cap in (33, 64):
        def part(n, cap=cap):
            H, W = _chain_size(n, 8)
            return [_chain(n, 8, 4, cap), _chain(10, 8, 4, 3), _chain(cap // 2, 8, 4, 4)], H, W
        ctx = dict(max_peaks=512, max_humans=128, max_part=cap)
        C[f"part_{cap}_at"] = (ctx, CHAIN_H1, functools.partial(part, cap), 0, dict(people=cap))
        C[f"part_{cap}_over"] = (ctx, CHAIN_H1, functools.partial(part, cap + 1), OVF_PART, dict(people=cap + 1))
    # max_cand at the minimum and at the bench value, every candidate tied
    for cap, at, over in ((64, (8, 8), (5, 13)), (512, (16, 32), (19, 27))):
        def cand(ab):
            return [_tied(*ab, 4), _tied(4, 4, 4), _tied(3, 6, 4)], 24, 2 * sum(ab) + 16
        ctx = dict(max_peaks=512, max_humans=128, max_cand=cap)
        C[f"cand_{cap}_at"] = (ctx, TIED_H1, functools.partial(cand, at), 0, dict(tied=at[0] * at[1]))
        C[f"cand_{cap}_over"] = (ctx, TIED_H1, functools.partial(cand, over), OVF_CAND, dict(tied=over[0] * over[1]))
    # max_humans: rows before the prune; the row buffer holds max(max_humans, 32) rows
    for cap in (1, 31, 32, 33, 128, 129):
        def humans(n, cap=cap):
            H, W = _chain_size(max(n, 1), 8)
            return [_chain(n, 8, 4, cap), _chain(_cdiv(cap, 2), 8, 4, 5), _chain(cap, 8, 4, 6)], H, W
        ctx = dict(max_peaks=1024, max_humans=cap)
        C[f"humans_{cap}_at"] = (ctx, CHAIN_H1, functools.partial(humans, cap), 0, dict(people=cap))
        C[f"humans_{cap}_over"] = (ctx, CHAIN_H1, functools.partial(humans, cap + 1), OVF_HUMANS, dict(people=cap + 1))

    def pruned():   # 20 people + 13 neck-shoulder pairs: 33 rows before the prune, 20 people after it
        rows, bands = _chain(33, 8, 4, 7)
        rows = [r for k, r in enumerate(rows) if k < 80 or r[4] in (1, 2)]
        H, W = _chain_size(33, 8)
        return [(rows, bands), _chain(16, 8, 4, 8), _chain(32, 8, 4, 9)], H, W
    C["humans_32_rows_over_people_fit"] = (dict(max_peaks=1024, max_humans=32), CHAIN_H1, pruned, OVF_HUMANS, dict(people=20))
    # connections per limb around the register paths (<= 32, <= 64) and tied candidates around the parallel rank (16) and
    # the greedy step's 32-candidate chunks: no capacity is reached, every image equals the oracle
    C["conns_per_limb_32_33_64_65"] = (dict(max_peaks=512, max_humans=128), CHAIN_H1,
                                       lambda: ([_chain(n, 8, 4, n) for n in (32, 33, 64, 65)],) + _chain_size(65, 8), 0,
                                       dict(conns=[32, 33, 64, 65]))
    C["tied_16_17_32_33"] = (dict(max_peaks=512, max_humans=128), TIED_H1,
                             lambda: ([_tied(*ab, 4) for ab in ((4, 4), (1, 17), (4, 8), (3, 11))], 24, 64), 0,
                             dict(tied=[16, 17, 32, 33]))
    return C


STAGE45 = ["ingest_256_at", "ingest_256_over", "ingest_513_at", "ingest_513_over", "part_33_at", "part_33_over", "part_64_at",
           "part_64_over", "cand_64_at", "cand_64_over", "cand_512_at", "cand_512_over"] + \
          [f"humans_{c}_{k}" for c in (1, 31, 32, 33, 128, 129) for k in ("at", "over")] + \
          ["humans_32_rows_over_people_fit", "conns_per_limb_32_33_64_65", "tied_16_17_32_33"]


# total connections of one image at assemble_conn_cap (staged in shared memory) and one person past it (read from global
# memory): 512 and 513 four-part people, 3 connections each
CONN_CTX = dict(max_peaks=2304, max_humans=520, max_part=520)


def _conn_cap_scene(people):
    H, W = _chain_size(513, 32)
    return [_chain(people, 32, 4, people), _chain(100, 32, 4, 11), _chain(300, 32, 4, 12)], H, W


# one context at all four EKP_LIMIT_* values.  The edge scene sits at every limit at once: 1024 four-part people (1024
# peaks of each of parts 1-4, 1024 rows), 8192 candidates on limb 18 (64 LShoulders x 128 LEars on one row; limb 18 never
# starts a person), and clutter on 12 other parts up to 16384 peaks.  Each +1 variant moves exactly one count past its limit.
LIMIT_VARIANTS = {"at": 0, "peaks": OVF_PEAKS, "part": OVF_PART, "cand": OVF_CAND, "humans": OVF_HUMANS}
CLUTTER_PARTS = (0, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16)


@functools.lru_cache(maxsize=None)
def _limit_layout():
    people, bands = _chain(1024, 64, 4, 21)
    Hc, W = _chain_size(1024, 64)
    yt = Hc + 6
    tied, tb = _tied(64, 128, yt, limb=18, arms=False)
    extra_cand = [(4, yt + 12, 0.7, 0, 5), (12, yt + 12, 0.7, 0, 17)]
    extra_row = [(8, yt + 24, 0.7, 0, 0), (16, yt + 24, 0.7, 0, 14)]
    bands = bands + tb + [(26, yt + 11, yt + 14, 3, 14, 1.0), (30, yt + 23, yt + 26, 7, 18, 1.0)]
    return dict(people=people, tied=tied, extra_cand=extra_cand, extra_row=extra_row, H=yt + 30, W=W, Hc=Hc,
                paf=_paint(yt + 30, W, bands))


def _limit_scene(variant):
    L = _limit_layout()
    rows = L["people"] + L["tied"]
    if variant == "part":
        rows = rows + [(2, L["Hc"] - 1, 0.5, 0, 1)]   # a 1025th neck, in the clutter rows of no band
    if variant == "cand":
        rows = rows + L["extra_cand"]
    if variant == "humans":
        rows = rows + L["extra_row"]
    left = LIMITS["max_peaks"] + (variant == "peaks") - len(rows)
    counts = {p: left // len(CLUTTER_PARTS) + (k < left % len(CLUTTER_PARTS)) for k, p in enumerate(CLUTTER_PARTS)}
    return rows + _clutter(counts, 0, 3, L["W"], 22), []   # clutter in the rows above the first band (y < 3)


def _limit_batch(variant):
    L = _limit_layout()
    return _peak_batch([_limit_scene(variant), (L["people"][:200], []), (L["people"][:4 * 700], [])], L["H"], L["W"],
                       shared_paf=L["paf"])


# process_paf (the host operator surface): (name, peaks, limb pairs, route).  Routes: "small" = the zero-copy CUDA graph
# (npk <= SMALL_PEAKS and samples <= SMALL_MAX_SAMPLES), "listed" = the host lists the samples and uploads one block,
# "sparse" = pair_sample_offsets_kernel lists them.  Samples are 10 per pair, so the edges are at 1638 / 1639 and
# 6553 / 6554 pairs (16380 / 16390 and 65530 / 65540 samples).
PROCESS_PAF = [("pp_peaks_512", 512, None, "small"), ("pp_peaks_513", 513, None, "listed"),
               ("pp_pairs_1638", None, SMALL_MAX_SAMPLES // 10, "small"), ("pp_pairs_1639", None, SMALL_MAX_SAMPLES // 10 + 1, "listed"),
               ("pp_pairs_6553", None, LISTED_MAX_SAMPLES // 10, "listed"), ("pp_pairs_6554", None, LISTED_MAX_SAMPLES // 10 + 1, "sparse")]
PP_H1 = CHAIN_H1


def _pp_split(pairs):
    """(people, extra wrists, LKnees, LAnkles) with pairs = people * (3 people + wrists) + knees * ankles: chain people have
    3 people^2 pairs (limbs 0, 2, 3), extra wrists pair with every elbow, limb 11 (12 -> 13) is independent while part 11
    is empty; at most SMALL_PEAKS peaks in all"""
    for n in range(10, 41):
        for a in range(0, 60):
            r = pairs - n * (3 * n + a)
            if r < 0:
                break
            for d in range(0 if r == 0 else 1, 201):
                if (r == 0 and d == 0) or (d and r % d == 0 and r // d <= 200 and 4 * n + a + d + r // d <= SMALL_PEAKS):
                    return n, a, d, (r // d if d else 0)
    raise AssertionError(pairs)


def _pp_scene(name):
    _, npk, pairs, _ = next(p for p in PROCESS_PAF if p[0] == name)
    if npk is not None:
        n, a, d, e = 10, 0, 0, 0
    else:
        n, a, d, e = _pp_split(pairs)
    people, bands = _chain(n, 8, 4, n)
    Hc, W = _chain_size(n, 8)
    rows = people + _clutter({4: a, 12: d, 13: e}, Hc, Hc + 30, W, 31)
    if npk is not None:
        rows += _clutter({7: (npk - len(rows)) // 2, 10: npk - len(rows) - (npk - len(rows)) // 2}, Hc, Hc + 30, W, 32)
    peaks = np.array(rows, np.float32)
    return dict(peaks=peaks[np.random.default_rng(33).permutation(len(peaks))], paf=_paint(Hc + 30, W, bands))


def _pp_pairs(peaks):
    """candidate pairs as process_paf.cu counts them (pair_prefix with max_part = the default 256)"""
    cnt = np.bincount(peaks[:, 4].astype(int), minlength=18)
    return int(sum(min(cnt[a], 256) * min(cnt[b], 256) for a, b in LIMB_PARTS))


# ---- groups: one fresh process each ---------------------------------------------------------------------------------
GROUPS = {"frontend": [f"{f[0]}_{k}" for f in FRONTENDS for k in ("at", "over")],
          "stage45": STAGE45,
          "conn_cap": ["conns_1536_staged", "conns_1539_unstaged"],
          "limits": [f"limits_{v}" for v in LIMIT_VARIANTS],
          "process_paf": [p[0] for p in PROCESS_PAF],
          "growth": ["grow_once_at_the_x4_step", "over_the_limits_raises"]}
CASE_IDS = [(g, c) for g, cs in GROUPS.items() for c in cs]
# eager launches where a profiler trace proves which kernel ran; process_paf and the growth rule as a user runs them
GROUP_ENV = {"frontend": {"EKP_GRAPHS": "0"}, "stage45": {"EKP_GRAPHS": "0"}, "conn_cap": {"EKP_GRAPHS": "0"},
             "limits": {"EKP_GRAPHS": "0"}, "process_paf": {}, "growth": {}}


@functools.lru_cache(maxsize=None)
def _case(name):
    """dict(op, ctx, input, h1, flag, pre, ...) of one case; input is a dict of arrays"""
    if name.rsplit("_", 1)[0] in [f[0] for f in FRONTENDS]:
        fname, kind = name.rsplit("_", 1)
        _, layout, frontend, mat, h, w, npk, kernel = next(f for f in FRONTENDS if f[0] == fname)
        b = _frontend_batch(fname)
        cap = npk if kind == "at" else npk - 1
        return dict(op="run", ctx=dict(max_batch=len(b["heat"]), max_h=h, max_w=w, max_peaks=cap, max_humans=128), input=b,
                    layout=layout, frontend=frontend, materialize=mat, kernel=kernel, flag=0 if kind == "at" else OVF_PEAKS,
                    npk=npk)
    if name in STAGE45:
        ctx, h1, build, flag, pre = _stage45_cases()[name]
        scenes, H, W = build()
        b = _peak_batch(scenes, H, W)
        return dict(op="peaks", ctx=dict(ctx, max_batch=len(scenes), max_h=8, max_w=8), input=b, h1=h1, flag=flag, pre=pre)
    if name.startswith("conns_"):
        people = 512 if "1536" in name else 513
        scenes, H, W = _conn_cap_scene(people)
        return dict(op="peaks", ctx=dict(CONN_CTX, max_batch=3, max_h=8, max_w=8), input=_peak_batch(scenes, H, W), h1=CHAIN_H1,
                    flag=0, pre=dict(conns=3 * people))
    if name.startswith("limits_"):
        v = name[len("limits_"):]
        return dict(op="peaks", ctx=dict(LIMITS, max_batch=3, max_h=8, max_w=8), input=_limit_batch(v), h1=CHAIN_H1,
                    flag=LIMIT_VARIANTS[v], pre=dict(limit=v), shared_paf=True)
    if name.startswith("pp_"):
        return dict(op="process_paf", input=_pp_scene(name), route=next(p[3] for p in PROCESS_PAF if p[0] == name))
    if name == "grow_once_at_the_x4_step":     # 64 peaks, max_peaks 16: one x4 step fits exactly
        rng = np.random.default_rng(41)
        heat = _spikes(46, 54, 64, 41)[None].transpose(0, 3, 1, 2)
        paf = rng.normal(0, 0.5, (1, 38, 46, 54)).astype(np.float32)
        return dict(op="grow", input=dict(heat=np.ascontiguousarray(heat), paf=paf), max_peaks=16)
    if name == "over_the_limits_raises":       # a checkerboard: 1242 maxima on every part, 22356 in all
        heat = np.zeros((1, 19, 46, 54), np.float32)
        heat[:, :18] = (np.add.outer(np.arange(46), np.arange(54)) % 2 == 0).astype(np.float32)
        return dict(op="grow", input=dict(heat=heat, paf=np.zeros((1, 38, 46, 54), np.float32)), max_peaks=2048)
    raise KeyError(name)


# ---- the worker (a fresh process per group) ------------------------------------------------------------------------
def _worker(spec_path, out_path):
    import torch
    from torch.profiler import ProfilerActivity, profile

    import torch_ekpose_b200 as ek
    from torch_ekpose_b200 import paf_to_pose
    with open(spec_path) as f:
        spec = json.load(f)
    d = os.path.dirname(spec_path)
    out = {}
    for case in spec["cases"]:
        name = case["name"]
        with np.load(os.path.join(d, name + ".npz")) as z:
            data = {k: z[k] for k in z.files}
        try:
            if case["op"] == "grow":
                paf_to_pose._cache.clear()
                try:
                    humans = ek.postprocess_batch(data["heat"], data["paf"], max_peaks=case["max_peaks"], max_humans=128)
                    out[name + "/humans"] = np.array(len(humans[0]))
                    out[name + "/max_peaks"] = np.array(paf_to_pose._cache[(0,)].max_peaks)
                except ek._lib.EkpCapacityError as e:
                    out[name + "/raised"] = np.array(str(e))
                paf_to_pose._cache.clear()
                continue
            if case["op"] == "process_paf":
                heat_mat = np.zeros((PP_H1, 1, 19), np.float32)   # process_paf reads only its height
                ek.pafprocess.process_paf(data["peaks"][None], heat_mat, data["paf"])   # sizes the context, captures graphs
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    ek.pafprocess.process_paf(data["peaks"][None], heat_mat, data["paf"])
                    torch.cuda.synchronize()
                pf, npk = ek.pafprocess, len(data["peaks"])
                nh = pf.get_num_humans()
                out[name + "/events"] = np.array(json.dumps(sorted({e.name for e in prof.events()})))
                out[name + "/num_humans"] = np.array(nh)
                out[name + "/cids"] = np.array([[pf.get_part_cid(h, p) for p in range(18)] for h in range(nh)], np.int32).reshape(nh, 18)
                out[name + "/scores"] = np.array([pf.get_score(h) for h in range(nh)], np.float32)
                out[name + "/line"] = np.array([(pf.get_part_x(k), pf.get_part_y(k)) for k in range(npk)], np.int32)
                out[name + "/line_score"] = np.array([pf.get_part_score(k) for k in range(npk)], np.float32)
                continue
            pp = ek.PostProcessor(device=0, **case["ctx"])   # one context per case, in increasing size within a group
            for oi, order in enumerate(case["orders"]):
                key = f"{name}/{oi}/"
                if case["op"] == "run":
                    heat, paf = torch.from_numpy(data["heat"][order]).cuda(), torch.from_numpy(data["paf"][order]).cuda()
                else:
                    peaks, counts = torch.from_numpy(data["peaks"][order]).cuda(), torch.from_numpy(data["counts"][order]).cuda()
                    paf = torch.from_numpy(data["paf"]).cuda()
                    paf = paf.expand(len(order), *paf.shape[1:]).contiguous() if case.get("shared_paf") else paf[order]
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    if case["op"] == "run":
                        pp.run(heat, paf, layout=case["layout"], frontend=case["frontend"], materialize=case["materialize"])
                    else:
                        pp.run_peaks(peaks, counts, paf, h1=case["h1"])
                    res = pp.results(with_peaks=case["op"] == "run", raise_on_overflow=False)
                    torch.cuda.synchronize()
                try:
                    pp.results()
                    raised = False
                except ek._lib.EkpCapacityError:
                    raised = True
                out[key + "raised"] = np.array(raised)
                out[key + "kernels"] = np.array(json.dumps(sorted({e.name for e in prof.events()})))
                for k, v in res.items():
                    out[key + k] = v
                del paf
            pp.close()
        except Exception as e:   # a refused launch is this case's finding; the other cases still run
            out[name + "/error"] = np.array(f"{type(e).__name__}: {e}")
    np.savez(out_path, **out)


_WORKER = "import sys; from tests.test_capacity_edges import _worker; _worker(sys.argv[1], sys.argv[2])"


@pytest.fixture(scope="module")
def run_group(tmp_path_factory):
    done = {}

    def run(group):
        if group not in done:
            d = tmp_path_factory.mktemp(group)
            cases = []
            for name in GROUPS[group]:
                c = _case(name)
                np.savez(d / (name + ".npz"), **c["input"])
                spec = {k: v for k, v in c.items() if k not in ("input", "pre")}
                if c["op"] in ("run", "peaks"):
                    n = len(c["input"]["heat"] if c["op"] == "run" else c["input"]["counts"])
                    spec["orders"] = _orders(n)
                cases.append(dict(spec, name=name))
            with open(d / "spec.json", "w") as f:
                json.dump(dict(cases=cases), f)
            env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
            for k in ("EKP_GRAPHS", "EKP_LEAN_TILED", "EKP_BY_SAMPLE_MAX_PAIRS", "EKP_PROCESS_PAF_UPLOAD", "EKP_DEVICE"):
                env.pop(k, None)
            env.update(GROUP_ENV[group])
            r = subprocess.run([sys.executable, "-c", _WORKER, str(d / "spec.json"), str(d / "out.npz")], capture_output=True,
                               text=True, env=env, cwd=ROOT, timeout=1200)
            assert r.returncode == 0, f"worker for {group} exited {r.returncode}:\n{r.stderr[-3000:]}"
            with np.load(d / "out.npz") as z:
                done[group] = {k: z[k] for k in z.files}
        return done[group]
    return run


# ---- the oracle ------------------------------------------------------------------------------------------------------
def _hwc(a, layout, i):
    return np.ascontiguousarray(a[i].transpose(1, 2, 0)) if layout == "nchw" else np.ascontiguousarray(a[i])


@functools.lru_cache(maxsize=None)
def _oracle_frontend(name, i):
    """(peaks [N, 5], subset) of image i of a front-end case"""
    c = _case(name)
    hw, pw = _hwc(c["input"]["heat"], c["layout"], i), _hwc(c["input"]["paf"], c["layout"], i)
    fe = util.frontend()
    if c["frontend"] == "dense":
        peaks, paf_mat = fe.dense_peaks(hw), fe.upsample_bilinear(pw)
    else:
        peaks, paf_mat = fe.ref_nms(hw, gauss=c["frontend"] == "reference_gauss"), fe.upsample_nearest(pw)
    sub, _ = util.oracle_people(peaks, 8 * hw.shape[0], 8 * hw.shape[1], paf_mat)
    return peaks, sub


def _image_inputs(c, i):
    b = c["input"]
    paf = b["paf"][0] if c.get("shared_paf") else b["paf"][i]
    return b["peaks"][i, :b["counts"][i]], paf


@functools.lru_cache(maxsize=None)
def _oracle_peaks(name, i):
    """subset of image i of a run_peaks case, and what the C restatement saw: candidates and connections per limb"""
    c = _case(name)
    peaks, paf = _image_inputs(c, i)
    port = util.port()
    sub, _ = oracle.subset_of(port, peaks, c["h1"], paf.shape[1], paf)
    cands = [port.candidates(limb)["score"] for limb in range(19)]
    conns = [len(port.connections(limb)["cid1"]) for limb in range(19)]
    if util.ref_or_none() is not None:   # the people from the compiled reference where it was built
        sub, _ = util.oracle_people(peaks, c["h1"], paf.shape[1], paf)
    return sub, cands, conns


def _check_preconditions(name, c):
    """the edge image (0) really sits where the case says"""
    pre, flag = c["pre"], c["flag"]
    peaks, _ = _image_inputs(c, 0)
    parts = np.bincount(peaks[:, 4].astype(int), minlength=18)
    ctx = c["ctx"]
    if "peaks" in pre:
        assert len(peaks) == pre["peaks"] == ctx["max_peaks"] + (flag != 0)
    if "limit" in pre:
        v = pre["limit"]
        assert len(peaks) == LIMITS["max_peaks"] + (v == "peaks") and parts.max() == LIMITS["max_part"] + (v == "part")
        if v == "at" or flag:
            _, cands, conns = _oracle_peaks(name, 0)
            assert len(cands[18]) == LIMITS["max_cand"] + (v == "cand")
            assert max(len(s) for s in cands) == len(cands[18])
            assert conns[0] == conns[2] == conns[3] == 1024
            rows = 1024 + (v == "humans")   # limb 0 starts 1024 rows, limb 13 one more; limb 18 starts none
            assert conns[13] == (v == "humans") and rows <= LIMITS["max_humans"] + (v == "humans")
        return
    if c["op"] != "peaks" or "people" not in pre and "conns" not in pre and "tied" not in pre:
        return
    sub, cands, conns = _oracle_peaks(name, 0)
    if "people" in pre:
        n = pre["people"]
        assert conns[0] == n if "rows_over" not in name else conns[0] == 33
        if "part_" in name:
            assert parts[2] == n == ctx["max_part"] + (flag != 0)          # RShoulder: B of limb 0, A of limb 2
        if "humans_" in name:
            rows = conns[0]                                               # every limb-0 connection starts a row
            assert rows == ctx["max_humans"] + (flag != 0) and len(sub) == n
        assert max(len(s) for s in cands) <= ctx.get("max_cand", 2048)
    if "tied" in pre and isinstance(pre["tied"], int):
        assert len(cands[0]) == pre["tied"] == ctx["max_cand"] + (flag != 0)
        assert len(np.unique(cands[0])) == 1 and len(sub) == min(int(parts[1]), int(parts[2]))
    if "tied" in pre and isinstance(pre["tied"], list):
        for i, t in enumerate(pre["tied"]):
            s = _oracle_peaks(name, i)[1][0]
            assert len(s) == t and len(np.unique(s)) == 1
    if "conns" in pre and isinstance(pre["conns"], list):
        for i, k in enumerate(pre["conns"]):
            cn = _oracle_peaks(name, i)[2]
            assert cn[0] == cn[2] == cn[3] == k and sum(cn) == 3 * k
    if "conns" in pre and isinstance(pre["conns"], int):
        assert sum(conns) == pre["conns"] and len(sub) == pre["conns"] // 3
        assert conn_cap(ctx["max_humans"], ctx["max_part"]) == CONN_CAP_MAX
        assert (sum(conns) <= CONN_CAP_MAX) == ("staged" in name and "unstaged" not in name)


def _check_batch(name, c, out):
    n = len(c["input"]["heat"] if c["op"] == "run" else c["input"]["counts"])
    for oi, order in enumerate(_orders(n)):
        key = f"{name}/{oi}/"
        ovf = out[key + "overflow"]
        assert bool(out[key + "raised"]) == (c["flag"] != 0), f"{name} order {oi}: raised {out[key + 'raised']}"
        for pos, img in enumerate(order):
            want_flag = c["flag"] if img == 0 else 0
            assert int(ovf[pos]) == want_flag, f"{name} order {oi}: image {img} at {pos} has overflow {int(ovf[pos])}, want {want_flag}"
            if want_flag:
                continue   # what was kept of a scene that did not fit is not specified
            m = int(out[key + "num_humans"][pos])
            if c["op"] == "run":
                peaks, sub = _oracle_frontend(name, img)
                res = dict(n_peaks=out[key + "n_peaks"], peaks=out[key + "peaks"], part_off=out[key + "part_off"])
                assert_bits_equal(util.peaks_table(res, pos), peaks, f"{name} order {oi} image {img} peaks")
            else:
                sub = _oracle_peaks(name, img)[0]
            assert m == len(sub), f"{name} order {oi} image {img}: {m} people vs {len(sub)}"
            assert_bits_equal(out[key + "subset"][pos, :m], sub, f"{name} order {oi} image {img} subset")


@pytest.mark.gpu
@pytest.mark.parametrize("group,name", CASE_IDS, ids=[f"{g}-{c}" for g, c in CASE_IDS])
def test_capacity_edge_equals_the_oracle(run_group, group, name):
    c = _case(name)
    out = run_group(group)
    assert name + "/error" not in out, f"{name}: {out[name + '/error']}"
    if c["op"] == "grow":
        if name == "over_the_limits_raises":
            msg = str(out[name + "/raised"]) if name + "/raised" in out else ""
            assert f"peaks {LIMITS['max_peaks']}" in msg and f"peaks per part {LIMITS['max_part']}" in msg, msg
            return
        assert name + "/raised" not in out, str(out.get(name + "/raised"))
        hw = np.ascontiguousarray(c["input"]["heat"][0].transpose(1, 2, 0))
        pw = np.ascontiguousarray(c["input"]["paf"][0].transpose(1, 2, 0))
        peaks, sub = util.oracle_reference(hw, pw)
        assert len(peaks) == 4 * c["max_peaks"]                    # exactly one x4 step
        assert int(out[name + "/max_peaks"]) == 4 * c["max_peaks"]  # grown once, not twice
        assert int(out[name + "/humans"]) == len(sub)
        return
    if c["op"] == "process_paf":
        peaks = c["input"]["peaks"]
        route = c["route"]
        pairs = _pp_pairs(peaks)
        small = len(peaks) <= SMALL_PEAKS and 10 * pairs <= SMALL_MAX_SAMPLES
        listed = 10 * pairs <= LISTED_MAX_SAMPLES
        assert route == ("small" if small else "listed" if listed else "sparse")
        spec = next(p for p in PROCESS_PAF if p[0] == name)
        assert len(peaks) == spec[1] if spec[1] is not None else pairs == spec[2]
        ev = json.loads(str(out[name + "/events"]))
        assert any("paf_connect_kernel" in e or "cudaGraphLaunch" in e for e in ev), ev
        h2d = [e for e in ev if re.search(r"memcpy.*htod", e, re.I)]
        offsets = any("pair_sample_offsets_kernel" in e for e in ev)
        if route == "small":
            assert not h2d and not offsets, ev
        elif route == "listed":
            assert h2d and not offsets, ev
        else:
            assert offsets, ev
        sub, line = util.oracle_people(peaks, PP_H1, c["input"]["paf"].shape[1], c["input"]["paf"])
        nh = int(out[name + "/num_humans"])
        assert nh == len(sub) > 0, (nh, len(sub))
        assert np.array_equal(out[name + "/cids"], sub[:, :18].astype(np.int32))
        assert_bits_equal(out[name + "/scores"], (sub[:, 18] / sub[:, 19]).astype(np.float32), "human scores")
        assert np.array_equal(out[name + "/line"][:, 0], line[0]) and np.array_equal(out[name + "/line"][:, 1], line[1])
        assert_bits_equal(out[name + "/line_score"], line[2], "getter table scores")
        return
    if c["op"] == "run":
        peaks, _ = _oracle_frontend(name, 0)
        assert len(peaks) == c["npk"] == c["ctx"]["max_peaks"] + (c["flag"] != 0)
        for oi in range(2):
            names = json.loads(str(out[f"{name}/{oi}/kernels"]))
            assert any(re.search(c["kernel"], k) for k in names), f"{name}: no kernel matches {c['kernel']!r}; ran {names}"
        if name.startswith("dense_plane_sliced"):
            import torch
            assert 18 * len(c["input"]["heat"]) < torch.cuda.get_device_properties(0).multi_processor_count
        if name.startswith("dense_plane_") and "sliced" not in name:
            import torch
            assert 18 * len(c["input"]["heat"]) >= torch.cuda.get_device_properties(0).multi_processor_count
    else:
        _check_preconditions(name, c)
    _check_batch(name, c, out)


def test_case_table_matches_the_builders():
    """every case id names a case the builders know (no GPU: the scenes are CPU arrays)"""
    names = {f"{f[0]}_{k}" for f in FRONTENDS for k in ("at", "over")} | set(STAGE45) | set(_stage45_cases())
    names |= {"conns_1536_staged", "conns_1539_unstaged"} | {f"limits_{v}" for v in LIMIT_VARIANTS}
    names |= {p[0] for p in PROCESS_PAF} | {"grow_once_at_the_x4_step", "over_the_limits_raises"}
    assert set(STAGE45) == set(_stage45_cases())
    assert {c for _, c in CASE_IDS} <= names and len(CASE_IDS) == len(set(CASE_IDS))


def _source(*path):
    with open(os.path.join(ROOT, *path)) as f:
        return f.read()


def _const(src, pattern):
    m = re.search(pattern, src)
    assert m, f"{pattern!r} not found"
    return eval(m.group(1), {})   # a C integer expression of literals, e.g. 64 * 1024


def test_thresholds_are_the_ones_the_cases_sit_on():
    """The constants the GPU cases are built around, read from the sources: a changed threshold must fail here instead
    of silently moving the cases off their edges."""
    pp = _source("torch_ekpose_b200", "csrc", "process_paf.cu")
    assert _const(pp, r"const int kSmallPeaks = ([^;]+);") == SMALL_PEAKS
    assert _const(pp, r"const long long kSmallMaxSamples = ([^;]+);") == SMALL_MAX_SAMPLES
    assert _const(pp, r"const long long kListedMaxSamples = ([^;]+);") == LISTED_MAX_SAMPLES
    asm = _source("torch_ekpose_b200", "csrc", "assemble.cu")
    assert _const(asm, r"if \(c > (\d+)\) c = \d+;") == CONN_CAP_MAX
    assert _const(asm, r"if \(c < (\d+)\) c = \d+;") == CONN_CAP_MIN
    assert re.search(r"want = 24ll \* max_humans, all = 19ll \* max_part", asm)
    ps = _source("torch_ekpose_b200", "csrc", "peaks_sort.cu")
    assert _const(ps, r"constexpr int kOneMaxPeaks = (\d+);") == ONE_MAX_PEAKS
    assert _const(ps, r"constexpr int kSortThreads = (\d+);") == SORT_SLICE
    hdr = _source("include", "ekpose_b200.h")
    for name, key in (("PEAKS", "max_peaks"), ("HUMANS", "max_humans"), ("PART", "max_part"), ("CAND", "max_cand")):
        assert _const(hdr, rf"#define EKP_LIMIT_{name} (\d+)") == LIMITS[key]
    # the cases that sit on them
    assert conn_cap(CONN_CTX["max_humans"], CONN_CTX["max_part"]) == CONN_CAP_MAX == 3 * 512 < 3 * 513
    assert conn_cap(LIMITS["max_humans"], LIMITS["max_part"]) == CONN_CAP_MAX
    assert conn_cap(1, 1) == CONN_CAP_MIN and conn_cap(40, 256) == 960 and conn_cap(128, 33) == 627
    assert [f[6] for f in FRONTENDS if f[6] % SORT_SLICE == 0] and [f[6] for f in FRONTENDS if f[6] % SORT_SLICE == 1]
    assert 10 * (SMALL_MAX_SAMPLES // 10) <= SMALL_MAX_SAMPLES < 10 * (SMALL_MAX_SAMPLES // 10 + 1)
    assert 10 * (LISTED_MAX_SAMPLES // 10) <= LISTED_MAX_SAMPLES < 10 * (LISTED_MAX_SAMPLES // 10 + 1)
    for name, npk, pairs, route in PROCESS_PAF:
        peaks = _pp_scene(name)["peaks"]
        assert len(peaks) == npk if npk is not None else (_pp_pairs(peaks) == pairs and len(peaks) <= SMALL_PEAKS)
        assert len(peaks) <= ONE_MAX_PEAKS   # the one-block ingest and sort
