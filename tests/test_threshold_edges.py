"""Every score threshold of stages 4-5 and every comparison of the tracker, run at its exact edge and one past it,
against the oracle.

Random scenes never land on a threshold, so a kernel that compares with `>=` where the reference compares with `>`, or
that contracts a dot product into an FMA, passes every random test.  Here each edge is a pair of images (or frame
sequences) built so that the compared quantity equals the threshold bit for bit on one side and is the neighbouring
float (or the next integer) on the other, and the oracle's decision differs between the two:

* A, limb scoring (stage 4): a sample's score against 0.05 and the sample count against 6, in every position of the ten
  samples; pass 1's prefilter on samples 3..6; a dot product that is exactly 0.05 only without FMA contraction;
  criterion2 at exactly 0 and the distance penalty at its kink; roundpaf's `(int)(v + 0.5)` on positions that are
  exactly (or, for inexact steps, rounded onto) k + 0.5.
* B, the human prune (stage 5): a person whose r[18] / r[19] is exactly 0.3f and one float below it, with the closing
  peak score entering r[18] through a new row, an extension and a merge; 4, 5, 7 and 18 parts; 3 against 4 parts.
* D, the tracker: similarities that are exact (k / 4) on every device; min_oks on a similarity and one float above it;
  ties at min_oks 0 among 40 people and 40 tracks, in two row orders; a chain that needs one matching round per pair;
  expiry after max_age and max_age + 1 missing frames; eviction among tracks last seen in the same frame; P x L at the
  shared similarity cache's capacity and one pair past it.

Every case asserts its own edge on the CPU: stage 4-5 quantities are recomputed in NumPy float32 / float64 in the
reference's operation order and the oracle's people differ between the two sides; the tracker's similarities are all
k / 4 and the oracle's ids differ between the sides (or, for ties, from the reversed tie-break).  The GPU runs the stage
4-5 cases through run_peaks with both stage 4 routes (one thread per pair in two passes, EKP_BY_SAMPLE_MAX_PAIRS=0; ten
lanes per pair, EKP_BY_SAMPLE_MAX_PAIRS=1000000; a fresh process each, as in test_launch_variants.py) and through the host
process_paf on its listed, sparse and dense upload routes, and the tracker cases through Tracker.update; the tracker's
host hook (the kernel's code on one CPU thread) runs them without a GPU.  test_score_thresholds_are_the_ones_the_cases_sit_on
reads the constants from the sources."""
import functools
import json
import os
import re
import subprocess
import sys
from fractions import Fraction

import numpy as np
import pytest

import oracle
from tests import test_capacity_edges as ce
from tests import test_tracking as tt
from tests import util
from tests.util import assert_bits_equal

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32
THR_SAMPLE = f32(0.05)      # THRESH_VECTOR_SCORE: a sample passes when its score is > this
THR_COUNT = 6               # THRESH_VECTOR_CNT1: a pair needs more passing samples than this
THR_PARTS = 4               # THRESH_PART_CNT: a person needs at least this many parts
THR_HUMAN = f32(0.3)        # THRESH_HUMAN_SCORE: ... and r[18] / r[19] at least this
FAR_H1 = 4096               # heat height for which no pair of these scenes is penalised
PASS, FAIL = f32(0.5), f32(0.0)


def _up(v, n=1):
    for _ in range(n):
        v = np.nextafter(f32(v), f32(np.inf))
    return f32(v)


def _down(v, n=1):
    for _ in range(n):
        v = np.nextafter(f32(v), f32(-np.inf))
    return f32(v)


# ---- the reference's arithmetic, restated in NumPy float32 / float64 (pafprocess.cpp:59-94, 220-242) ------------------
def roundpaf(v):
    return int(np.float64(f32(v)) + 0.5)


def pair_geometry(a, b):
    """(vx, vy, norm, [(lx, ly)] of the ten samples) of the pair a -> b, as get_paf_vectors computes them"""
    dx, dy = f32(b[0] - a[0]), f32(b[1] - a[1])
    norm = f32(np.sqrt(f32(f32(dx * dx) + f32(dy * dy))))
    vx, vy = f32(dx / norm), f32(dy / norm)
    sx, sy = f32(dx / f32(10)), f32(dy / f32(10))
    cells = [(roundpaf(f32(f32(a[0]) + f32(f32(i) * sx))), roundpaf(f32(f32(a[1]) + f32(f32(i) * sy)))) for i in range(10)]
    return vx, vy, norm, cells


def sample_score(vx, vy, px, py):
    """no contraction: both products rounded, then the sum"""
    return f32(f32(vx * px) + f32(vy * py))


def pair_criteria(a, b, values, h1):
    """(criterion1, criterion2) of the pair with sample values [(px, py)] * 10"""
    vx, vy, norm, _ = pair_geometry(a, b)
    s = [sample_score(vx, vy, px, py) for px, py in values]
    scores = f32(0)
    for v in s:
        scores = f32(scores + v)
    penalty = 0.5 * float(h1) / float(norm) - 1.0
    c2 = f32(float(f32(scores / f32(10))) + min(0.0, penalty))
    return sum(v > THR_SAMPLE for v in s), c2


def accepted(a, b, values, h1):
    c1, c2 = pair_criteria(a, b, values, h1)
    return c1 > THR_COUNT and c2 > 0


# ---- scenes: one peak per part, every limb painted only along its own samples ------------------------------------------
# A scene is drawn from (peaks {part: (x, y, score)}, limbs {limb: [(px, py)] * 10 or (px, py)}, extra rows, H, W) into
# (peak rows (x, y, score, 0, part), full-resolution PAF [H, W, 38]).
def _paint_limb(paf, limb, a, b, values):
    ch = ce.LIMB_CH[limb]
    _, _, _, cells = pair_geometry(a, b)
    for (lx, ly), (px, py) in zip(cells, values):
        old = paf[ly, lx, ch:ch + 2].copy()
        assert not old.any() or (old == (px, py)).all(), f"limb {limb}: cell {(lx, ly)} sampled with two values"
        paf[ly, lx, ch], paf[ly, lx, ch + 1] = px, py


def _render(scene):
    peaks, limbs, extra, H, W = scene
    paf = np.zeros((H, W, 38), np.float32)
    for limb, values in limbs.items():
        if values is None:   # painted by the caller
            continue
        pa, pb = ce.LIMB_PARTS[limb]
        vals = values if isinstance(values, list) else [values] * 10
        _paint_limb(paf, limb, peaks[pa][:2], peaks[pb][:2], vals)
    rows = [(x, y, s, 0, p) for p, (x, y, s) in sorted(peaks.items())] + list(extra)
    return rows, paf


def _arm(a, values, dx=10, dy=0, score=PASS):
    """neck at a, RShoulder at a + (dx, dy), RElbow and RWrist 10 and 20 px right of it: limb 0 carries the samples
    under test, limbs 2 and 3 pass with score 1.  The pair decides whether there is a four-part person (kept) or a
    three-part one (pruned), so the subset shows the decision."""
    x0, y0 = a
    xb, yb = x0 + dx, y0 + dy
    peaks = {1: (x0, y0, score), 2: (xb, yb, score), 3: (xb + 10, yb, score), 4: (xb + 20, yb, score)}
    limbs = {0: values, 2: (f32(1), f32(0)), 3: (f32(1), f32(0))}
    return peaks, limbs


def _scene(peaks, limbs, extra=(), H=None, W=None):
    xs = [p[0] for p in peaks.values()] + [r[0] for r in extra]
    ys = [p[1] for p in peaks.values()] + [r[1] for r in extra]
    return _render((peaks, limbs, list(extra), H or max(ys) + 8, W or max(xs) + 8))


def _values(spec):
    """ten (px, py) from a list of x-channel values (a horizontal limb: the score is the value)"""
    return [(f32(v), f32(0)) for v in spec]


# ---- A: limb scoring -----------------------------------------------------------------------------------------------------
A_ORIGIN = (4, 6)


def _case_sample_threshold(k):
    """sample k at exactly 0.05 (fails) with 6 other passing samples: 6 pass, rejected; at nextafter(0.05, 1): 7 pass"""
    others = [j for j in range(10) if j != k]
    base = [FAIL] * 10
    for j in others[:6]:
        base[j] = PASS
    base[others[6]] = THR_SAMPLE     # a second sample on the edge: 0.05 never counts
    at, past = list(base), list(base)
    at[k], past[k] = THR_SAMPLE, _up(THR_SAMPLE)
    imgs = [_scene(*_arm(A_ORIGIN, _values(v))) for v in (at, past)]
    return dict(images=imgs, h1=FAR_H1, accept=[False, True], edge=("sample", k))


def _clutter_arms(n, y0):
    """n necks and n RShoulders in rows where no PAF is painted: n * n more limb-0 pairs that all fail"""
    return [(2 + 3 * j, y0 + (j % 4), f32(0.5), 0, 1) for j in range(n)] + \
           [(3 + 3 * j, y0 + 6 + (j % 4), f32(0.5), 0, 2) for j in range(n)]


PREFILTER_CLUTTER = 23   # 24 x 24 = 576 limb-0 pairs: more than 2 x 256 threads, so pass 1 runs in the per-pair route


def _case_prefilter():
    """exactly 7 passing samples, the only passing middle one (3..6) being k: accepted for every k; all four middle
    samples at exactly 0.05 and the six outer ones passing: rejected"""
    imgs, acc = [], []
    for k in (3, 4, 5, 6, None):
        v = [PASS, PASS, PASS, THR_SAMPLE, THR_SAMPLE, THR_SAMPLE, THR_SAMPLE, PASS, PASS, PASS]
        if k is not None:
            v[k] = PASS
        peaks, limbs = _arm(A_ORIGIN, _values(v))
        imgs.append(_scene(peaks, limbs, _clutter_arms(PREFILTER_CLUTTER, 24)))
        acc.append(k is not None)
    return dict(images=imgs, h1=FAR_H1, accept=acc, edge=("prefilter",))


DIAG = (30, 40)    # a 3-4-5 limb: vx = 0.6f, vy = 0.8f, samples on whole cells 3 and 4 px apart


@functools.lru_cache(maxsize=None)
def contraction_sample():
    """(sx, sy_at, sy_past): fl(fl(0.6 sx) + fl(0.8 sy_at)) == 0.05f while the fused fma(0.6, sx, fl(0.8 sy_at)) is
    above it; with sy_past the stepwise score is the next float above 0.05f"""
    vx, vy, _, _ = pair_geometry((0, 0), DIAG)
    sx, sy = f32(0.14277099), f32(-0.044578243)
    past = None
    for n in range(1, 4096):
        for cand in (_up(sy, n), _down(sy, n)):
            if sample_score(vx, vy, sx, cand) == _up(THR_SAMPLE):
                past = cand
                break
        if past is not None:
            break
    assert past is not None
    return sx, sy, past


def fused_score(vx, vy, px, py):
    """fma(vx, px, fl(vy py)) rounded once, exactly (Fraction), as a contracting compiler would compute a sample"""
    exact = Fraction(float(vx)) * Fraction(float(px)) + Fraction(float(f32(vy * py)))
    lo = f32(float(exact))
    hi = _up(lo) if Fraction(float(lo)) < exact else _down(lo)
    lo_d, hi_d = abs(Fraction(float(lo)) - exact), abs(Fraction(float(hi)) - exact)
    return lo if lo_d < hi_d or (lo_d == hi_d and int(lo.view(np.uint32)) % 2 == 0) else hi


def _case_contraction(k):
    sx, sy_at, sy_past = contraction_sample()
    base = [(PASS, PASS)] * 6 + [(FAIL, FAIL)] * 4
    base = base[:k] + [None] + base[k:9]
    imgs = []
    for sy in (sy_at, sy_past):
        v = [(sx, sy) if e is None else e for e in base]
        imgs.append(_scene(*_arm(A_ORIGIN, v, *DIAG)))
    return dict(images=imgs, h1=FAR_H1, accept=[False, True], edge=("contraction", k))


PENALTY_H1 = 20    # limbs 2 and 3 (10 px) are not penalised: 0.5 * 20 / 10 - 1 == 0


def _case_criterion2_zero():
    """norm == h1: penalty exactly -0.5; ten samples of 0.5 give scores / 10 == 0.5f and criterion2 == 0 (rejected);
    the last sample raised by 2^-21 makes scores / 10 the next float above 0.5 (accepted)"""
    at = [PASS] * 10
    past = [PASS] * 9 + [f32(0.5 + 2.0 ** -21)]
    imgs = [_scene(*_arm(A_ORIGIN, _values(v), dx=PENALTY_H1)) for v in (at, past)]
    return dict(images=imgs, h1=PENALTY_H1, accept=[False, True], edge=("criterion2",))


def _case_penalty_kink():
    """norm == h1 / 2: no penalty (accepted); norm == h1 / 2 + 1: the penalty takes the small mean below zero"""
    v = _values([0.0625] * 7 + [0] * 3)
    imgs = [_scene(*_arm(A_ORIGIN, v, dx=PENALTY_H1 // 2 + d)) for d in (0, 1)]
    return dict(images=imgs, h1=PENALTY_H1, accept=[True, False], edge=("penalty",))


def _positions(ax, dx):
    """(float32 x position, roundpaf cell) of the ten samples of a horizontal pair ax -> ax + dx"""
    st = f32(f32(dx) / f32(10))
    pos = [f32(f32(ax) + f32(f32(i) * st)) for i in range(10)]
    return pos, [roundpaf(p) for p in pos]


@functools.lru_cache(maxsize=None)
def roundpaf_layout(dx):
    """(ax, pass cells up, pass cells down) for a horizontal pair of length dx: some sample sits exactly on k + 0.5 with
    k even, where roundpaf takes k + 1 and a round-half-even (rintf) takes k.  `up`: roundpaf's cells give 7 or more
    passing samples, rint's 6 or fewer; `down` the other way round."""
    for ax in range(4, 14):
        pos, cells = _positions(ax, dx)
        alt = [int(np.rint(p)) for p in pos]
        if cells == alt:
            continue
        uni = sorted(set(cells) | set(alt))
        found = {}
        for mask in range(1 << len(uni)):
            good = {c for j, c in enumerate(uni) if mask >> j & 1}
            n, m = sum(c in good for c in cells), sum(c in good for c in alt)
            if n > THR_COUNT >= m and "up" not in found:
                found["up"] = good
            if m > THR_COUNT >= n and "down" not in found:
                found["down"] = good
        if len(found) == 2:
            return ax, found["up"], found["down"]
    raise AssertionError(f"no roundpaf layout for dx = {dx}")


ROUNDPAF_EXACT = (5, 15, 25)      # step 0.5, 1.5, 2.5: the odd samples land exactly on k + 0.5
ROUNDPAF_INEXACT = (3, 7, 13)     # step 0.3f, 0.7f, 1.3f: the float product lands next to k + 0.5


def _case_roundpaf(dx):
    """the same pair twice: the cells roundpaf reads pass in `up` (accepted) and the cells only a round-half-even would
    read pass in `down` (rejected)"""
    ax, up, down = roundpaf_layout(dx)
    y = A_ORIGIN[1]
    imgs = []
    for good in (up, down):
        peaks, limbs = _arm((ax, y), None, dx=dx)
        rows, paf = _scene(peaks, limbs)
        for c in good:
            paf[y, c, ce.LIMB_CH[0]] = PASS
        imgs.append((rows, paf))
    return dict(images=imgs, h1=FAR_H1, accept=[True, False], edge=("roundpaf", dx))


# ---- B: the human prune --------------------------------------------------------------------------------------------------
def assemble(conns, score_of):
    """pafprocess.cpp:127-191 restated in float32: conns {limb: [(cid1, cid2, score)]}, score_of {cid: peak score}.
    Returns (rows before the prune, rows kept, the branch every connection took)."""
    rows, log = [], []
    for limb in range(19):
        p1, p2 = ce.LIMB_PARTS[limb]
        for cid1, cid2, sc in conns.get(limb, []):
            sc = f32(sc)
            hits = [s for s, r in enumerate(rows) if r[p1] == f32(cid1) or r[p2] == f32(cid2)]
            if len(hits) == 1:
                r = rows[hits[0]]
                if r[p2] != f32(cid2):
                    r[p2], r[19] = f32(cid2), f32(r[19] + f32(1))
                    r[18] = f32(r[18] + f32(f32(score_of[cid2]) + sc))
                    log.append("extend")
            elif len(hits) == 2:
                r1, r2 = rows[hits[0]], rows[hits[1]]
                if not any(r1[q] > 0 and r2[q] > 0 for q in range(18)):
                    for q in range(18):
                        r1[q] = f32(r1[q] + f32(r2[q] + f32(1)))
                    r1[19] = f32(r1[19] + r2[19])
                    r1[18] = f32(r1[18] + r2[18])
                    r1[18] = f32(r1[18] + sc)
                    del rows[hits[1]]
                    log.append("merge")
                else:
                    r1[p2], r1[19] = f32(cid2), f32(r1[19] + f32(1))
                    r1[18] = f32(r1[18] + f32(f32(score_of[cid2]) + sc))
                    log.append("membership")
            elif not hits and limb < 18:
                r = np.full(20, -1, np.float32)
                r[p1], r[p2], r[19] = cid1, cid2, 2
                r[18] = f32(f32(f32(score_of[cid1]) + f32(score_of[cid2])) + sc)
                rows.append(r)
                log.append("new")
    kept = [r for r in rows if not (r[19] < f32(THR_PARTS) or f32(r[18] / r[19]) < THR_HUMAN)]
    return rows, kept, log


CONN = f32(0.0625)    # ten samples of 0.0625 on a horizontal limb: criterion2 is exactly 0.0625 (and every sample passes)
BODY = f32(0.25)      # the score of every peak but the closing one
# person: (limbs, closing part, the branch through which the closing peak's score enters r[18])
PRUNE = {"new_row_4": ((0, 2, 3), 1, "new"), "extend_4": ((0, 2, 3), 4, "extend"), "extend_5": ((0, 1, 2, 3), 4, "extend"),
         "extend_7": ((0, 1, 2, 3, 4, 5), 7, "extend"), "extend_18": (tuple(range(17)), 17, "extend"),
         "merge_5": ((0, 2, 14, 17), 16, "merge")}


def _person_positions(limbs, x0):
    """every limb horizontal and 10 px long, B right of A (peaks of different parts may share a position)"""
    x = {ce.LIMB_PARTS[limbs[0]][0]: x0}
    while len(x) < len({p for l in limbs for p in ce.LIMB_PARTS[l]}):
        for l in limbs:
            pa, pb = ce.LIMB_PARTS[l]
            if pa in x and pb not in x:
                x[pb] = x[pa] + 10
            elif pb in x and pa not in x:
                x[pa] = x[pb] - 10
    return x


def _person(limbs, closing, closing_score, y=6, score=BODY):
    x = _person_positions(limbs, 14)
    peaks = {p: (x[p], y, closing_score if p == closing else score) for p in x}
    return _scene(peaks, {l: (CONN, f32(0)) for l in limbs})


def _restated(rows, limbs):
    """assemble() on the connections the construction intends: ids are input rows, which are sorted by part"""
    cid = {int(r[4]): i for i, r in enumerate(rows)}
    conns = {l: [(cid[ce.LIMB_PARTS[l][0]], cid[ce.LIMB_PARTS[l][1]], CONN)] for l in limbs}
    return assemble(conns, {i: r[2] for i, r in enumerate(rows)})


@functools.lru_cache(maxsize=None)
def closing_scores(name):
    """(keep, prune): closing peak scores for which r[18] / r[19] is exactly 0.3f and the float below it"""
    limbs, closing, _ = PRUNE[name]

    def ratio(bits):
        rows, _ = _person(limbs, closing, f32(np.uint32(bits).view(np.float32)))
        r = _restated(rows, limbs)[0][0]
        return f32(r[18] / r[19])

    out = []
    for target in (THR_HUMAN, _down(THR_HUMAN)):
        lo, hi = int(f32(1e-4).view(np.uint32)), int(f32(4).view(np.uint32))   # ratio() is monotone in the closing score
        while lo < hi:
            mid = (lo + hi) // 2
            if ratio(mid) >= target:
                hi = mid
            else:
                lo = mid + 1
        assert ratio(lo) == target, f"{name}: no closing score puts r[18] / r[19] on {target!r}"
        out.append(f32(np.uint32(lo).view(np.float32)))
    return tuple(out)


def _case_prune(name):
    limbs, closing, _ = PRUNE[name]
    imgs = [_person(limbs, closing, s) for s in closing_scores(name)]
    return dict(images=imgs, h1=FAR_H1, people=[1, 0], edge=("prune", name))


def _case_part_count():
    """3 parts against 4 at a peak score of 1: only the count prunes"""
    imgs = [_person(limbs, None, None, score=f32(1)) for limbs in ((0, 2), (0, 2, 3))]
    return dict(images=imgs, h1=FAR_H1, people=[0, 1], edge=("parts",))


# ---- the case table --------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def cases():
    C = {f"sample_{k}": _case_sample_threshold(k) for k in range(10)}
    C["prefilter_3456"] = _case_prefilter()
    for k in (3, 8):
        C[f"contraction_{k}"] = _case_contraction(k)
    C["criterion2_zero"] = _case_criterion2_zero()
    C["penalty_kink"] = _case_penalty_kink()
    for dx in ROUNDPAF_EXACT + ROUNDPAF_INEXACT:
        C[f"roundpaf_dx{dx}"] = _case_roundpaf(dx)
    for name in PRUNE:
        C[f"prune_{name}"] = _case_prune(name)
    C["prune_3_vs_4_parts"] = _case_part_count()
    for c in C.values():
        c.setdefault("people", [int(a) for a in c.get("accept", [])])
    return C


CASES = ["sample_0", "sample_1", "sample_2", "sample_3", "sample_4", "sample_5", "sample_6", "sample_7", "sample_8",
         "sample_9", "prefilter_3456", "contraction_3", "contraction_8", "criterion2_zero", "penalty_kink"] + \
        [f"roundpaf_dx{dx}" for dx in ROUNDPAF_EXACT + ROUNDPAF_INEXACT] + [f"prune_{n}" for n in PRUNE] + ["prune_3_vs_4_parts"]


def _batch(images):
    """run_peaks inputs: peak rows in the given order (ids are input rows, sorted by part where r[18] matters), PAFs
    padded with zeros to one shape"""
    H = max(p.shape[0] for _, p in images)
    W = max(p.shape[1] for _, p in images)
    counts = np.array([len(r) for r, _ in images], np.int32)
    peaks = np.zeros((len(images), counts.max(), 5), np.float32)
    paf = np.zeros((len(images), H, W, 38), np.float32)
    for i, (r, p) in enumerate(images):
        peaks[i, :len(r)] = np.array(r, np.float32)
        paf[i, :p.shape[0], :p.shape[1]] = p
    return dict(peaks=peaks, counts=counts, paf=paf)


@functools.lru_cache(maxsize=None)
def _oracle(name, i):
    """(subset, peak line, connections per limb) of image i from the C restatement, and the people from
    util.oracle_people (the compiled reference where it was built)"""
    c = cases()[name]
    b = _batch(c["images"])
    peaks, paf = b["peaks"][i, :b["counts"][i]], b["paf"][i]
    port = util.port()
    sub, line = oracle.subset_of(port, peaks, c["h1"], paf.shape[1], paf)
    conns = {l: port.connections(l) for l in range(19)}
    ref_sub, ref_line = util.oracle_people(peaks, c["h1"], paf.shape[1], paf)
    return ref_sub, ref_line, sub, line, conns


# ---- the edges, proven on the CPU ------------------------------------------------------------------------------------------
def _arm_pair(rows):
    a = next(r for r in rows if r[4] == 1)
    b = next(r for r in rows if r[4] == 2)
    return a[:2], b[:2]


def _limb0_values(rows, paf):
    a, b = _arm_pair(rows)
    _, _, _, cells = pair_geometry(a, b)
    return a, b, [(paf[ly, lx, 12], paf[ly, lx, 13]) for lx, ly in cells]


def check_edge(name):
    """the case's quantity sits on its threshold (NumPy, the reference's operation order) and the oracle's people
    differ between the two sides"""
    c = cases()[name]
    kind = c["edge"][0]
    got = [len(_oracle(name, i)[0]) for i in range(len(c["images"]))]
    assert got == c["people"], f"{name}: the oracle finds {got} people, the construction {c['people']}"
    assert len(set(got)) > 1
    if kind in ("sample", "prefilter", "contraction", "criterion2", "penalty", "roundpaf"):
        for i, (rows, paf) in enumerate(c["images"]):   # the oracle's limb-0 decision is the one under test
            assert len(_oracle(name, i)[4][0]["cid1"]) == int(c["accept"][i]), (name, i)
    if kind == "sample":
        k = c["edge"][1]
        for i, want in enumerate((THR_SAMPLE, _up(THR_SAMPLE))):
            a, b, vals = _limb0_values(*c["images"][i])
            vx, vy, _, _ = pair_geometry(a, b)
            assert (vx, vy) == (1, 0)
            s = sample_score(vx, vy, *vals[k])
            assert s.view(np.uint32) == want.view(np.uint32)
            c1, c2 = pair_criteria(a, b, vals, c["h1"])
            assert c1 == THR_COUNT + i and c2 > 0 and accepted(a, b, vals, c["h1"]) == bool(i)
    elif kind == "prefilter":
        for i, (rows, paf) in enumerate(c["images"]):
            assert sum(r[4] == 1 for r in rows) * sum(r[4] == 2 for r in rows) > 2 * 256   # pass 1 runs
            a, b, vals = _limb0_values(rows, paf)
            vx, vy, _, _ = pair_geometry(a, b)
            mid = [sample_score(vx, vy, *vals[j]) > THR_SAMPLE for j in range(3, 7)]
            assert sum(mid) == int(c["accept"][i]) and (i == 4 or mid[i])
            assert all(sample_score(vx, vy, *vals[j]) == THR_SAMPLE for j in range(3, 7) if not mid[j - 3])
            assert pair_criteria(a, b, vals, c["h1"])[0] == THR_COUNT + int(c["accept"][i])
    elif kind == "contraction":
        k = c["edge"][1]
        for i, want in enumerate((THR_SAMPLE, _up(THR_SAMPLE))):
            a, b, vals = _limb0_values(*c["images"][i])
            vx, vy, _, _ = pair_geometry(a, b)
            assert (vx, vy) == (f32(0.6), f32(0.8))
            assert sample_score(vx, vy, *vals[k]).view(np.uint32) == want.view(np.uint32)
            assert fused_score(vx, vy, *vals[k]) > THR_SAMPLE   # contracted, the at side passes too
            assert pair_criteria(a, b, vals, c["h1"])[0] == THR_COUNT + i
    elif kind == "criterion2":
        for i in range(2):
            a, b, vals = _limb0_values(*c["images"][i])
            _, _, norm, _ = pair_geometry(a, b)
            assert float(norm) == c["h1"] and 0.5 * c["h1"] / float(norm) - 1.0 == -0.5
            c1, c2 = pair_criteria(a, b, vals, c["h1"])
            assert c1 == 10 and c2 == (0 if i == 0 else f32(2.0 ** -24))
    elif kind == "penalty":
        for i in range(2):
            a, b, vals = _limb0_values(*c["images"][i])
            _, _, norm, _ = pair_geometry(a, b)
            penalty = 0.5 * c["h1"] / float(norm) - 1.0
            assert (penalty == 0.0) if i == 0 else (penalty < 0.0)
            c1, c2 = pair_criteria(a, b, vals, c["h1"])
            assert c1 == THR_COUNT + 1 and (c2 > 0) == (i == 0)
    elif kind == "roundpaf":
        dx = c["edge"][1]
        ax, up, down = roundpaf_layout(dx)
        pos, cells = _positions(ax, dx)
        halves = [p for p in pos if float(p) % 1 == 0.5 and int(p) % 2 == 0]
        assert halves, f"dx {dx}: no sample on k + 0.5 with k even"
        st = f32(f32(dx) / f32(10))
        if dx in ROUNDPAF_INEXACT:   # the step is not exact, the position is rounded onto k + 0.5 by the float sum
            assert Fraction(float(st)) != Fraction(dx, 10)
        for i, good in enumerate((up, down)):
            rows, paf = c["images"][i]
            row = paf[A_ORIGIN[1], :, 12]
            n = sum(row[x] > THR_SAMPLE for x in cells)
            m = sum(row[int(np.rint(p))] > THR_SAMPLE for p in pos)
            assert (n > THR_COUNT >= m) if i == 0 else (m > THR_COUNT >= n)
    elif kind == "prune":
        limbs, closing, branch = PRUNE[c["edge"][1]]
        for i, want in enumerate((THR_HUMAN, _down(THR_HUMAN))):
            rows, _ = c["images"][i]
            ref_sub, _, sub, line, conns = _oracle(name, i)
            oc = {l: list(zip(conns[l]["cid1"], conns[l]["cid2"], conns[l]["score"])) for l in range(19) if len(conns[l]["cid1"])}
            assert sorted(oc) == sorted(limbs) and all(len(v) == 1 and v[0][2] == CONN for v in oc.values())
            before, kept, log = assemble(oc, dict(enumerate(line[2])))
            assert len(before) == 1 and before[0][19] == len({p for l in limbs for p in ce.LIMB_PARTS[l]})
            assert f32(before[0][18] / before[0][19]).view(np.uint32) == want.view(np.uint32)
            assert branch in log and (branch == "new" or log[limbs.index(max(limbs)) if branch == "extend" else -1] == branch)
            assert_bits_equal(np.array(kept, np.float32).reshape(-1, 20), sub, f"{name}: restated assembly vs oracle")
            assert_bits_equal(ref_sub, sub, f"{name}: oracle people")
    elif kind == "parts":
        for i in range(2):
            before, _, _ = _restated(c["images"][i][0], ((0, 2), (0, 2, 3))[i])
            assert before[0][19] == THR_PARTS - 1 + i and f32(before[0][18] / before[0][19]) > THR_HUMAN


@pytest.mark.parametrize("name", CASES)
def test_edge_cases_sit_on_their_edges(name):
    """no GPU: every scene is a CPU array and the oracle runs here"""
    check_edge(name)


def test_case_list_matches_the_builders():
    assert CASES == list(cases())


# ---- the GPU: run_peaks in a fresh process per stage 4 route, process_paf on its three upload routes ------------------------
ROUTES = {"per_pair": "0", "by_sample": "1000000"}   # EKP_BY_SAMPLE_MAX_PAIRS
UPLOADS = ("listed", "sparse", "dense")              # EKP_PROCESS_PAF_UPLOAD, read on every call


def _worker(spec_path, out_path):
    import torch

    import torch_ekpose_b200 as ek
    with open(spec_path) as f:
        spec = json.load(f)
    d = os.path.dirname(spec_path)
    out = {}
    pp = ek.PostProcessor(device=0, max_batch=spec["max_batch"], max_h=8, max_w=8, max_peaks=128, max_humans=32)
    for case in spec["cases"]:
        name, h1 = case["name"], case["h1"]
        with np.load(os.path.join(d, name + ".npz")) as z:
            b = {k: z[k] for k in z.files}
        try:
            pp.run_peaks(torch.from_numpy(b["peaks"]).cuda(), torch.from_numpy(b["counts"]).cuda(),
                         torch.from_numpy(b["paf"]).cuda(), h1=h1)
            res = pp.results()
            out[name + "/num_humans"], out[name + "/subset"] = res["num_humans"], res["subset"]
            for route in UPLOADS:
                os.environ["EKP_PROCESS_PAF_UPLOAD"] = route
                pf = ek.pafprocess
                for i, n in enumerate(b["counts"]):
                    peaks = b["peaks"][i, :n]
                    pf.process_paf(peaks[None], np.zeros((h1, 1, 19), np.float32), b["paf"][i])
                    nh = pf.get_num_humans()
                    key = f"{name}/{route}/{i}/"
                    out[key + "num_humans"] = np.array(nh)
                    out[key + "cids"] = np.array([[pf.get_part_cid(h, p) for p in range(18)] for h in range(nh)], np.int32).reshape(nh, 18)
                    out[key + "scores"] = np.array([pf.get_score(h) for h in range(nh)], np.float32)
                    out[key + "line"] = np.array([(pf.get_part_x(k), pf.get_part_y(k)) for k in range(n)], np.int32).reshape(n, 2)
                    out[key + "line_score"] = np.array([pf.get_part_score(k) for k in range(n)], np.float32)
            os.environ.pop("EKP_PROCESS_PAF_UPLOAD", None)
        except Exception as e:   # a refused launch is this case's finding; the other cases still run
            out[name + "/error"] = np.array(f"{type(e).__name__}: {e}")
    pp.close()
    np.savez(out_path, **out)


_WORKER = "import sys; from tests.test_threshold_edges import _worker; _worker(sys.argv[1], sys.argv[2])"


@pytest.fixture(scope="module")
def run_route(tmp_path_factory):
    done = {}

    def run(route):
        if route not in done:
            d = tmp_path_factory.mktemp(route)
            specs = []
            for name in CASES:
                c = cases()[name]
                np.savez(d / (name + ".npz"), **_batch(c["images"]))
                specs.append(dict(name=name, h1=c["h1"]))
            with open(d / "spec.json", "w") as f:
                json.dump(dict(cases=specs, max_batch=max(len(c["images"]) for c in cases().values())), f)
            env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
            for k in ("EKP_GRAPHS", "EKP_LEAN_TILED", "EKP_PROCESS_PAF_UPLOAD", "EKP_DEVICE"):
                env.pop(k, None)
            env["EKP_BY_SAMPLE_MAX_PAIRS"] = ROUTES[route]
            r = subprocess.run([sys.executable, "-c", _WORKER, str(d / "spec.json"), str(d / "out.npz")], capture_output=True,
                               text=True, env=env, cwd=ROOT, timeout=1200)
            assert r.returncode == 0, f"worker for {route} exited {r.returncode}:\n{r.stderr[-3000:]}"
            with np.load(d / "out.npz") as z:
                done[route] = {k: z[k] for k in z.files}
        return done[route]
    return run


@pytest.mark.gpu
@pytest.mark.parametrize("route", list(ROUTES))
@pytest.mark.parametrize("name", CASES)
def test_edge_equals_the_oracle(run_route, route, name):
    """run_peaks and the host process_paf (listed, sparse, dense uploads): people bit for bit equal to the oracle's on
    both sides of the edge"""
    out = run_route(route)
    assert name + "/error" not in out, f"{name}: {out[name + '/error']}"
    c = cases()[name]
    for i in range(len(c["images"])):
        sub, line = _oracle(name, i)[:2]
        assert len(sub) == c["people"][i]
        m = int(out[name + "/num_humans"][i])
        assert m == len(sub), f"{name} image {i}: run_peaks finds {m} people, the oracle {len(sub)}"
        assert_bits_equal(out[name + "/subset"][i, :m], sub, f"{name} image {i} run_peaks subset")
        for up in UPLOADS:
            key = f"{name}/{up}/{i}/"
            nh = int(out[key + "num_humans"])
            assert nh == len(sub), f"{name} image {i} process_paf ({up}): {nh} people, the oracle {len(sub)}"
            assert np.array_equal(out[key + "cids"], sub[:, :18].astype(np.int32)), f"{name} image {i} process_paf ({up})"
            assert_bits_equal(out[key + "scores"], (sub[:, 18] / sub[:, 19]).astype(np.float32), f"{name} {up} scores")
            assert np.array_equal(out[key + "line"][:, 0], line[0]) and np.array_equal(out[key + "line"][:, 1], line[1])
            assert_bits_equal(out[key + "line_score"], line[2], f"{name} {up} getter table scores")


# ---- the constants the cases sit on ----------------------------------------------------------------------------------------
def test_score_thresholds_are_the_ones_the_cases_sit_on():
    """a changed threshold, a third scoring copy or FMA contraction switched back on must fail here instead of silently
    moving the cases off their edges"""
    orc = ce._source("oracle", "paf_oracle.c")
    assert f32(ce._const(orc, r"OKP_THRESH_VECTOR_SCORE = ([0-9.]+);")) == THR_SAMPLE
    assert ce._const(orc, r"OKP_THRESH_VECTOR_CNT1 = (\d+);") == THR_COUNT
    assert ce._const(orc, r"OKP_THRESH_PART_CNT = (\d+);") == THR_PARTS
    assert f32(ce._const(orc, r"OKP_THRESH_HUMAN_SCORE = ([0-9.]+);")) == THR_HUMAN
    conn = ce._source("torch_ekpose_b200", "csrc", "paf_connect.cu")
    # score_pair, score_pairs_by_sample and pass 1 (pair_may_pass): one sample threshold each, strict
    assert len(re.findall(r"\bs > 0\.05f", conn)) == 2 and len(re.findall(r"\)\) > 0\.05f;", conn)) == 1
    assert len(re.findall(r"0\.05f", conn)) == 3
    assert len(re.findall(r"criterion1 > 6 && (criterion2|crit) > 0\.0f", conn)) == 2
    assert len(re.findall(r"for \(int k = 0; k < 4; k\+\+\)", conn)) == 2 and "const int i = 3 + k;" in conn
    assert "fmaf" not in conn and "__fmaf" not in conn
    asm = ce._source("torch_ekpose_b200", "csrc", "assemble.cu")
    assert len(re.findall(r"c < 4\.0f \|\| __fdiv_rn\(sc, c\) < 0\.3f", asm)) == 1
    mk = ce._source("torch_ekpose_b200", "csrc", "Makefile")
    assert re.search(r"^NVCCFLAGS = .*-fmad=false", mk, re.M)
    assert ce.LIMB_CH[0] == 12 and ce.LIMB_PARTS[0] == (1, 2)
    # the tracker: the shared memory and the working-set layout that track_cache_cap() restates (the cache_* case's edge)
    trk = ce._source("torch_ekpose_b200", "csrc", "track.cu")
    assert ce._const(trk, r"static const size_t kTrackSmemMax = ([^;]+);") == TRACK_SMEM_MAX
    assert "sizeof(TrackSlot) == 160 && sizeof(PersonPose) == 152" in trk
    body = trk[trk.index("HD size_t track_work_layout"):trk.index("t.cache_cap = cache_cap;")]
    assert re.findall(r"take\(([^;]+)\);", body) == [
        "sizeof(double) * kCoco", "sizeof(TrackSlot) * max_tracks", "sizeof(PersonPose) * max_humans"] + \
        ["sizeof(int) * max_tracks"] * 5 + ["sizeof(int) * max_humans"] * 2 + ["sizeof(int) * 4", "sizeof(double) * cache_cap"]
    assert "const size_t room = (kTrackSmemMax - rest) / sizeof(double);" in trk
    assert "return (int) (room < (size_t) max_humans * max_tracks ? room : (size_t) max_humans * max_tracks);" in trk
    assert track_cache_cap(512, 512) == 7276


# ---- D: the tracker ----------------------------------------------------------------------------------------------------
# Every pose has the same four COCO keypoints (reference parts ORDER_COCO[:4]) in a 3 x 3 px box (area 9) around its base;
# bases are 200 px apart.  A person's keypoint either sits exactly on a track's keypoint (exp(0) = 1) or 200 px or more
# off (exp underflows to exactly 0), so every similarity is k / 4, exact in float64 on every device, and
# Oracle(check_margin=False) pins the ids.
KP_PARTS = [int(p) for p in tt.ORDER_COCO[:4]]
KP_OFF = [(0, 0), (2, 0), (0, 2), (2, 2)]
FAR = None
TRACK_SMEM_MAX = 227 * 1024      # track.cu kTrackSmemMax


def _base(b):
    return (100 + 200 * (b % 24), 100 + 200 * (b // 24)) if b is not FAR else (90000, 90000)


def _pose(sources):
    """one person row [18, 4]: keypoint j at the position of base sources[j]'s keypoint j"""
    row = np.zeros((18, 4), np.int32)
    row[:, 3] = -1
    for j, (part, b) in enumerate(zip(KP_PARTS, sources)):
        x, y = _base(b)
        row[part] = (x + KP_OFF[j][0], y + KP_OFF[j][1], 0, part)
    return row


def _frames(frames, mh):
    """frames [[row, ...], ...] -> (num [F], parts [F, mh, 18, 4])"""
    num = np.array([len(f) for f in frames], np.int32)
    parts = np.zeros((len(frames), mh, 18, 4), np.int32)
    for i, f in enumerate(frames):
        for p, r in enumerate(f):
            parts[i, p] = r
    return num, parts


def track_cache_cap(mh, mt):
    """track.cu's track_cache_cap: the shared-memory similarity matrix gets what track_work_layout's other arrays leave"""
    r16 = lambda b: (b + 15) & ~15   # noqa: E731
    rest = sum(r16(b) for b in (8 * 17, 160 * mt, 152 * mh, 4 * mt, 4 * mt, 4 * mt, 4 * mt, 4 * mt, 4 * mh, 4 * mh, 16))
    return min((TRACK_SMEM_MAX - rest) // 8, mh * mt)


def _same(n):
    return [_pose([b] * 4) for b in range(n)]


def _track_cases():
    """name -> list of variants dict(mh, mt, min_oks, max_age, calls: [[frame rows, ...] per call]); the variants of one
    name are the two sides of its edge"""
    C = {}
    for s in (1.0, 0.75, 0.5, 0.25, 0.0):   # min_oks on the similarity (accepted) and one float above it (a new track)
        k = int(4 * s)
        later = _pose([0] * k + [FAR] * (4 - k))
        C[f"min_oks_{s}"] = [dict(mh=4, mt=4, min_oks=m, max_age=30, calls=[[_same(1)], [[later]]])
                             for m in (f32(s), _up(f32(s)))]
    rng = np.random.default_rng(7)
    src = [list(rng.choice([FAR] + list(range(40)), 4)) for _ in range(40)]
    src = [[FAR if b == FAR else int(b) for b in s] for s in src]
    perm = rng.permutation(40)
    # min_oks 0: every pair competes, ties at every level; more than 32 people and tracks
    C["ties_40x40"] = [dict(mh=48, mt=48, min_oks=f32(0), max_age=30, calls=[[_same(40)], [[_pose(src[p]) for p in order]]])
                       for order in (range(40), perm)]
    chain = [_pose([0, 0, FAR, FAR])] + [_pose([i - 1, i - 1, i, i]) for i in range(1, 40)]
    C["chain_40"] = [dict(mh=40, mt=40, min_oks=f32(0.5), max_age=30, calls=[[_same(40)], [chain]])]
    for age in (0, 1, 30):   # a person missing for max_age frames keeps the id, for max_age + 1 gets a new one
        C[f"expiry_{age}"] = [dict(mh=2, mt=4, min_oks=f32(0.5), max_age=age,
                                   calls=[[_same(1)]] + ([[[]] * gap] if gap else []) + [[_same(1)]]) for gap in (age, age + 1)]
    C["evict_ties"] = [dict(mh=4, mt=4, min_oks=f32(0.5), max_age=30,
                            calls=[[_same(4)], [[_pose([4] * 4), _pose([5] * 4)]], [_same(4)]])]
    cap = track_cache_cap(512, 512)
    variants = []
    for P, L in ((68, 107), (19, 383)):
        assert P * L in (cap, cap + 1)
        r = np.random.default_rng(P)
        people = [_pose([FAR if b < 0 else int(b) for b in r.integers(-1, L, 4)]) for _ in range(P)]
        variants.append(dict(mh=512, mt=512, min_oks=f32(0.25), max_age=30, calls=[[_same(L)], [people]]))
    C["cache_7276_7277"] = variants
    return C


@functools.lru_cache(maxsize=None)
def track_cases():
    return _track_cases()


TRACK_CASES = [f"min_oks_{s}" for s in (1.0, 0.75, 0.5, 0.25, 0.0)] + ["ties_40x40", "chain_40"] + \
              [f"expiry_{a}" for a in (0, 1, 30)] + ["evict_ties", "cache_7276_7277"]


def _oracle_ids(v, record=None):
    """ids per call from Oracle(check_margin=False); record: a list that gets every similarity matrix"""
    o = tt.Oracle(1, v["mt"], v["min_oks"], v["max_age"], check_margin=False)
    orig = tt.oks_matrix

    def rec(*a):
        s = orig(*a)
        record.append(s)
        return s
    if record is not None:
        tt.oks_matrix = rec
    try:
        return [o.update(*_frames(c, v["mh"])) for c in v["calls"]]
    finally:
        tt.oks_matrix = orig


def _greedy(sim, tids, reverse):
    """the greedy walk over pairs with sim >= 0, ties by (track id, row), or both reversed"""
    sg = -1 if reverse else 1
    pairs = sorted((-sim[p, k], sg * tids[k], sg * p, p, k) for p in range(sim.shape[0]) for k in range(sim.shape[1]))
    ids, taken = [-1] * sim.shape[0], set()
    for _, _, _, p, k in pairs:
        if ids[p] < 0 and k not in taken:
            ids[p] = tids[k]
            taken.add(k)
    return ids


def _rounds(sim, min_oks):
    """rounds of mutual first choices track.cu needs for one frame (ties by track index = id, row)"""
    P, L = sim.shape
    pm, tm, n = [-1] * P, [-1] * L, 0
    while True:
        n += 1
        pb = [max((k for k in range(L) if tm[k] < 0 and sim[p, k] >= min_oks), key=lambda k: (sim[p, k], -k), default=-1)
              if pm[p] < 0 else -1 for p in range(P)]
        tb = [max((p for p in range(P) if pm[p] < 0 and sim[p, k] >= min_oks), key=lambda p: (sim[p, k], -p), default=-1)
              for k in range(L)]
        pending = False
        for p in range(P):
            if pm[p] < 0 and pb[p] >= 0:
                if tb[pb[p]] == p:
                    pm[p], tm[pb[p]] = pb[p], p
                else:
                    pending = True
        if not pending:
            return n


def check_track_edge(name):
    vs = track_cases()[name]
    sims = []
    ids = [_oracle_ids(v, sims) for v in vs]
    assert all(np.isin(s, [0, 0.25, 0.5, 0.75, 1]).all() for s in sims), f"{name}: a similarity that is not k / 4"
    if len(vs) == 2 and not name.startswith(("ties", "cache")):
        assert not all(np.array_equal(a, b) for a, b in zip(*ids)), f"{name}: the two sides give the same ids"
    if name.startswith("min_oks"):
        s = float(name.rsplit("_", 1)[1])
        assert sims[-1][0, 0] == s == vs[0]["min_oks"] and np.float64(vs[1]["min_oks"]) > s
        assert ids[0][1].tolist() == [[0, -1, -1, -1]] and ids[1][1].tolist() == [[1, -1, -1, -1]]
    elif name == "ties_40x40":
        s1 = [s for s in sims if s.shape == (40, 40)]
        assert len(s1) == 2
        for s in s1:   # the tie-break decides: reversed, the ids differ, and ties exist on both sides
            assert _greedy(s, list(range(40)), False) != _greedy(s, list(range(40)), True)
            assert any(len(set(r[r > 0])) < len(r[r > 0]) for r in s) and any(len(set(c[c > 0])) < len(c[c > 0]) for c in s.T)
    elif name == "chain_40":
        assert _rounds(sims[-1], 0.5) == 40 and ids[0][1][0, :40].tolist() == list(range(40))
    elif name.startswith("expiry"):
        assert ids[0][-1][0, 0] == 0 and ids[1][-1][0, 0] == 1
    elif name == "evict_ties":
        assert [i[:, :4].tolist() for i in ids[0]] == [[[0, 1, 2, 3]], [[4, 5, -1, -1]], [[6, 7, 2, 3]]]
    elif name.startswith("cache"):
        cap = track_cache_cap(512, 512)
        assert [len(v["calls"][1][0]) * len(v["calls"][0][0]) for v in vs] == [cap, cap + 1]
        assert all((i[1] < len(v["calls"][0][0])).any() for v, i in zip(vs, ids))   # people continue tracks
    return ids


@pytest.mark.parametrize("name", TRACK_CASES)
def test_tracker_edge_host_hook_equals_the_oracle(name):
    """no GPU: the edge is proven from the oracle, and the kernel's own code (ekp_debug_track_host, one thread) gives its ids"""
    ids = check_track_edge(name)
    for v, want in zip(track_cases()[name], ids):
        st = tt.host_state(1, v["mt"])
        for call, w in zip(v["calls"], want):
            num, parts = _frames(call, v["mh"])
            assert np.array_equal(tt.host_track(num, parts, st, 1, v["mt"], v["min_oks"], v["max_age"]), w), name


@pytest.mark.gpu
@pytest.mark.parametrize("name", TRACK_CASES)
def test_tracker_edge_equals_the_oracle(name):
    """Tracker.update on the device, the frames split across calls as listed"""
    import torch

    import torch_ekpose_b200 as ek
    for v, want in zip(track_cases()[name], [_oracle_ids(v) for v in track_cases()[name]]):
        tr = ek.Tracker(0, max_tracks=v["mt"], min_oks=float(v["min_oks"]), max_age=v["max_age"])
        for call, w in zip(v["calls"], want):
            got = tr.update(tt._tables(torch, *_frames(call, v["mh"]))).cpu().numpy()
            assert np.array_equal(got, w), (name, got.tolist(), w.tolist())
