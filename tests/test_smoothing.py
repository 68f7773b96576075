"""Keypoints smoothed per track id (ekp_smooth_humans / Smoother) against a NumPy restatement of the specification in
include/ekpose_b200.h ("smoothing"): the Restatement below, pinned to a scalar transcription of the One Euro filter of
Casiez, Roussel and Vogel (CHI 2012) and to hand-worked cases.  On the CPU, ekp_debug_smooth_host (the kernel's own code
run serially) must equal it bit for bit on thousands of random sequences whose ids come from tests/test_tracking.py's
Oracle; on the GPU, Smoother.update must."""
import ctypes
import itertools
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from torch_ekpose_b200 import _lib
from tests.test_tracking import Oracle, _person, random_sequences

PI2 = 2.0 * math.pi


class Restatement:
    """The specification, one sequence at a time.  An entry is a dict: id, last (frame of the last use) and, per
    (part, axis) component c = 2 * part + axis, xh / dxh float64 and fl (frame of the last sample, -1: none)."""

    def __init__(self, n_seq=1, max_tracks=256, max_age=30, fps=30.0, min_cutoff=1.0, beta=0.007, d_cutoff=1.0):
        self.max_tracks, self.max_age = max_tracks, max_age
        self.fps, self.min_cutoff, self.beta = float(fps), float(min_cutoff), float(beta)
        self.tau_d = 1.0 / (PI2 * float(d_cutoff))
        self.seq = [dict(frame=0, entries={}) for _ in range(n_seq)]
        self.evictions = self.tied_evictions = 0   # the latter: another candidate had the same last_seen

    def _filter(self, e, raw, on, f):
        """one row's 36 components: raw int [36], on bool [36] at frame f; returns xh after the step"""
        x = raw.astype(np.float64)
        te = (f - e["fl"]).astype(np.float64) / self.fps     # components without a sample compute garbage, unused
        a_d = 1.0 / (1.0 + self.tau_d / te)
        dx = (x - e["xh"]) / te
        dxh = a_d * dx + (1.0 - a_d) * e["dxh"]
        c = self.min_cutoff + self.beta * np.abs(dxh)
        tau = 1.0 / (PI2 * c)
        a = 1.0 / (1.0 + tau / te)
        xh = a * x + (1.0 - a) * e["xh"]
        first, step = on & (e["fl"] < 0), on & (e["fl"] >= 0)
        e["xh"] = np.where(first, x, np.where(step, xh, e["xh"]))
        e["dxh"] = np.where(first, 0.0, np.where(step, dxh, e["dxh"]))
        e["fl"] = np.where(on, f, e["fl"])
        return e["xh"]

    def _frame(self, S, rows, ids):
        """rows int [P, 18, 4], ids int [P] -> xy float32 [P, 18, 2]"""
        f = S["frame"]
        ent = S["entries"] = {i: e for i, e in S["entries"].items() if f - e["last"] <= self.max_age + 1}
        P = len(rows)
        on = np.repeat(rows[:, :, 3] >= 0, 2, axis=1)                       # [P, 36]
        raw = rows[:, :, :2].reshape(P, 36).astype(np.int64)
        out = np.where(on, raw, 0).astype(np.float64)
        use = {}
        for p in range(P):                     # rows whose id has an entry first
            if ids[p] >= 0 and int(ids[p]) in ent:
                use[p] = ent[int(ids[p])]
                use[p]["last"] = f
        for p in range(P):                     # then births, in row order
            i = int(ids[p])
            if i < 0 or p in use:
                continue
            if len(ent) == self.max_tracks:
                cand = sorted((e["last"], k) for k, e in ent.items() if e["last"] != f)
                del ent[cand[0][1]]
                self.evictions += 1
                self.tied_evictions += len(cand) > 1 and cand[1][0] == cand[0][0]
            ent[i] = use[p] = dict(id=i, last=f, xh=np.zeros(36), dxh=np.zeros(36), fl=np.full(36, -1, np.int64))
        for p, e in use.items():
            out[p] = np.where(on[p], self._filter(e, raw[p], on[p], f), 0.0)
        S["frame"] += 1
        return out.astype(np.float32).reshape(P, 18, 2)

    def update(self, num_humans, parts, ids):
        """num_humans [n], parts [n, max_humans, 18, 4] int, ids [n, max_humans] -> xy float32 [n, max_humans, 18, 2]"""
        parts = np.asarray(parts).reshape(len(num_humans), -1, 18, 4)
        n, mh = parts.shape[:2]
        F = n // len(self.seq)
        out = np.zeros((n, mh, 18, 2), np.float32)
        for i in range(n):
            P = min(max(int(num_humans[i]), 0), mh)
            out[i, :P] = self._frame(self.seq[i // F], parts[i, :P], np.asarray(ids[i, :P]))
        return out

    def live(self, s=0):
        """{id: last} of sequence s's entries that are still live at its next frame"""
        S = self.seq[s]
        return {i: e["last"] for i, e in S["entries"].items() if S["frame"] - e["last"] <= self.max_age + 1}


class PaperOneEuro:
    """An independent scalar transcription of the paper's Algorithm 1 (timestamped samples, rate = 1 / (T_i - T_i-1),
    alpha = 1 / (1 + tau / T_e), T_e = 1 / rate, the derivative taken against the previous filtered value)."""

    def __init__(self, mincutoff, beta, dcutoff):
        self.mincutoff, self.beta, self.dcutoff = mincutoff, beta, dcutoff
        self.xprev = self.dxprev = self.tprev = None

    @staticmethod
    def alpha(rate, cutoff):
        tau = 1.0 / (2 * math.pi * cutoff)
        te = 1.0 / rate
        return 1.0 / (1.0 + tau / te)

    def __call__(self, x, t):
        if self.xprev is None:
            self.xprev, self.dxprev, self.tprev = x, 0.0, t
            return x
        rate = 1.0 / (t - self.tprev)
        dx = (x - self.xprev) * rate
        ad = self.alpha(rate, self.dcutoff)
        edx = ad * dx + (1 - ad) * self.dxprev
        cutoff = self.mincutoff + self.beta * abs(edx)
        a = self.alpha(rate, cutoff)
        xh = a * x + (1 - a) * self.xprev
        self.xprev, self.dxprev, self.tprev = xh, edx, t
        return xh


def one_person(xs, present=None):
    """tables of one person over len(xs) frames: part 0's x takes the values xs, every other coordinate is 100"""
    F = len(xs)
    parts = np.zeros((F, 1, 18, 4), np.int32)
    parts[:, 0, :, :2] = 100
    parts[:, 0, :, 3] = np.arange(18)
    parts[:, 0, 0, 0] = xs
    if present is not None:
        parts[~np.asarray(present), 0, 0, 3] = -1
    return np.ones(F, np.int32), parts, np.zeros((F, 1), np.int32)


def host_state(n_seq, max_tracks):
    nb = _lib.lib.ekp_smooth_state_bytes(n_seq, max_tracks)
    return np.zeros(nb // 8, np.float64)   # 8-byte aligned, zero = reset


def host_smooth(num, parts, ids, state, n_seq, max_tracks, max_age, fps=30.0, min_cutoff=1.0, beta=0.007, d_cutoff=1.0):
    n, mh = parts.shape[:2]
    xy = np.full((n, mh, 18, 2), np.nan, np.float32)   # dirty: every element must be written
    num = np.ascontiguousarray(num, np.int32)
    parts = np.ascontiguousarray(parts, np.int32)
    ids = np.ascontiguousarray(ids, np.int32)
    _lib.check(_lib.lib.ekp_debug_smooth_host(num.ctypes.data, parts.ctypes.data, ids.ctypes.data, n, mh, state.ctypes.data,
                                              n_seq, max_tracks, max_age, fps, min_cutoff, beta, d_cutoff, xy.ctypes.data))
    return xy


def state_live(state, s, max_tracks):
    """({id: last_seen} of the entries sequence s holds, its frame count) from a host state (smooth.cu's layout: a 16-byte
    head with the frame count, then (uint32 tag = id + 1, 0 = free; int32 last_seen) per entry, then the filter values)"""
    seq_bytes = _lib.lib.ekp_smooth_state_bytes(1, max_tracks)
    raw = state.view(np.uint8)[s * seq_bytes:(s + 1) * seq_bytes]
    frame = int(raw[:4].view(np.int32)[0])
    ent = raw[16:16 + 8 * max_tracks].view(np.int32).reshape(max_tracks, 2)
    return {int(t) - 1: int(l) for t, l in ent if t != 0}, frame


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


# ---- CPU: the restatement ------------------------------------------------------------------------------------------------
def test_restatement_hand_worked_cases():
    R = Restatement(fps=30.0, min_cutoff=1.0, beta=0.007, d_cutoff=1.0)
    # the first sample is the raw value
    xy = R.update(*one_person([137]))
    assert xy[0, 0, 0, 0] == 137.0 and xy[0, 0, 0, 1] == 100.0
    # a constant signal stays constant (float32 output exactly the input, every frame)
    R = Restatement()
    xy = R.update(*one_person([250] * 40))
    assert (xy[:, 0, :, :] == np.where(np.arange(36).reshape(18, 2) == 0, 250.0, 100.0)).all()
    # one step by hand: a jump of 10 px after one frame
    x0, x1, te = 100.0, 110.0, 1.0 / 30.0
    a_d = 1.0 / (1.0 + (1.0 / (PI2 * 1.0)) / te)
    dxh = a_d * ((x1 - x0) / te) + (1.0 - a_d) * 0.0
    a = 1.0 / (1.0 + (1.0 / (PI2 * (1.0 + 0.007 * abs(dxh)))) / te)
    want = a * x1 + (1.0 - a) * x0
    assert 100.0 < want < 110.0
    assert Restatement().update(*one_person([100, 110]))[1, 0, 0, 0] == np.float32(want)
    # a gap of g frames (the part absent in between) uses te = g / fps
    for g in (2, 5):
        te = g / 30.0
        a_d = 1.0 / (1.0 + (1.0 / (PI2 * 1.0)) / te)
        dxh = a_d * ((x1 - x0) / te)
        a = 1.0 / (1.0 + (1.0 / (PI2 * (1.0 + 0.007 * abs(dxh)))) / te)
        want_g = a * x1 + (1.0 - a) * x0
        xs = [100] + [0] * (g - 1) + [110]
        got = Restatement().update(*one_person(xs, present=[True] + [False] * (g - 1) + [True]))
        assert got[-1, 0, 0, 0] == np.float32(want_g) and want_g > want, g   # a longer gap follows the jump further
        assert (got[1:-1, 0, 0] == 0).all()                                   # absent parts are 0
    # min_cutoff 1e300, beta 0: alpha == 1, the raw coordinates exactly
    rng = np.random.default_rng(0)
    xs = rng.integers(-5000, 5000, 50)
    assert np.array_equal(Restatement(min_cutoff=1e300, beta=0.0).update(*one_person(xs))[:, 0, 0, 0], xs.astype(np.float32))


def test_restatement_equals_the_papers_filter_on_random_signals():
    rng = np.random.default_rng(1)
    for _ in range(200):
        fps = float(rng.choice([15.0, 30.0, 60.0, 120.0]))
        mc, beta, dc = float(rng.uniform(0.05, 5)), float(rng.choice([0.0, 0.007, 0.1, 1.0])), float(rng.uniform(0.1, 3))
        F = int(rng.integers(2, 60))
        xs = np.cumsum(rng.integers(-20, 21, F)) + 500
        present = rng.random(F) < 0.7
        present[0] = True
        got = Restatement(fps=fps, min_cutoff=mc, beta=beta, d_cutoff=dc).update(*one_person(xs, present))[:, 0, 0, 0]
        paper = PaperOneEuro(mc, beta, dc)
        for f in range(F):
            if present[f]:
                want = paper(float(xs[f]), f / fps)
                assert abs(got[f] - want) <= 1e-4 * max(1.0, abs(want)), (f, got[f], want)   # float32 output of the same filter


# ---- CPU: the host hook against the restatement --------------------------------------------------------------------------
def _fuzz_case(rng):
    max_humans = int(rng.integers(1, 7))
    max_tracks = int(rng.integers(max_humans, max_humans + 5))
    n_seq = int(rng.integers(1, 4))
    max_age = int(rng.integers(0, 4))
    fps = float(rng.choice([10.0, 30.0, 60.0]))
    mc, beta, dc = float(rng.choice([0.3, 1.0, 4.0])), float(rng.choice([0.0, 0.007, 0.3])), float(rng.choice([0.5, 1.0, 2.0]))
    return max_humans, max_tracks, n_seq, max_age, fps, mc, beta, dc


def test_host_hook_equals_restatement_on_random_sequences():
    """ids from the tracker's Oracle with the same (n_seq, max_tracks, max_age), so entries are born, expire at the
    tracker's edge and are evicted (ties included: several tracks are born in one frame); some rows get id -1; the frames
    go in over random splits into calls."""
    rng = np.random.default_rng(7)
    done = frames = negatives = evictions = ties = 0
    while done < 2000:
        mh, mt, n_seq, max_age, fps, mc, beta, dc = _fuzz_case(rng)
        F = int(rng.integers(2, 13))
        num, parts = random_sequences(rng, n_seq, F, mh)
        ids = Oracle(n_seq, mt, 0.5, max_age, check_margin=False).update(num, parts)
        for i in range(len(num)):
            for p in range(min(int(num[i]), mh)):
                if rng.random() < 0.05:
                    ids[i, p] = -1
                    negatives += 1
        R = Restatement(n_seq, mt, max_age, fps, mc, beta, dc)
        st = host_state(n_seq, mt)
        at = 0
        while at < F:   # a random split of the frames into calls: the same frames of every sequence in each
            k = int(rng.integers(1, F - at + 1))
            sel = np.concatenate([np.arange(s * F + at, s * F + at + k) for s in range(n_seq)])
            want = R.update(num[sel], parts[sel], ids[sel])
            got = host_smooth(num[sel], parts[sel], ids[sel], st, n_seq, mt, max_age, fps, mc, beta, dc)
            assert np.array_equal(bits(got), bits(want)), (mh, mt, n_seq, max_age, at, k)
            at += k
        evictions += R.evictions
        ties += R.tied_evictions
        frames += len(num)
        done += n_seq
    assert frames > 10000 and negatives > 500 and evictions > 500 and ties > 50, (frames, negatives, evictions, ties)


def test_host_hook_state_carries_across_every_split_of_the_frames():
    rng = np.random.default_rng(11)
    F = 7
    for _ in range(6):
        num, parts = random_sequences(rng, 1, F, 4)
        ids = Oracle(1, 6, 0.5, 1, check_margin=False).update(num, parts)
        whole = host_smooth(num, parts, ids, host_state(1, 6), 1, 6, 1)
        assert np.array_equal(bits(whole), bits(Restatement(1, 6, 1).update(num, parts, ids)))
        for cuts in itertools.product([0, 1], repeat=F - 1):   # all 64 compositions of 7 frames
            bounds = [0] + [i + 1 for i, c in enumerate(cuts) if c] + [F]
            st = host_state(1, 6)
            got = np.concatenate([host_smooth(num[a:b], parts[a:b], ids[a:b], st, 1, 6, 1) for a, b in zip(bounds, bounds[1:])])
            assert np.array_equal(bits(got), bits(whole)), bounds


def test_live_entries_equal_the_trackers_live_tracks_after_every_frame():
    rng = np.random.default_rng(13)
    checked = 0
    for _ in range(150):
        mh, mt, n_seq, max_age, *_ = _fuzz_case(rng)
        F = int(rng.integers(4, 16))
        num, parts = random_sequences(rng, n_seq, F, mh)
        o = Oracle(n_seq, mt, 0.5, max_age, check_margin=False)
        R = Restatement(n_seq, mt, max_age)
        st = host_state(n_seq, mt)
        for t in range(F):   # one frame of every sequence per call
            sel = np.arange(n_seq) * F + t
            ids = o.update(num[sel], parts[sel])
            R.update(num[sel], parts[sel], ids)
            host_smooth(num[sel], parts[sel], ids, st, n_seq, mt, max_age)
            for s in range(n_seq):
                S = o.seq[s]
                tracks = {tr["id"]: tr["last"] for tr in S["tracks"] if S["frame"] - tr["last"] <= max_age + 1}
                hook, frame = state_live(st, s, mt)
                hook = {i: l for i, l in hook.items() if frame - l <= max_age + 1}
                assert R.live(s) == tracks == hook, (t, s)
                checked += 1
    assert checked > 1000


def test_expiry_at_max_age_plus_one_and_plus_two_frames():
    """id 0 seen at frame 0, then unseen until frame k: its filter continues at k = max_age + 1 and restarts (the raw
    value) at k = max_age + 2."""
    for max_age in (0, 1, 3):
        for k in (max_age + 1, max_age + 2):
            xs = [100] + [0] * (k - 1) + [160]
            num, parts, ids = one_person(xs)
            num[1:k] = 0
            got = host_smooth(num, parts, ids, host_state(1, 2), 1, 2, max_age)
            assert np.array_equal(bits(got), bits(Restatement(1, 2, max_age).update(num, parts, ids)))
            assert (got[-1, 0, 0, 0] == 160.0) == (k == max_age + 2), (max_age, k)


def test_births_follow_lookups_and_evict_the_oldest_then_lowest_id():
    p = _person(np.random.default_rng(2), 300, 300, 100)

    def frames(id_rows):
        F = len(id_rows)
        mh = max(len(r) for r in id_rows)
        num = np.array([len(r) for r in id_rows], np.int32)
        parts = np.zeros((F, mh, 18, 4), np.int32)
        ids = np.full((F, mh), -1, np.int32)
        for t, r in enumerate(id_rows):
            for q, i in enumerate(r):
                parts[t, q] = p
                parts[t, q, :, :2] += 10 * t + 3 * q   # moving, so a continued filter differs from the raw value
                ids[t, q] = i
        return num, parts, ids

    def restarted(id_rows):
        num, parts, ids = frames(id_rows)
        got = host_smooth(num, parts, ids, host_state(1, 2), 1, 2, 30)
        assert np.array_equal(bits(got), bits(Restatement(1, 2, 30).update(num, parts, ids)))
        raw = parts[..., :2].astype(np.float32)
        return [bool((got[-1, q] == raw[-1, q]).all()) for q in range(int(num[-1]))]

    # ids 5 and 3 both last seen at frame 0; id 7 evicts 3 (the tie goes to the lower id), so 3 restarts, 5 continues
    assert restarted([[5, 3], [7], [5, 3]]) == [False, True]
    # frame 2: row 0 is a birth, row 1 continues id 1 (the oldest entry): the birth evicts id 2 instead
    assert restarted([[1, 2], [2], [9, 1]]) == [True, False]


def test_large_tables_cross_the_chunk_of_frames():
    """512 entries leave room for 64 frames of the inverse map per chunk: 100 frames take two chunks."""
    rng = np.random.default_rng(5)
    num, parts = random_sequences(rng, 1, 100, 40, dup=False)
    ids = Oracle(1, 512, 0.5, 30, check_margin=False).update(num, parts)
    got = host_smooth(num, parts, ids, host_state(1, 512), 1, 512, 30)
    assert np.array_equal(bits(got), bits(Restatement(1, 512, 30).update(num, parts, ids)))


def test_huge_min_cutoff_without_beta_returns_the_raw_coordinates():
    rng = np.random.default_rng(3)
    num, parts = random_sequences(rng, 2, 10, 5)
    ids = Oracle(2, 8, 0.5, 2, check_margin=False).update(num, parts)
    got = host_smooth(num, parts, ids, host_state(2, 8), 2, 8, 2, min_cutoff=1e300, beta=0.0)
    for i in range(len(num)):
        P = int(num[i])
        on = parts[i, :P, :, 3:4] >= 0
        assert np.array_equal(got[i, :P], np.where(on, parts[i, :P, :, :2], 0).astype(np.float32))
        assert (got[i, P:] == 0).all()


def test_argument_errors():
    num = np.zeros(4, np.int32)
    parts = np.zeros((4, 2, 18, 4), np.int32)
    ids = np.zeros((4, 2), np.int32)
    xy = np.zeros((4, 2, 18, 2), np.float32)
    st = host_state(2, 4)
    inf, nan = float("inf"), float("nan")

    def call(n=4, mh=2, state=st.ctypes.data, n_seq=2, mt=4, max_age=3, fps=30.0, mc=1.0, beta=0.007, dc=1.0,
             nump=num.ctypes.data, idp=ids.ctypes.data, xyp=xy.ctypes.data):
        return _lib.lib.ekp_debug_smooth_host(nump, parts.ctypes.data, idp, n, mh, state, n_seq, mt, max_age, fps, mc, beta, dc, xyp)

    assert call() == _lib.OK
    for bad in (dict(n=3), dict(n=0), dict(n_seq=0), dict(mt=1), dict(mt=_lib.LIMIT_TRACKS + 1), dict(max_age=-1), dict(mh=0),
                dict(fps=0.0), dict(fps=-30.0), dict(fps=inf), dict(fps=nan), dict(mc=0.0), dict(mc=inf), dict(mc=nan),
                dict(dc=0.0), dict(dc=-1.0), dict(dc=inf), dict(dc=nan), dict(beta=-0.1), dict(beta=inf), dict(beta=nan),
                dict(state=None), dict(nump=None), dict(idp=None), dict(xyp=None), dict(state=st.ctypes.data + 4),
                dict(nump=num.ctypes.data + 2), dict(xyp=xy.ctypes.data + 2)):
        assert call(**bad) == _lib.ERR_ARG, bad
    assert call(beta=0.0) == _lib.OK
    assert _lib.lib.ekp_smooth_state_bytes(0, 4) == 0 and _lib.lib.ekp_smooth_state_bytes(1, _lib.LIMIT_TRACKS + 1) == 0
    assert _lib.lib.ekp_smooth_state_bytes(3, 4) == 3 * _lib.lib.ekp_smooth_state_bytes(1, 4) == 3 * (16 + 728 * 4)
    dummy = ctypes.c_uint64(0)
    assert _lib.lib.ekp_smooth_humans(None, num.ctypes.data, parts.ctypes.data, ids.ctypes.data, 4, 2, ctypes.addressof(dummy), 2,
                                      4, 3, 30.0, 1.0, 0.007, 1.0, xy.ctypes.data, None) == _lib.ERR_ARG
    assert _lib.lib.ekp_smooth_reset(None, ctypes.addressof(dummy), 1, 4, None) == _lib.ERR_ARG


def test_infer_human_tensors_needs_a_tracker_for_a_smoother():
    from torch_ekpose_b200 import estimator
    with pytest.raises(ValueError):
        estimator.infer_human_tensors(None, None, "vgg", 0, smoother=object())


def test_package_imports_without_torch():
    code = ("import sys; sys.modules['torch'] = None\n"
            "import torch_ekpose_b200 as ek\n"
            "assert ek.Smoother and ek.Tracker\n"
            "try:\n    ek.Smoother(0)\nexcept ImportError:\n    print('ok')\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-c", code], cwd=root, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == "ok", out.stderr


# ---- GPU ----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


def _tables(torch, num, parts):
    return dict(num_humans=torch.from_numpy(np.ascontiguousarray(num, np.int32)).cuda(),
                parts=torch.from_numpy(np.ascontiguousarray(parts, np.int32)).cuda())


def _ids(torch, ids):
    return torch.from_numpy(np.ascontiguousarray(ids, np.int32)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("n_seq,Fs,mh,mt", [(1, (64, 1, 7, 32), 8, 16), (4, (1, 16, 5, 3), 6, 8), (64, (1, 2, 4), 5, 256),
                                            (3, (5, 9), 1, 1), (1, (100, 7), 40, 512)])
def test_update_equals_restatement(torch, n_seq, Fs, mh, mt):
    import torch_ekpose_b200 as ek
    rng = np.random.default_rng(n_seq * 100 + mh)
    o = Oracle(n_seq, mt, 0.5, 2, check_margin=False)
    R = Restatement(n_seq, mt, 2, 30.0, 1.0, 0.05, 1.0)
    sm = ek.Smoother(0, n_seq=n_seq, max_tracks=mt, max_age=2, fps=30.0, min_cutoff=1.0, beta=0.05, d_cutoff=1.0)
    for F in Fs:
        num, parts = random_sequences(rng, n_seq, F, mh)
        ids = o.update(num, parts)
        ids[rng.random(ids.shape) < 0.03] = -1
        want = R.update(num, parts, ids)
        got = sm.update(_tables(torch, num, parts), _ids(torch, ids)).cpu().numpy()
        assert np.array_equal(bits(got), bits(want)), (n_seq, F)


@pytest.mark.gpu
def test_dirty_out_is_fully_overwritten(torch):
    import torch_ekpose_b200 as ek
    rng = np.random.default_rng(2)
    num, parts = random_sequences(rng, 1, 8, 6)
    ids = Oracle(1, 8, 0.5, 30, check_margin=False).update(num, parts)
    sm = ek.Smoother(0, max_tracks=8)
    out = torch.full((8, 6, 18, 2), float("nan"), dtype=torch.float32, device="cuda")
    got = sm.update(_tables(torch, num, parts), _ids(torch, ids), out=out)
    assert got.data_ptr() == out.data_ptr()
    xy = got.cpu().numpy()
    assert np.array_equal(bits(xy), bits(Restatement(1, 8, 30).update(num, parts, ids)))
    for i in range(8):
        assert (xy[i, num[i]:] == 0).all()
        assert (xy[i, :num[i]][parts[i, :num[i], :, 3] < 0] == 0).all()
    with pytest.raises(ValueError):
        sm.update(_tables(torch, num, parts), _ids(torch, ids), out=torch.zeros((8, 6, 18, 3), device="cuda"))
    with pytest.raises(ValueError):
        sm.update(_tables(torch, num, parts), _ids(torch, ids[:, :5]))


@pytest.mark.gpu
def test_one_launch_no_host_wait_and_reset(torch):
    import torch_ekpose_b200 as ek
    rng = np.random.default_rng(4)
    num, parts = random_sequences(rng, 1, 16, 4)
    ids = Oracle(1, 256, 0.5, 30, check_margin=False).update(num, parts)
    tabs, idt = _tables(torch, num, parts), _ids(torch, ids)
    sm = ek.Smoother(0)
    first = sm.update(tabs, idt).cpu().numpy()
    k0 = sm.kernel_launches()
    torch.cuda.synchronize()
    torch.cuda._sleep(200_000_000)    # ~0.1 s of device time queued in front of the update
    ev = torch.cuda.Event()
    sm.update(tabs, idt)
    ev.record()
    assert not ev.query(), "update waited for the device"
    torch.cuda.synchronize()
    assert sm.kernel_launches() == k0 + 1
    sm.reset()
    assert np.array_equal(bits(sm.update(tabs, idt).cpu().numpy()), bits(first))


@pytest.mark.gpu
@pytest.mark.parametrize("frontend", ["reference", "dense"])
def test_end_to_end_jittery_sliding_scene(torch, frontend):
    """Synthetic people sliding right by half a stride-8 cell per frame, with a random +-1 cell jitter, through run ->
    result_tensors -> Tracker.update -> Smoother.update (device-only records): the smoothed keypoints equal the
    restatement on the host tables, and move less from frame to frame than the raw ones."""
    import torch_ekpose_b200 as ek
    from torch_ekpose_b200 import synthetic
    h, w, F = 46, 82, 24
    rng = np.random.default_rng(17)
    jit = rng.integers(-1, 2, F)
    base_h, base_p = synthetic.make_scene(h, w + F // 2 + 4, 3, seed=9, noise=False)
    heats, pafs = [], []
    for t in range(F):
        sh = t // 2 + 1 + int(jit[t])
        heats.append(np.roll(base_h, sh, axis=1)[:, :w])
        pafs.append(np.roll(base_p, sh, axis=1)[:, :w])
    heat = torch.from_numpy(np.ascontiguousarray(np.stack(heats).transpose(0, 3, 1, 2))).cuda()
    paf = torch.from_numpy(np.ascontiguousarray(np.stack(pafs).transpose(0, 3, 1, 2))).cuda()
    pp = ek.PostProcessor(device=0, max_batch=F, max_h=h, max_w=w, max_peaks=512, max_humans=16)
    pp.set_host_copy(False)
    tr = ek.Tracker(0, max_tracks=32)
    sm = ek.Smoother(0, max_tracks=32)
    R = Restatement(1, 32, 30)
    raw_tr, smooth_tr = {}, {}    # (id, part, axis) -> per-frame values
    for half in range(2):
        sl = slice(half * F // 2, (half + 1) * F // 2)
        pp.run(heat[sl], paf[sl], frontend=frontend)
        tabs = pp.result_tensors()
        ids = tr.update(tabs)
        xy = sm.update(tabs, ids).cpu().numpy()
        ids = ids.cpu().numpy()
        num, hparts, _ = pp.human_tables()
        host = np.zeros((len(num), 16, 18, 4), np.int32)
        for f, name in enumerate(("x", "y", "score", "id")):
            host[..., f] = hparts[name].view(np.int32) if name == "score" else hparts[name]
        assert num.min() > 0, num
        assert np.array_equal(bits(xy), bits(R.update(num, host, ids)))
        for i in range(len(num)):
            for p in range(int(num[i])):
                for part in range(18):
                    if host[i, p, part, 3] >= 0:
                        for ax in range(2):
                            raw_tr.setdefault((ids[i, p], part, ax), []).append(float(host[i, p, part, ax]))
                            smooth_tr.setdefault((ids[i, p], part, ax), []).append(float(xy[i, p, part, ax]))
    long = [k for k, v in raw_tr.items() if len(v) >= F // 2]
    assert len(long) >= 3 * 2 * 10, len(long)
    raw_var = np.mean([np.var(np.diff(raw_tr[k])) for k in long])
    smooth_var = np.mean([np.var(np.diff(smooth_tr[k])) for k in long])
    assert smooth_var < 0.5 * raw_var, (smooth_var, raw_var)


@pytest.mark.gpu
def test_infer_human_tensors_returns_smoothed_xy(torch):
    import torch_ekpose_b200 as ek
    from torch_ekpose_b200 import estimator, synthetic

    heat, paf = synthetic.make_batch(2, 46, 54, (2, 3), seed=3)
    heat_t, paf_t = torch.from_numpy(heat).cuda(), torch.from_numpy(paf).cuda()

    class Model(torch.nn.Module):   # stands in for the network: returns the synthetic maps
        def forward(self, x):
            return [paf_t[:x.shape[0]], heat_t[:x.shape[0]]], None

    frames = torch.zeros((2, 368, 432, 3), dtype=torch.uint8, device="cuda")
    tr, sm = ek.Tracker(0), ek.Smoother(0)
    tensors, _ = estimator.infer_human_tensors(frames, Model(), "vgg", 0, tracker=tr, smoother=sm)
    xy = tensors["smoothed_xy"]
    n, mh = tensors["track_id"].shape
    assert tuple(xy.shape) == (n, mh, 18, 2) and xy.dtype == torch.float32
    num = tensors["num_humans"].cpu().numpy()
    parts = tensors["parts"].cpu().numpy()
    want = Restatement().update(num, parts, tensors["track_id"].cpu().numpy())
    assert np.array_equal(bits(xy.cpu().numpy()), bits(want))
    plain, _ = estimator.infer_human_tensors(frames, Model(), "vgg", 0)
    assert "smoothed_xy" not in plain and "track_id" not in plain
