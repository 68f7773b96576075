"""Stable person ids across frames (ekp_track_humans / Tracker) against a NumPy restatement of the specification in
include/ekpose_b200.h: the oracle below.  On the CPU, ekp_debug_track_host (the kernel's own code run serially) is checked
on thousands of random sequences; on the GPU, Tracker.update."""
import ctypes
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from torch_ekpose_b200 import _lib
from torch_ekpose_b200.coco import ORDER_COCO

SIGMAS = np.array([.26, .25, .25, .35, .35, .79, .79, .72, .72, .62, .62, 1.07, 1.07, .87, .87, .89, .89]) / 10.0
VARS = (SIGMAS * 2) ** 2   # as pycocotools computes them
MARGIN = 1e-9


class MarginError(AssertionError):
    """Two competing similarities, or a similarity and min_oks, closer than MARGIN without being equal: the device's exp
    and NumPy's may order them differently, so such a scene does not pin the ids."""


def _poses(parts_rows):
    """[P, 18, 4] int rows -> (xy [P, 17, 2] int64, present [P, 17] bool) in COCO order."""
    rows = np.asarray(parts_rows).reshape(-1, 18, 4)[:, ORDER_COCO]
    return rows[..., :2].astype(np.int64), rows[..., 3] >= 0


def oks_matrix(pxy, pon, txy, ton):
    """sim [P, T] of people against tracks (the tracks' poses are the ground truth), summed in keypoint order."""
    P, T = len(pxy), len(txy)
    sim = np.zeros((P, T))
    for t in range(T):
        on = ton[t]
        if on.any():
            xs, ys = txy[t, on, 0], txy[t, on, 1]
            area = float((xs.max() - xs.min() + 1) * (ys.max() - ys.min() + 1))
        for p in range(P):
            both = pon[p] & on
            m = int(both.sum())
            if m == 0:
                continue
            s = 0.0
            for j in np.nonzero(both)[0]:
                d2 = int((pxy[p, j, 0] - txy[t, j, 0]) ** 2 + (pxy[p, j, 1] - txy[t, j, 1]) ** 2)
                s += math.exp(-(d2 / VARS[j] / area / 2.0))
            sim[p, t] = s / m
    return sim


class Oracle:
    """The specification, one sequence at a time."""

    def __init__(self, n_seq=1, max_tracks=256, min_oks=0.5, max_age=30, check_margin=True):
        self.min_oks = float(np.float32(min_oks))     # the C ABI takes a float
        self.max_tracks, self.max_age, self.check_margin = max_tracks, max_age, check_margin
        self.seq = [dict(frame=0, next_id=0, tracks=[]) for _ in range(n_seq)]

    def _frame(self, S, xy, on):
        f = S["frame"]
        S["tracks"] = [t for t in S["tracks"] if f - t["last"] <= self.max_age + 1]
        tr = S["tracks"]
        P = len(xy)
        sim = oks_matrix(xy, on, np.array([t["xy"] for t in tr]).reshape(-1, 17, 2),
                         np.array([t["on"] for t in tr]).reshape(-1, 17)) if tr and P else np.zeros((P, len(tr)))
        if self.check_margin and sim.size:
            near = np.abs(sim - self.min_oks)
            if ((near < MARGIN) & (near > 0)).any():
                raise MarginError("a similarity within 1e-9 of min_oks")
            v = np.unique(sim[sim >= self.min_oks])
            if len(v) > 1 and (np.diff(v) < MARGIN).any():
                raise MarginError("two similarities within 1e-9")
        pairs = sorted(((-sim[p, k], tr[k]["id"], p, k) for p in range(P) for k in range(len(tr)) if sim[p, k] >= self.min_oks))
        ids = [-1] * P
        taken = set()
        for _, tid, p, k in pairs:
            if ids[p] < 0 and k not in taken:
                ids[p] = tid
                taken.add(k)
                tr[k].update(xy=xy[p].copy(), on=on[p].copy(), last=f)
        opened = set()
        for p in range(P):
            if ids[p] >= 0:
                continue
            new = dict(id=S["next_id"], xy=xy[p].copy(), on=on[p].copy(), last=f)
            S["next_id"] += 1
            if len(tr) == self.max_tracks:
                cand = [k for k in range(len(tr)) if k not in taken and tr[k]["id"] not in opened]
                victim = min(cand, key=lambda k: (tr[k]["last"], tr[k]["id"]))
                tr[victim] = new
            else:
                tr.append(new)
            opened.add(new["id"])
            ids[p] = new["id"]
        S["frame"] += 1
        return ids

    def update(self, num_humans, parts):
        """num_humans [n], parts [n, max_humans, 18, 4] int -> ids [n, max_humans]"""
        parts = np.asarray(parts).reshape(len(num_humans), -1, 18, 4)
        n, mh = parts.shape[:2]
        F = n // len(self.seq)
        out = np.full((n, mh), -1, np.int32)
        for i in range(n):
            P = min(max(int(num_humans[i]), 0), mh)
            xy, on = _poses(parts[i, :P])
            out[i, :P] = self._frame(self.seq[i // F], xy, on)
        return out


# ---- scene generators ---------------------------------------------------------------------------------------------------
def _person(rng, cx, cy, scale):
    """one reference-part pose [18, 4] (x, y, score bits, id)"""
    tpl = rng.uniform(-0.5, 0.5, (18, 2)) * scale
    row = np.zeros((18, 4), np.int64)
    row[:, 0] = np.round(cx + tpl[:, 0])
    row[:, 1] = np.round(cy + tpl[:, 1])
    row[:, 3] = np.arange(18)
    return row


def random_sequences(rng, n_seq, F, max_humans, dup=True):
    """tables of n_seq x F frames of people walking around, appearing, vanishing, losing parts, and (dup) duplicated."""
    num = np.zeros(n_seq * F, np.int32)
    parts = np.zeros((n_seq * F, max_humans, 18, 4), np.int32)
    for s in range(n_seq):
        world = [dict(row=_person(rng, rng.uniform(0, 600), rng.uniform(0, 400), rng.uniform(20, 200)),
                      v=rng.normal(0, 4, 2)) for _ in range(rng.integers(1, max_humans + 3))]
        for t in range(F):
            i = s * F + t
            people = []
            for w in world:
                w["row"][:, :2] += np.round(w["v"] + rng.normal(0, 1.5, (18, 2))).astype(np.int64)
                if rng.random() < 0.8:
                    r = w["row"].copy()
                    r[rng.random(18) < 0.15, 3] = -1
                    if rng.random() < 0.03:
                        r[ORDER_COCO, 3] = -1   # only the neck left: no COCO keypoint in common with anyone
                    people.append(r)
            if dup and people and rng.random() < 0.2:
                people.append(people[rng.integers(len(people))].copy())   # an exact tie
            if rng.random() < 0.1:
                people = []
            rng.shuffle(people)
            people = people[:max_humans]
            num[i] = len(people)
            for p, r in enumerate(people):
                parts[i, p] = r
            if rng.random() < 0.2:
                world.append(dict(row=_person(rng, rng.uniform(0, 600), rng.uniform(0, 400), rng.uniform(20, 200)),
                                  v=rng.normal(0, 4, 2)))
            if len(world) > 1 and rng.random() < 0.1:
                world.pop(rng.integers(len(world)))
    return num, parts


def host_track(num, parts, state, n_seq, max_tracks, min_oks, max_age):
    n, mh = parts.shape[:2]
    ids = np.full((n, mh), 0x7f7f7f7f, np.int32)
    num = np.ascontiguousarray(num, np.int32)
    parts = np.ascontiguousarray(parts, np.int32)
    rc = _lib.lib.ekp_debug_track_host(num.ctypes.data, parts.ctypes.data, n, mh, state.ctypes.data, n_seq, max_tracks,
                                       min_oks, max_age, ids.ctypes.data)
    _lib.check(rc)
    return ids


def host_state(n_seq, max_tracks):
    nb = _lib.lib.ekp_track_state_bytes(n_seq, max_tracks)
    return np.zeros(nb // 8, np.float64)   # 8-byte aligned, zero = reset


# ---- CPU ----------------------------------------------------------------------------------------------------------------
def test_oracle_hand_worked_two_people():
    a = np.full((18, 4), -1, np.int64)
    a[0] = (100, 100, 0, 0)      # nose (COCO 0)
    a[5] = (110, 120, 0, 1)      # left shoulder (COCO 5)
    b = a.copy()
    b[:, 0] += 300
    o = Oracle(min_oks=0.5)
    ids = o.update([2], np.stack([a, b])[None])
    assert ids[0, :2].tolist() == [0, 1]
    # frame 2: b moved by one pixel right on both keypoints, a by one down on its nose only; rows swapped
    a2, b2 = a.copy(), b.copy()
    a2[0, 1] += 1
    b2[[0, 5], 0] += 1
    area = (110 - 100 + 1) * (120 - 100 + 1)   # 231: the tracks' box
    sa = (math.exp(-1 / VARS[0] / area / 2) + 1.0) / 2
    sb = (math.exp(-1 / VARS[0] / area / 2) + math.exp(-1 / VARS[5] / area / 2)) / 2
    sim = oks_matrix(*_poses(np.stack([b2, a2])), *_poses(np.stack([b, a])))
    assert sim[0, 0] == sb and sim[1, 1] == sa and sim[0, 1] == 0 and sim[1, 0] == 0
    assert 0.5 < sb < sa < 1
    assert o.update([2], np.stack([b2, a2])[None])[0, :2].tolist() == [1, 0]
    # min_oks above b's similarity: b opens track 2
    o2 = Oracle(min_oks=0.5)
    o2.update([2], np.stack([a, b])[None])
    o2.min_oks = (sb + sa) / 2
    assert o2.update([2], np.stack([b2, a2])[None])[0, :2].tolist() == [2, 0]


def _fuzz_case(rng):
    max_humans = int(rng.integers(1, 7))
    max_tracks = int(rng.integers(max_humans, max_humans + 5))
    n_seq = int(rng.integers(1, 4))
    F = int(rng.integers(1, 9))
    min_oks = float(rng.choice([0.1, 0.3, 0.5, 0.8]))   # 0 would make every tiny similarity compete
    max_age = int(rng.integers(0, 4))
    return max_humans, max_tracks, n_seq, F, min_oks, max_age


def test_host_hook_equals_oracle_on_random_sequences():
    rng = np.random.default_rng(7)
    done = skipped = frames = 0
    while done < 3000:
        mh, mt, n_seq, F, min_oks, max_age = _fuzz_case(rng)
        o = Oracle(n_seq, mt, min_oks, max_age)
        st = host_state(n_seq, mt)
        try:
            for _ in range(3):   # calls carry the state
                num, parts = random_sequences(rng, n_seq, F, mh)
                want = o.update(num, parts)
                got = host_track(num, parts, st, n_seq, mt, min_oks, max_age)
                assert np.array_equal(got, want), (mh, mt, n_seq, F, min_oks, max_age, got, want)
                frames += len(num)
        except MarginError:
            skipped += 1
            continue
        done += n_seq
    assert skipped < done / 10
    assert frames > 10000


def test_host_hook_ages_tracks_out_after_max_age_plus_one_frames():
    p = _person(np.random.default_rng(1), 200, 200, 100)
    for max_age in (0, 1, 3):
        for gap in (max_age, max_age + 1):   # frames the person is missing
            num = np.array([1] + [0] * gap + [1], np.int32)
            parts = np.zeros((len(num), 1, 18, 4), np.int32)
            parts[0, 0] = parts[-1, 0] = p
            st = host_state(1, 4)
            ids = host_track(num, parts, st, 1, 4, 0.5, max_age)
            assert ids[-1, 0] == (0 if gap <= max_age else 1), (max_age, gap)
            assert np.array_equal(ids, Oracle(1, 4, 0.5, max_age).update(num, parts))


def test_host_hook_reuses_the_slot_of_the_oldest_then_lowest_id_track():
    rng = np.random.default_rng(3)
    people = [_person(rng, 100 + 150 * k, 200, 60) for k in range(6)]
    # frame 0: people 0, 1; frame 1: 2, 3 (0, 1 unmatched); frame 2: 1 (matched), 4, 5 -> 2 new tracks in a full table of 4
    frames = [[0, 1], [2, 3], [1, 4, 5]]
    num = np.array([len(f) for f in frames], np.int32)
    parts = np.zeros((3, 3, 18, 4), np.int32)
    for i, f in enumerate(frames):
        for r, k in enumerate(f):
            parts[i, r] = people[k]
    st = host_state(1, 4)
    ids = host_track(num, parts, st, 1, 4, 0.5, 30)
    assert ids.tolist() == [[0, 1, -1], [2, 3, -1], [1, 4, 5]]
    # track 0 (oldest, lowest id) and then track 2 were evicted: person 0 and 2 come back as new tracks, 3 keeps its id
    num2 = np.array([3], np.int32)
    p2 = np.zeros((1, 3, 18, 4), np.int32)
    for r, k in enumerate([0, 2, 3]):
        p2[0, r] = people[k]
    assert host_track(num2, p2, st, 1, 4, 0.5, 30).tolist() == [[6, 7, 3]]
    o = Oracle(1, 4, 0.5, 30)
    o.update(num, parts)
    assert o.update(num2, p2).tolist() == [[6, 7, 3]]


def test_host_hook_state_carries_across_any_split_of_the_frames():
    rng = np.random.default_rng(11)
    for _ in range(20):
        num, parts = random_sequences(rng, 1, 24, 5)
        st = host_state(1, 8)
        whole = host_track(num, parts, st, 1, 8, 0.5, 2)
        for splits in ([24], [1] * 24, [5, 7, 12], [12, 12], [3, 1, 20]):
            st = host_state(1, 8)
            got, at = [], 0
            for F in splits:
                got.append(host_track(num[at:at + F], parts[at:at + F], st, 1, 8, 0.5, 2))
                at += F
            assert np.array_equal(np.concatenate(got), whole), splits


def test_host_hook_large_frames_use_the_state_scratch():
    """300 people against 300 tracks: more pairs than shared memory holds, so the similarities go to the state."""
    rng = np.random.default_rng(5)
    people = [_person(rng, 40 * (k % 30), 60 * (k // 30), 30) for k in range(300)]
    parts = np.zeros((2, 300, 18, 4), np.int32)
    for k in range(300):
        parts[0, k] = people[k]
        parts[1, 299 - k] = people[k]
        parts[1, 299 - k, :, 0] += 1
    num = np.array([300, 300], np.int32)
    st = host_state(1, 300)
    ids = host_track(num, parts, st, 1, 300, 0.5, 30)
    assert ids[0].tolist() == list(range(300)) and ids[1].tolist() == list(range(299, -1, -1))
    assert np.array_equal(ids, Oracle(1, 300, 0.5, 30, check_margin=False).update(num, parts))


def test_package_imports_without_torch(tmp_path):
    """torch is optional for the host surface: the Tracker must not make it a requirement of the package import."""
    code = ("import sys; sys.modules['torch'] = None\n"
            "import torch_ekpose_b200 as ek\n"
            "assert ek.pafprocess and ek.paf_to_pose_cpp and ek.Tracker\n"
            "try:\n    ek.Tracker(0)\nexcept ImportError:\n    print('ok')\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-c", code], cwd=root, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == "ok", out.stderr


def test_argument_errors():
    num = np.zeros(4, np.int32)
    parts = np.zeros((4, 2, 18, 4), np.int32)
    ids = np.zeros((4, 2), np.int32)
    st = host_state(2, 4)

    def call(n=4, mh=2, state=st.ctypes.data, n_seq=2, mt=4, min_oks=0.5, max_age=3, nump=num.ctypes.data, idp=ids.ctypes.data):
        return _lib.lib.ekp_debug_track_host(nump, parts.ctypes.data, n, mh, state, n_seq, mt, min_oks, max_age, idp)

    assert call() == _lib.OK
    for bad in (dict(n=3), dict(n=0), dict(n_seq=0), dict(mt=1), dict(mt=_lib.LIMIT_TRACKS + 1), dict(max_age=-1),
                dict(min_oks=-0.1), dict(min_oks=float("nan")), dict(min_oks=float("inf")), dict(state=None),
                dict(nump=None), dict(idp=None), dict(state=st.ctypes.data + 4), dict(nump=num.ctypes.data + 2), dict(mh=0)):
        assert call(**bad) == _lib.ERR_ARG, bad
    assert _lib.lib.ekp_track_state_bytes(0, 4) == 0 and _lib.lib.ekp_track_state_bytes(1, _lib.LIMIT_TRACKS + 1) == 0
    assert _lib.lib.ekp_track_state_bytes(3, 4) == 3 * _lib.lib.ekp_track_state_bytes(1, 4)
    dummy = ctypes.c_uint64(0)
    assert _lib.lib.ekp_track_humans(None, num.ctypes.data, parts.ctypes.data, 4, 2, ctypes.addressof(dummy), 2, 4, 0.5, 3,
                                     ids.ctypes.data, None) == _lib.ERR_ARG
    assert _lib.lib.ekp_track_reset(None, ctypes.addressof(dummy), 1, 4, None) == _lib.ERR_ARG


# ---- GPU ----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


def _tables(torch, num, parts):
    return dict(num_humans=torch.from_numpy(np.ascontiguousarray(num, np.int32)).cuda(),
                parts=torch.from_numpy(np.ascontiguousarray(parts, np.int32)).cuda())


@pytest.mark.gpu
@pytest.mark.parametrize("n_seq,Fs,mh,mt", [(1, (64, 1, 7, 32), 8, 16), (4, (1, 16, 5, 3), 6, 8), (64, (1, 2, 4), 5, 256),
                                            (2, (3, 9), 40, 64)])
def test_update_equals_oracle(torch, n_seq, Fs, mh, mt):
    import torch_ekpose_b200 as ek
    rng = np.random.default_rng(n_seq * 100 + mh)
    for attempt in range(20):
        o = Oracle(n_seq, mt, 0.5, 2)
        tr = ek.Tracker(0, n_seq=n_seq, max_tracks=mt, min_oks=0.5, max_age=2)
        try:
            for F in Fs:
                num, parts = random_sequences(rng, n_seq, F, mh)
                want = o.update(num, parts)
                got = tr.update(_tables(torch, num, parts)).cpu().numpy()
                assert np.array_equal(got, want), (n_seq, F)
            return
        except MarginError:
            continue
    pytest.fail("no scene kept the similarity margin")


@pytest.mark.gpu
def test_update_large_frames_use_the_state_scratch(torch):
    import torch_ekpose_b200 as ek
    rng = np.random.default_rng(5)
    people = [_person(rng, 40 * (k % 30), 60 * (k // 30), 30) for k in range(300)]
    parts = np.zeros((2, 300, 18, 4), np.int32)
    for k in range(300):
        parts[0, k] = people[k]
        parts[1, 299 - k] = people[k]
        parts[1, 299 - k, :, 0] += 1
    num = np.array([300, 300], np.int32)
    tr = ek.Tracker(0, max_tracks=300)
    ids = tr.update(_tables(torch, num, parts)).cpu().numpy()
    assert np.array_equal(ids, Oracle(1, 300, 0.5, 30, check_margin=False).update(num, parts))


@pytest.mark.gpu
def test_permuting_rows_permutes_ids(torch):
    """Every person of frames 1.. continues a track (births take ids in row order, so only matches are permutable)."""
    import torch_ekpose_b200 as ek
    rng = np.random.default_rng(21)
    K, F = 8, 6
    for _ in range(20):
        people = [_person(rng, 150 * k + 50, rng.uniform(50, 300), rng.uniform(60, 120)) for k in range(K)]
        parts = np.zeros((F, K, 18, 4), np.int32)
        for t in range(F):
            for k in range(K):
                parts[t, k] = people[k]
                people[k][:, :2] += rng.integers(-2, 3, (18, 2))
        num = np.full(F, K, np.int32)
        try:
            want = Oracle(1, 16).update(num, parts)
        except MarginError:
            continue
        assert (want[1:] == want[0]).all()       # nobody opened a track after frame 0
        perm = [np.arange(K)] + [rng.permutation(K) for _ in range(1, F)]
        parts2 = np.stack([parts[t, perm[t]] for t in range(F)])
        ia = ek.Tracker(0, max_tracks=16).update(_tables(torch, num, parts)).cpu().numpy()
        ib = ek.Tracker(0, max_tracks=16).update(_tables(torch, num, parts2)).cpu().numpy()
        assert np.array_equal(ia, want)
        for t in range(F):
            assert np.array_equal(ib[t], ia[t, perm[t]]), t
        return
    pytest.fail("no scene kept the similarity margin")


@pytest.mark.gpu
def test_rows_past_num_humans_are_minus_one_over_dirty_out(torch):
    import torch_ekpose_b200 as ek
    rng = np.random.default_rng(2)
    num, parts = random_sequences(rng, 1, 8, 6)
    tr = ek.Tracker(0, max_tracks=8)
    out = torch.full((8, 6), 0x7f7f7f7f, dtype=torch.int32, device="cuda")
    got = tr.update(_tables(torch, num, parts), out=out)
    assert got.data_ptr() == out.data_ptr()
    ids = got.cpu().numpy()
    for i in range(8):
        assert (ids[i, num[i]:] == -1).all() and (ids[i, :num[i]] >= 0).all()
    with pytest.raises(ValueError):
        tr.update(_tables(torch, num, parts), out=torch.zeros((8, 5), dtype=torch.int32, device="cuda"))


@pytest.mark.gpu
def test_one_launch_no_host_wait_and_reset(torch):
    import torch_ekpose_b200 as ek
    rng = np.random.default_rng(4)
    num, parts = random_sequences(rng, 1, 16, 4)
    tabs = _tables(torch, num, parts)
    tr = ek.Tracker(0)
    first = tr.update(tabs).cpu().numpy()
    k0 = tr.kernel_launches()
    torch.cuda.synchronize()
    torch.cuda._sleep(200_000_000)    # ~0.1 s of device time queued in front of the update
    ev = torch.cuda.Event()
    out = tr.update(tabs)
    ev.record()
    assert not ev.query(), "update waited for the device"
    torch.cuda.synchronize()
    assert tr.kernel_launches() == k0 + 1
    assert out.max().item() >= first.max()   # the same people again: matched to the live tracks
    tr.reset()
    assert np.array_equal(tr.update(tabs).cpu().numpy(), first)


@pytest.mark.gpu
@pytest.mark.parametrize("frontend", ["reference", "dense"])
def test_end_to_end_moving_people(torch, frontend):
    """Synthetic people shifted a few pixels per frame through run -> result_tensors -> update (device-only records):
    the ids equal the oracle's on the host tables, and each synthetic person keeps one id."""
    import torch_ekpose_b200 as ek
    from torch_ekpose_b200 import synthetic
    h, w, F = 46, 82, 12
    heats, pafs = [], []
    base_h, base_p = synthetic.make_scene(h, w + 4 * F // 8 + 2, 3, seed=9, noise=False)
    for t in range(F):     # the whole scene slides right by 4 map pixels (half a stride-8 cell) per frame
        heats.append(np.roll(base_h, t // 2, axis=1)[:, :w])
        pafs.append(np.roll(base_p, t // 2, axis=1)[:, :w])
    heat = torch.from_numpy(np.ascontiguousarray(np.stack(heats).transpose(0, 3, 1, 2))).cuda()
    paf = torch.from_numpy(np.ascontiguousarray(np.stack(pafs).transpose(0, 3, 1, 2))).cuda()
    pp = ek.PostProcessor(device=0, max_batch=F, max_h=h, max_w=w, max_peaks=512, max_humans=16)
    pp.set_host_copy(False)
    tr = ek.Tracker(0, max_tracks=32)
    o = Oracle(1, 32, 0.5, 30, check_margin=False)
    for half in range(2):
        sl = slice(half * F // 2, (half + 1) * F // 2)
        pp.run(heat[sl], paf[sl], frontend=frontend)
        tabs = pp.result_tensors()
        ids = tr.update(tabs).cpu().numpy()
        num, hparts, _ = pp.human_tables()
        host = np.zeros((len(num), 16, 18, 4), np.int32)
        for f, name in enumerate(("x", "y", "score", "id")):
            host[..., f] = hparts[name].view(np.int32) if name == "score" else hparts[name]
        assert num.min() > 0, num    # the front-end found the synthetic people in every frame
        assert np.array_equal(ids, o.update(num, host))
        for i in range(len(num)):
            assert sorted(ids[i, :num[i]].tolist()) == list(range(int(num[i]))), ids   # no new track: every person kept its id


@pytest.mark.gpu
def test_infer_human_tensors_returns_track_ids(torch):
    import torch_ekpose_b200 as ek
    from torch_ekpose_b200 import estimator, synthetic

    heat, paf = synthetic.make_batch(2, 46, 54, (2, 3), seed=3)
    heat_t, paf_t = torch.from_numpy(heat).cuda(), torch.from_numpy(paf).cuda()

    class Model(torch.nn.Module):   # stands in for the network: returns the synthetic maps
        def forward(self, x):
            return [paf_t[:x.shape[0]], heat_t[:x.shape[0]]], None

    frames = torch.zeros((2, 368, 432, 3), dtype=torch.uint8, device="cuda")
    tr = ek.Tracker(0)
    tensors, _ = estimator.infer_human_tensors(frames, Model(), "vgg", 0, tracker=tr)
    ids = tensors["track_id"].cpu().numpy()
    num = tensors["num_humans"].cpu().numpy()
    assert ids.shape == tuple(tensors["scores"].shape)
    assert (ids[0, :num[0]] >= 0).all() and (ids[:, max(num):] == -1).all()
