"""Every kernel variant the launchers choose, each reached on purpose and checked against the oracle bit for bit.

Each launcher picks one of several compiled variants by batch size, SM count, layout, map size and capacities; several
of them are reached by no ordinary workload.  Every case below names the variant it targets and proves, from a
torch.profiler trace of its own run (EKP_GRAPHS=0: eager launches), that the variant ran.  Sizes that depend on the SM
count are derived from the device, so a changed threshold fails a test instead of silently dropping its coverage.

The cases run in fresh worker processes (one per group of cases that share an environment), because kernel attributes
such as cudaFuncAttributeMaxDynamicSharedMemorySize are process-wide and the EKP_* variables are read once: a context
created earlier in a long-lived process would hide a set-up bug that a user with one context meets.  The worker writes
its results to an .npz; the oracle runs here, on the CPU."""
import functools
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from tests import util
from tests.util import assert_bits_equal

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# launcher constants (csrc/dense_frontend.cu, csrc/paf_connect.cu): the dense front-end's tiled lean kernel switches to
# 4-row-block tiles once the 2-row-block grid has 8 * SMs * kLeanBlocks CTAs; the connect kernel takes 256 threads while
# 19 * n blocks fit 4 per SM, else 128, and scores one pair per thread beyond 18 * threads / 32 pairs of a limb.
LEAN_BLOCKS = 5
PLANE_SMEM_MAX = 200 * 1024
ONE_BLOCK_SORT_MAX = 4096     # peaks_one_max(): process_paf's one-block ingest + sort


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _cdiv(a, b):
    return -(-a // b)


def _tile_cols(w):
    nt = _cdiv(w, 32)
    return _cdiv(w, _cdiv(w, nt))


def _tiled_tb(n, h, w, sms):
    """row blocks per tile of the tiled lean kernel for this batch"""
    return 4 if _tile_cols(w) * _cdiv(h, 2) * n >= 8 * sms * LEAN_BLOCKS else 2


def _n_tall(h, w, sms):
    """the smallest batch of h x w maps that the tiled lean kernel runs with 4-row-block tiles"""
    return _cdiv(8 * sms * LEAN_BLOCKS, _tile_cols(w) * _cdiv(h, 2))


def _plane_bytes(h, w):
    """dense_plane_kernel's dynamic shared memory for an unsliced plane"""
    nstrips = (8 * w + 29) // 30
    return 4 * ((h * w + 3) & ~3) + 4 * h * nstrips + 2 * ((_cdiv(h, 2) * nstrips + 1) & ~1)


def _dense_kernel(n, h, w, layout, sms, lean_tiled=False):
    if layout == "nchw" and _plane_bytes(h, w) <= PLANE_SMEM_MAX and not lean_tiled:
        return r"dense_plane_kernel\("
    return rf"dense_frontend_kernel<false, false, {_tiled_tb(n, h, w, sms)}>"


def _ref_kernel(h, w, layout):
    plane = layout == "nchw" and 4 * ((h * w + 3) & ~3) <= PLANE_SMEM_MAX and w <= 256
    return rf"ref_scan_kernel<{'true' if plane else 'false'}>"


# ---- inputs (seeded; built once per test process) --------------------------------------------------------------------
def _fuzz_scene(rng, H, W, people, drop, block, levels, per_part_cap=250):
    """People on a jittered grid with randomly missing parts over a PAF field that is piecewise constant on
    block x block cells with few distinct values: many pairs pass, many scores tie exactly, rows start
    at different limbs and have to be merged, connections reach across people."""
    tmpl = np.array([(0, -20), (0, -12), (-8, -12), (-12, -4), (-14, 4), (8, -12), (12, -4), (14, 4), (-5, 4), (-6, 14),
                     (-6, 24), (5, 4), (6, 14), (6, 24), (-2, -22), (2, -22), (-4, -21), (4, -21)], np.float32)
    rows, per_part = [], np.zeros(18, int)
    for _ in range(people):
        cx, cy = rng.integers(16, W - 16), rng.integers(26, H - 28)
        sc = rng.uniform(0.6, 1.2)
        for part in range(18):
            if rng.random() < drop or per_part[part] >= per_part_cap:
                continue
            x = int(np.clip(cx + sc * tmpl[part, 0] + rng.integers(-1, 2), 0, W - 1))
            y = int(np.clip(cy + sc * tmpl[part, 1] + rng.integers(-1, 2), 0, H - 1))
            rows.append((x, y, rng.choice([0.25, 0.5, 0.75, 1.0]), 0, part))
            per_part[part] += 1
    peaks = np.array(rows, np.float32).reshape(-1, 5)
    peaks = peaks[rng.permutation(len(peaks))]
    hb, wb = (H + block - 1) // block, (W + block - 1) // block
    coarse = rng.choice(levels, size=(hb, wb, 38)).astype(np.float32)
    paf = np.repeat(np.repeat(coarse, block, axis=0), block, axis=1)[:H, :W].copy()
    return peaks, paf


PAIRS_H, PAIRS_W = 128, 192
FUZZ = [(4, 0.0, 8, [0.0, 1.0]), (12, 0.3, 16, [-1.0, 0.0, 0.5, 1.0]), (40, 0.15, 8, [0.0, 0.25, 1.0]),
        (60, 0.5, 32, [0.5, 1.0]), (25, 0.6, 64, [1.0])]


def _limb0_scene(rng, n_a, n_b):
    """Exactly n_a necks (part 1) and n_b right shoulders (part 2), so that limb 0 has n_a x n_b pairs, over a PAF whose
    limb-0 channels point right in piecewise-constant blocks (many candidates, exact score ties); the other parts come
    from a fuzz scene."""
    H, W = PAIRS_H, PAIRS_W
    peaks, paf = _fuzz_scene(rng, H, W, 8, 0.2, 8, [0.0, 0.5, 1.0])
    peaks = peaks[(peaks[:, 4] != 1) & (peaks[:, 4] != 2)]
    score = lambda: rng.choice([0.25, 0.5, 0.75, 1.0])   # noqa: E731
    a = [(rng.integers(0, W // 3), rng.integers(0, H), score(), 0, 1) for _ in range(n_a)]
    b = [(rng.integers(W // 2, W), rng.integers(0, H), score(), 0, 2) for _ in range(n_b)]
    hb, wb = H // 8, W // 8
    paf[:, :, 12] = np.repeat(np.repeat(rng.choice([0.5, 1.0], (hb, wb)), 8, 0), 8, 1)
    paf[:, :, 13] = np.repeat(np.repeat(rng.choice([-0.25, 0.0, 0.25], (hb, wb)), 8, 0), 8, 1)
    peaks = np.concatenate([peaks, np.array(a + b, np.float32)])
    return peaks[rng.permutation(len(peaks))], paf


def _pair_batch(n, exact, seed):
    """run_peaks inputs: images 0.. with the exact limb-0 pair counts `exact`, the rest fuzz scenes"""
    rng = np.random.default_rng(seed)
    scenes = [_limb0_scene(rng, a, b) for a, b in exact]
    scenes += [_fuzz_scene(rng, PAIRS_H, PAIRS_W, *FUZZ[i % len(FUZZ)]) for i in range(n - len(exact))]
    counts = np.array([len(s[0]) for s in scenes], np.int32)
    peaks = np.zeros((n, counts.max(), 5), np.float32)
    for i, s in enumerate(scenes):
        peaks[i, :counts[i]] = s[0]
    return dict(peaks=peaks, counts=counts, paf=np.stack([s[1] for s in scenes]))


PP_H, PP_W = 256, 384
PP_CLUTTER = (4, 7, 10, 13)          # wrists and ankles: their only limbs lead to parts 3, 6, 9, 12, which stay empty


def _process_paf_scene(seed):
    """More than 4096 peaks with few candidate pairs: 1010 peaks on each of four parts whose limb partners are empty,
    plus a dozen people on the parts that do not touch them.  process_paf keeps the listed route (the host lists every
    sample) but has to ingest and sort with the two-kernel path."""
    rng = np.random.default_rng(seed)
    people, paf = _fuzz_scene(rng, PP_H, PP_W, 12, 0.1, 8, [0.0, 0.25, 0.5, 1.0])
    people = people[~np.isin(people[:, 4], PP_CLUTTER + (3, 6, 9, 12))]
    rows = [(rng.integers(0, PP_W), rng.integers(0, PP_H), rng.choice([0.25, 0.5, 0.75, 1.0]), 0, part)
            for part in PP_CLUTTER for _ in range(1010)]
    peaks = np.concatenate([people, np.array(rows, np.float32)])
    return dict(peaks=peaks[rng.permutation(len(peaks))], paf=paf)


@functools.lru_cache(maxsize=None)
def _batch(name):
    """Input arrays by name; maps are float32 in the layout the name says (nhwc* / tiny*: NHWC, else NCHW)."""
    from torch_ekpose_b200 import synthetic
    sms = _sms()
    kind, _, arg = name.partition(":")
    if kind == "crowd":                       # 16 x 92x164 (1312x736), 20-30 people
        heat, paf = synthetic.make_batch(16, 92, 164, (20, 30), seed=71)
    elif kind == "large":                     # 184x328 (2624x1472), just enough images for the tall tiled kernel
        heat, paf = synthetic.make_batch(_n_tall(184, 328, sms), 184, 328, (10, 20), seed=72)
    elif kind == "h234":                      # 234x164 / 233x164: tiled / plane just under 200 KB, unsliced batch
        heat, paf = synthetic.make_batch(_cdiv(sms, 18), 234, 164, (6, 12), seed=73)
    elif kind == "h233":
        b = _batch("h234")
        heat, paf = np.ascontiguousarray(b["heat"][:, :, :233]), np.ascontiguousarray(b["paf"][:, :, :233])
    elif kind == "r201":                      # reference scan: 201x256 generic, 200x256 plane of exactly 200 KB
        heat, paf = synthetic.make_batch(2, 201, 256, (4, 8), seed=74)
    elif kind == "r200":
        b = _batch("r201")
        heat, paf = np.ascontiguousarray(b["heat"][:, :, :200]), np.ascontiguousarray(b["paf"][:, :, :200])
    elif kind == "r257":                      # w > 256: generic
        heat, paf = synthetic.make_batch(2, 100, 257, (3, 6), seed=75)
    elif kind == "w300":
        heat, paf = synthetic.make_batch(3, 40, 300, (2, 6), seed=76)
    elif kind == "nhwc48":                    # NHWC 48x54, enough images for the tall kernel at every height 45..48
        heat, paf = synthetic.make_batch(max(_n_tall(h, 54, sms) for h in (45, 46, 47, 48)), 48, 54, (1, 6), seed=77,
                                         layout="nhwc")
    elif kind == "nhwc":                      # nhwc:<h>: the first rows of nhwc48
        b, h = _batch("nhwc48"), int(arg)
        heat, paf = np.ascontiguousarray(b["heat"][:, :h]), np.ascontiguousarray(b["paf"][:, :h])
    elif kind == "tiny":                      # 5x5 NHWC noise: 3 tiles per image, thousands of images
        rng = np.random.default_rng(78)
        n = _n_tall(5, 5, sms)
        heat = rng.random((n, 5, 5, 19), dtype=np.float32)
        paf = rng.normal(0, 0.5, (n, 5, 5, 38)).astype(np.float32)
    elif kind == "pairs128":                  # 128 threads: 72 pairs (by sample) vs 80 (per pair), 300 (two passes)
        return _pair_batch(_connect_n(sms, 128), [(9, 8), (10, 8), (20, 15)], 79)
    elif kind == "pairs256":                  # 256 threads: 144 vs 154, 576 (two passes)
        return _pair_batch(_connect_n(sms, 256), [(12, 12), (11, 14), (24, 24)], 80)
    elif kind == "ppbig":
        return _process_paf_scene(81)
    else:
        raise KeyError(name)
    return dict(heat=heat, paf=paf)


def _connect_n(sms, threads):
    """the biggest batch with 256-thread connect blocks, or the smallest with 128"""
    n = 4 * sms // 19
    return n if threads == 256 else n + 1


# ---- the cases ------------------------------------------------------------------------------------------------------
def _case(name, batch, n=None, layout="nchw", frontend="dense", op="run", expect=(), absent=(), people=None):
    return dict(name=name, batch=batch, n=n, layout=layout, frontend=frontend, op=op, expect=list(expect),
                absent=list(absent), people=people)


def _groups():
    """{group: dict(env, ctx, cases)}: the cases of a group run in one fresh process, in order, on ONE context."""
    sms = _sms()
    nl = _n_tall(184, 328, sms)
    n9 = _cdiv(sms, 18)
    big = [_case("crowd16_dense", "crowd", 16, expect=[_dense_kernel(16, 92, 164, "nchw", sms)]),
           _case("crowd16_reference", "crowd", 16, frontend="reference", expect=[_ref_kernel(92, 164, "nchw")])]
    big += [_case(f"plane_sliced_n{n}", "crowd", n, expect=[_dense_kernel(n, 92, 164, "nchw", sms)], people=[0, n - 1])
            for n in range(1, n9 + 1)]
    big += [_case("large_tall", "large", nl, expect=[_dense_kernel(nl, 184, 328, "nchw", sms)], people=[0, nl - 1]),
            _case("large_below_tall", "large", nl - 1, expect=[_dense_kernel(nl - 1, 184, 328, "nchw", sms)], people=[0]),
            _case("large_reference", "large", 2, frontend="reference", expect=[_ref_kernel(184, 328, "nchw")]),
            _case("large_gauss", "large", 2, frontend="reference_gauss", expect=[_ref_kernel(184, 328, "nchw")])]
    edges = [_case("h233_plane", "h233", n9, expect=[_dense_kernel(n9, 233, 164, "nchw", sms)], people=[0, n9 - 1]),
             _case("h234_tiled", "h234", n9, expect=[_dense_kernel(n9, 234, 164, "nchw", sms)], people=[0, n9 - 1]),
             _case("ref_200x256_plane", "r200", 2, frontend="reference", expect=[_ref_kernel(200, 256, "nchw")]),
             _case("ref_201x256_generic", "r201", 2, frontend="reference", expect=[_ref_kernel(201, 256, "nchw")]),
             _case("ref_100x257_generic", "r257", 2, frontend="reference", expect=[_ref_kernel(100, 257, "nchw")]),
             _case("ref_40x300_generic", "w300", 3, frontend="reference", expect=[_ref_kernel(40, 300, "nchw")]),
             _case("gauss_40x300_generic", "w300", 3, frontend="reference_gauss", expect=[_ref_kernel(40, 300, "nchw")])]
    nhwc = []
    for h in (45, 46, 47, 48):
        n = _n_tall(h, 54, sms)
        nhwc.append(_case(f"nhwc_tall_h{h}", f"nhwc:{h}", n, "nhwc", expect=[_dense_kernel(n, h, 54, "nhwc", sms)],
                          people=list(range(0, n, 16)) + [n - 1]))
    n = _n_tall(46, 54, sms)
    nhwc.append(_case("nhwc_below_tall_h46", "nhwc:46", n - 1, "nhwc", expect=[_dense_kernel(n - 1, 46, 54, "nhwc", sms)],
                      people=[0, n - 2]))
    n5 = _n_tall(5, 5, sms)
    nhwc.append(_case("nhwc_tall_5x5", "tiny", n5, "nhwc", expect=[_dense_kernel(n5, 5, 5, "nhwc", sms)],
                      people=list(range(0, n5, 64)) + [n5 - 1]))
    tiled = [_case("lean_tiled_crowd16", "crowd", 16, expect=[_dense_kernel(16, 92, 164, "nchw", sms, lean_tiled=True)]),
             _case("lean_tiled_h233", "h233", n9, expect=[_dense_kernel(n9, 233, 164, "nchw", sms, lean_tiled=True)],
                   people=[0, n9 - 1])]
    n128, n256 = _connect_n(sms, 128), _connect_n(sms, 256)

    def connect(tag):
        return [_case(f"connect128{tag}", "pairs128", n128, op="peaks", expect=[r"paf_connect_kernel<\d+, 128>"]),
                _case(f"connect256{tag}", "pairs256", n256, op="peaks", expect=[r"paf_connect_kernel<\d+, 256>"])]
    pp_big = _case("process_paf_4096plus", "ppbig", op="process_paf", expect=[r"peaks_ingest_kernel\(", r"peaks_sort_kernel\("],
                   absent=["peaks_ingest_sort_one_kernel", "pair_sample_offsets_kernel"])
    caps = dict(max_peaks=4096, max_humans=512, max_part=512, max_cand=4096)
    return {
        # bug 1: the first and only context is sized for 2624x1472 inputs; smaller maps must still get the plane kernels
        "big_context": dict(env={}, ctx=dict(max_batch=max(16, nl), max_h=184, max_w=328, **caps), cases=big),
        "plane_edges": dict(env={}, ctx=dict(max_batch=max(n9, 3), max_h=234, max_w=328, **caps), cases=edges),
        "nhwc_tall": dict(env={}, ctx=dict(max_batch=max(n5, 129), max_h=48, max_w=54, max_peaks=1024, max_humans=64),
                          cases=nhwc),
        "lean_tiled": dict(env={"EKP_LEAN_TILED": "1"}, ctx=dict(max_batch=16, max_h=234, max_w=328, **caps), cases=tiled),
        "connect": dict(env={}, ctx=dict(max_batch=n128, max_h=16, max_w=24, max_peaks=2048, max_humans=512),
                        cases=connect("") + [pp_big]),
        "connect_per_pair": dict(env={"EKP_BY_SAMPLE_MAX_PAIRS": "0"},
                                 ctx=dict(max_batch=n128, max_h=16, max_w=24, max_peaks=2048, max_humans=512),
                                 cases=connect("_per_pair")),
        "connect_by_sample": dict(env={"EKP_BY_SAMPLE_MAX_PAIRS": "1000000"},
                                  ctx=dict(max_batch=n128, max_h=16, max_w=24, max_peaks=2048, max_humans=512),
                                  cases=connect("_by_sample")),
    }


# the table the tests are parametrized by: (group, case name), fixed at collection without a device
CASE_IDS = [("big_context", c) for c in ["crowd16_dense", "crowd16_reference"] + [f"plane_sliced_n{n}" for n in range(1, 10)] +
            ["large_tall", "large_below_tall", "large_reference", "large_gauss"]] + \
           [("plane_edges", c) for c in ["h233_plane", "h234_tiled", "ref_200x256_plane", "ref_201x256_generic",
                                         "ref_100x257_generic", "ref_40x300_generic", "gauss_40x300_generic"]] + \
           [("nhwc_tall", c) for c in ["nhwc_tall_h45", "nhwc_tall_h46", "nhwc_tall_h47", "nhwc_tall_h48",
                                       "nhwc_below_tall_h46", "nhwc_tall_5x5"]] + \
           [("lean_tiled", c) for c in ["lean_tiled_crowd16", "lean_tiled_h233"]] + \
           [("connect", c) for c in ["connect128", "connect256", "process_paf_4096plus"]] + \
           [("connect_per_pair", c) for c in ["connect128_per_pair", "connect256_per_pair"]] + \
           [("connect_by_sample", c) for c in ["connect128_by_sample", "connect256_by_sample"]]


# ---- the worker (a fresh process per group) ------------------------------------------------------------------------
def _worker(spec_path, out_path):
    import torch_ekpose_b200 as ek
    from torch.profiler import ProfilerActivity, profile
    with open(spec_path) as f:
        spec = json.load(f)
    inputs = {name: np.load(os.path.join(os.path.dirname(spec_path), name.replace(":", "_") + ".npz"))
              for name in {c["batch"] for c in spec["cases"]}}
    pp = ek.PostProcessor(device=0, **spec["ctx"])   # the process's first and only context
    heat_mat = np.zeros((PP_H, 1, 19), np.float32)   # process_paf reads only its height
    out = {}
    for case in spec["cases"]:
        key, data = case["name"], inputs[case["batch"]]
        try:
            if case["op"] == "run":
                n = case["n"]
                heat, paf = torch.from_numpy(data["heat"][:n]).cuda(), torch.from_numpy(data["paf"][:n]).cuda()
            elif case["op"] == "peaks":
                peaks, counts, paf = (torch.from_numpy(data[k]).cuda() for k in ("peaks", "counts", "paf"))
            else:
                ek.pafprocess.process_paf(data["peaks"][None], heat_mat, data["paf"])  # grows its context first
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                if case["op"] == "run":
                    pp.run(heat, paf, layout=case["layout"], frontend=case["frontend"])
                    res = pp.results(with_peaks=True, raise_on_overflow=False)
                elif case["op"] == "peaks":
                    pp.run_peaks(peaks, counts, paf, h1=PAIRS_H)
                    res = pp.results(raise_on_overflow=False)
                else:
                    ek.pafprocess.process_paf(data["peaks"][None], heat_mat, data["paf"])
                    pf = ek.pafprocess
                    nh = pf.get_num_humans()
                    res = dict(num_humans=np.array([nh], np.int32),
                               cids=np.array([[pf.get_part_cid(h, p) for p in range(18)] for h in range(nh)], np.int32).reshape(nh, 18),
                               scores=np.array([pf.get_score(h) for h in range(nh)], np.float32),
                               line=np.array([(pf.get_part_x(k), pf.get_part_y(k)) for k in range(len(data["peaks"]))], np.int32),
                               line_score=np.array([pf.get_part_score(k) for k in range(len(data["peaks"]))], np.float32))
                torch.cuda.synchronize()
            out[key + "/kernels"] = np.array(json.dumps(sorted({e.name for e in prof.events()})))
            for k, v in res.items():
                out[key + "/" + k] = v
        except Exception as e:   # a refused launch is this case's finding; the other cases still run
            out[key + "/error"] = np.array(f"{type(e).__name__}: {e}")
    pp.close()
    np.savez(out_path, **out)


_WORKER = "import sys; from tests.test_launch_variants import _worker; _worker(sys.argv[1], sys.argv[2])"


@pytest.fixture(scope="module")
def run_group(tmp_path_factory):
    done = {}

    def run(group):
        if group not in done:
            g = _groups()[group]
            d = tmp_path_factory.mktemp(group)
            for name in {c["batch"] for c in g["cases"]}:
                np.savez(d / (name.replace(":", "_") + ".npz"), **_batch(name))
            with open(d / "spec.json", "w") as f:
                json.dump(dict(ctx=g["ctx"], cases=g["cases"]), f)
            env = dict(os.environ, EKP_GRAPHS="0", PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
            for k in ("EKP_LEAN_TILED", "EKP_BY_SAMPLE_MAX_PAIRS"):
                env.pop(k, None)
            env.update(g["env"])
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
def _oracle_peaks(batch, layout, frontend, i):
    hw = _hwc(_batch(batch)["heat"], layout, i)
    fe = util.frontend()
    return fe.dense_peaks(hw) if frontend == "dense" else fe.ref_nms(hw, gauss=frontend == "reference_gauss")


@functools.lru_cache(maxsize=None)
def _oracle_subset(batch, layout, frontend, i):
    pw = _hwc(_batch(batch)["paf"], layout, i)
    fe = util.frontend()
    paf_mat = fe.upsample_bilinear(pw) if frontend == "dense" else fe.upsample_nearest(pw)
    sub, _ = util.oracle_people(_oracle_peaks(batch, layout, frontend, i), 8 * pw.shape[0], 8 * pw.shape[1], paf_mat)
    return sub


@functools.lru_cache(maxsize=None)
def _oracle_run_peaks(batch, i):
    b = _batch(batch)
    sub, _ = util.oracle_people(b["peaks"][i, :b["counts"][i]], PAIRS_H, PAIRS_W, b["paf"][i])
    return sub


def _assert_kernels(out, case):
    names = json.loads(str(out[case["name"] + "/kernels"]))
    for pat in case["expect"]:
        assert any(re.search(pat, k) for k in names), f"{case['name']}: no kernel matches {pat!r}; ran {names}"
    for pat in case["absent"]:
        assert not any(re.search(pat, k) for k in names), f"{case['name']}: {pat!r} ran; ran {names}"


@pytest.mark.parametrize("group,name", CASE_IDS, ids=[f"{g}-{c}" for g, c in CASE_IDS])
def test_launch_variant_equals_the_oracle(run_group, group, name):
    case = next(c for c in _groups()[group]["cases"] if c["name"] == name)
    out = run_group(group)
    key = name + "/"
    assert key + "error" not in out, f"{name}: {out[key + 'error']}"
    _assert_kernels(out, case)
    if case["op"] == "process_paf":
        b = _batch(case["batch"])
        assert len(b["peaks"]) > ONE_BLOCK_SORT_MAX
        sub, line = util.oracle_people(b["peaks"], PP_H, PP_W, b["paf"])
        nh = int(out[key + "num_humans"][0])
        assert nh == len(sub) > 0, (nh, len(sub))
        assert np.array_equal(out[key + "cids"], sub[:, :18].astype(np.int32))
        assert_bits_equal(out[key + "scores"], (sub[:, 18] / sub[:, 19]).astype(np.float32), "human scores")
        assert np.array_equal(out[key + "line"][:, 0], line[0]) and np.array_equal(out[key + "line"][:, 1], line[1])
        assert_bits_equal(out[key + "line_score"], line[2], "getter table scores")
        return
    n = case["n"]
    assert len(out[key + "num_humans"]) == n
    assert not out[key + "overflow"].any(), f"{name}: overflow {np.unique(out[key + 'overflow'])}"
    if case["op"] == "peaks":
        for i in range(n):
            sub = _oracle_run_peaks(case["batch"], i)
            m = int(out[key + "num_humans"][i])
            assert m == len(sub), f"{name} image {i}: {m} people vs {len(sub)}"
            assert_bits_equal(out[key + "subset"][i, :m], sub, f"{name} image {i} subset")
        return
    res = dict(n_peaks=out[key + "n_peaks"], peaks=out[key + "peaks"], part_off=out[key + "part_off"])
    for i in range(n):   # the peak table of every image
        assert_bits_equal(util.peaks_table(res, i), _oracle_peaks(case["batch"], case["layout"], case["frontend"], i),
                          f"{name} image {i} peaks")
    for i in (range(n) if case["people"] is None else case["people"]):
        sub = _oracle_subset(case["batch"], case["layout"], case["frontend"], i)
        m = int(out[key + "num_humans"][i])
        assert m == len(sub), f"{name} image {i}: {m} people vs {len(sub)}"
        assert_bits_equal(out[key + "subset"][i, :m], sub, f"{name} image {i} subset")
    assert out[key + "num_humans"].sum() > 0


def test_case_table_matches_the_groups():
    """CASE_IDS (fixed at collection) lists every case the groups define on this device, and only those."""
    assert sorted(CASE_IDS) == sorted((g, c["name"]) for g, v in _groups().items() for c in v["cases"])


def test_sizes_sit_on_the_thresholds():
    """The batch sizes really sit on either side of each launcher threshold on this device."""
    sms = _sms()
    assert _plane_bytes(233, 164) <= PLANE_SMEM_MAX < _plane_bytes(234, 164)
    assert 4 * 200 * 256 == PLANE_SMEM_MAX
    assert 18 * _cdiv(sms, 18) >= sms > 18 * (_cdiv(sms, 18) - 1)         # 9 images: the first unsliced plane batch
    for h, w in ((45, 54), (46, 54), (47, 54), (48, 54), (5, 5), (184, 328)):
        n = _n_tall(h, w, sms)
        assert _tiled_tb(n, h, w, sms) == 4 and _tiled_tb(n - 1, h, w, sms) == 2
    assert [(h - 1) % 4 + 1 for h in (45, 46, 47, 48)] == [1, 2, 3, 4]    # rows of the last 4-row-block tile
    n128, n256 = _connect_n(sms, 128), _connect_n(sms, 256)
    assert 19 * n256 <= 4 * sms < 19 * n128
    assert 9 * 8 == 18 * 128 // 32 < 10 * 8 <= 2 * 128 < 20 * 15
    assert 12 * 12 == 18 * 256 // 32 < 11 * 14 <= 2 * 256 < 24 * 24
