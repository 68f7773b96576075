"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the golden fixtures.

Bars (BASELINE.json north_star): peak coordinates, peak counts, person count and part indices
bit-exact; connection scores within 1e-5 relative -- the tests below demand BIT equality of the
float32 scores as well, because scores decide sort order and ties (SURVEY.md A.2).
Only the reference front-end's peak SCORES carry a tolerance (2.5e-7 abs) when compared with cv2's
default IPP build; against OpenCV's own code path they too are bit-exact.
"""
import numpy as np
import pytest

from tests import util
from tests.util import assert_bits_equal, golden

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def ek():
    import torch_ekpose_b200 as ek
    return ek


@pytest.fixture(scope="module")
def pp(ek):
    p = ek.PostProcessor(device=0, max_batch=64, max_h=92, max_w=164, max_peaks=2048, max_humans=128)
    yield p
    p.close()


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _nchw(hwc):
    return np.ascontiguousarray(hwc.transpose(2, 0, 1))[None]


# ---------------------------------------------------------------------------------------------
# the reference operator surface: process_paf / get_*  (stages 4-5 on host pointers)
# ---------------------------------------------------------------------------------------------
def _compat_subset(ek):
    pf = ek.pafprocess
    n = pf.get_num_humans()
    cids = np.array([[pf.get_part_cid(h, p) for p in range(18)] for h in range(n)], np.int32).reshape(n, 18)
    scores = np.array([pf.get_score(h) for h in range(n)], np.float32)
    return n, cids, scores


@pytest.mark.parametrize("case", ["chain", "chain_reversed", "short", "long_limb", "same_pixel"])
def test_process_paf_known_answers(ek, case):
    g = golden("kat")
    pk, want = g[case + "_peaks"], g[case + "_subset"]
    assert ek.pafprocess.process_paf(pk[None], np.zeros((64, 64, 19), np.float32), g["paf"]) == 0
    n, cids, scores = _compat_subset(ek)
    assert n == len(want)
    if n:
        assert np.array_equal(cids, want[:, :18].astype(np.int32))
        assert_bits_equal(scores, want[:, 18] / want[:, 19], "human score")
        # the A.1 quirk: get_part_x(cid) indexes the part-sorted table by input-order id
        for cid in range(len(pk)):
            assert ek.pafprocess.get_part_x(cid) == int(g[case + "_line_x"][cid])
    if case == "chain":
        assert n == 1 and float(scores[0]) == 1.5 and list(cids[0][1:5]) == [0, 1, 2, 3]


@pytest.mark.parametrize("upload", ["listed", "sparse", "dense"])
@pytest.mark.parametrize("scene", util.SCENES)
def test_process_paf_golden(ek, scene, upload, monkeypatch):
    """Reference peaks + nearest-upsampled PAF in, the compiled reference's subset out (bit-exact), both when
    only the sampled PAF values are uploaded (default) and when the whole tensor is."""
    monkeypatch.setenv("EKP_PROCESS_PAF_UPLOAD", upload)
    g = golden(scene)
    pk = g["ref_peaks"]
    h, w = g["heat"].shape[:2]
    paf_up = np.repeat(np.repeat(g["paf"], 8, axis=0), 8, axis=1)
    if len(pk) == 0:
        return  # the reference never calls process_paf without peaks (paf_to_pose.py:354)
    assert ek.pafprocess.process_paf(pk[None], np.zeros((8 * h, 8 * w, 19), np.float32), paf_up) == 0
    n, cids, scores = _compat_subset(ek)
    want = g["ref_subset"]
    assert n == len(want)
    assert np.array_equal(cids, want[:, :18].astype(np.int32))
    assert_bits_equal(scores, (want[:, 18] / want[:, 19]).astype(np.float32), "human score")
    for cid in range(len(pk)):
        assert ek.pafprocess.get_part_x(cid) == int(g["ref_line_x"][cid])
        assert ek.pafprocess.get_part_y(cid) == int(g["ref_line_y"][cid])
        assert np.float32(ek.pafprocess.get_part_score(cid)).view(np.uint32) == g["ref_line_score"][cid].view(np.uint32)


def test_process_paf_stream_of_frames(ek):
    """A video stream through the operator surface: frames with 1-7 people at two shapes, one after the other in one process.
    Small scenes are replayed as one CUDA graph launch per call (fixed block layout, the peak count travels in the block; a
    graph per shape and sample size class), bigger ones take the eager path: every frame's people, scores and the
    part-sorted table behind the getters are the oracle's."""
    from torch_ekpose_b200 import synthetic
    fe = util.frontend()
    frames = [(46, 54, p, 700 + i) for i, p in enumerate([1, 3, 2, 6, 1, 7, 4, 2])] + [(46, 82, p, 720 + i) for i, p in enumerate([2, 5, 3])] + \
             [(46, 54, p, 740 + i) for i, p in enumerate([3, 0, 5])]
    for (h, w, people, seed) in frames:
        heat, paf = synthetic.make_scene(h, w, people, seed)
        peaks = fe.ref_nms(heat)
        paf_up = fe.upsample_nearest(paf)
        if len(peaks) == 0:
            continue
        sub, line = util.oracle_people(peaks, 8 * h, 8 * w, paf_up)
        assert ek.pafprocess.process_paf(peaks[None], np.zeros((8 * h, 8 * w, 19), np.float32), paf_up) == 0
        n, cids, scores = _compat_subset(ek)
        assert n == len(sub), (h, w, people)
        assert np.array_equal(cids, sub[:, :18].astype(np.int32))
        if n:
            assert_bits_equal(scores, (sub[:, 18] / sub[:, 19]).astype(np.float32), "human score")
        for cid in range(0, len(peaks), 7):
            assert ek.pafprocess.get_part_x(cid) == int(line[0][cid]) and ek.pafprocess.get_part_y(cid) == int(line[1][cid])
            assert np.float32(ek.pafprocess.get_part_score(cid)).view(np.uint32) == np.float32(line[2][cid]).view(np.uint32)


@pytest.mark.parametrize("seed", range(4))
def test_process_paf_host_entry_fuzz(ek, seed):
    """The host-pointer operator surface on adversarial scenes (piecewise-constant PAF: exact score ties, merges, connections
    across people; fractional and border coordinates, which the sample positions' float arithmetic sees), sized to take each
    of its routes: the zero-copy graph (a few people), the listed upload (dozens), positions listed by a kernel (a crowd).
    People, scores and the getter table against the compiled reference."""
    rng = np.random.default_rng(4100 + seed)
    H, W = 128, 192
    for people, drop, block, levels in [(1, 0.0, 8, [1.0]), (3, 0.0, 8, [0.0, 1.0]), (5, 0.2, 16, [-1.0, 0.0, 0.5, 1.0]), (2, 0.5, 4, [0.5, 1.0]),
                                        (14, 0.3, 16, [0.0, 0.25, 1.0]), (30, 0.15, 8, [0.0, 0.25, 1.0]), (70, 0.2, 4, [-0.5, 0.0, 0.5, 1.0])]:
        peaks, paf = _fuzz_scene(rng, H, W, people, drop, block, levels)
        if len(peaks) == 0:
            continue
        peaks = peaks.copy()
        frac = rng.random(len(peaks)) < 0.3   # the reference truncates float coordinates (pafprocess.cpp:30-31)
        peaks[frac, 0] = np.minimum(peaks[frac, 0] + rng.random(int(frac.sum())).astype(np.float32) * 0.99, np.float32(W - 1))
        peaks[frac, 1] = np.minimum(peaks[frac, 1] + rng.random(int(frac.sum())).astype(np.float32) * 0.99, np.float32(H - 1))
        edge = rng.random(len(peaks)) < 0.1
        peaks[edge, 0] = rng.choice([0.0, W - 1.0], int(edge.sum()))
        sub, line = util.oracle_people(peaks, H, W, paf)
        assert ek.pafprocess.process_paf(peaks[None], np.zeros((H, W, 19), np.float32), paf) == 0
        n, cids, scores = _compat_subset(ek)
        assert n == len(sub), f"{people} people: {n} vs {len(sub)}"
        assert np.array_equal(cids, sub[:, :18].astype(np.int32)), f"{people} people"
        if n:
            assert_bits_equal(scores, (sub[:, 18] / sub[:, 19]).astype(np.float32), "human score")
        for cid in range(0, len(peaks), 11):
            assert ek.pafprocess.get_part_x(cid) == int(line[0][cid]) and ek.pafprocess.get_part_y(cid) == int(line[1][cid])


def test_process_paf_pools_all_p1_images(ek):
    """peaks[p1, p2, p3]: the reference walks every (p1, p2) row into ONE peak list (pafprocess.cpp:26-36)."""
    g = golden("c2_46x54_p6")
    pk = g["ref_peaks"]
    n = len(pk) // 2 * 2
    h, w = g["heat"].shape[:2]
    paf_up = np.repeat(np.repeat(g["paf"], 8, axis=0), 8, axis=1)
    heat_up = np.zeros((8 * h, 8 * w, 19), np.float32)
    assert ek.pafprocess.process_paf(pk[None, :n], heat_up, paf_up) == 0
    flat = _compat_subset(ek)
    assert ek.pafprocess.process_paf(pk[:n].reshape(2, n // 2, 5), heat_up, paf_up) == 0
    pooled = _compat_subset(ek)
    assert flat[0] == pooled[0] > 0 and np.array_equal(flat[1], pooled[1])
    assert_bits_equal(flat[2], pooled[2], "human scores")
    sub, _ = util.oracle_people(pk[:n], 8 * h, 8 * w, paf_up)
    assert flat[0] == len(sub) and np.array_equal(flat[1], sub[:, :18].astype(np.int32))


def test_process_paf_rejects_bad_input(ek):
    paf = np.zeros((16, 16, 38), np.float32)
    bad_part = np.array([[(1, 1, .5, 0, 18)]], np.float32)
    with pytest.raises(ValueError):
        ek.pafprocess.process_paf(bad_part, np.zeros((16, 16, 19), np.float32), paf)
    outside = np.array([[(99, 1, .5, 0, 1)]], np.float32)
    with pytest.raises(ValueError):
        ek.pafprocess.process_paf(outside, np.zeros((16, 16, 19), np.float32), paf)
    with pytest.raises(TypeError):
        ek.pafprocess.process_paf(np.zeros((2, 5), np.float32), np.zeros((16, 16, 19), np.float32), paf)
    # zero peaks: zero humans, no error
    assert ek.pafprocess.process_paf(np.zeros((1, 0, 5), np.float32), np.zeros((16, 16, 19), np.float32), paf) == 0
    assert ek.pafprocess.get_num_humans() == 0


# ---------------------------------------------------------------------------------------------
# reference front-end (stages 1-3 as the reference's Python does them) + stages 4-5
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("scene", util.SCENES)
def test_reference_frontend_golden(pp, scene, layout):
    g = golden(scene)
    heat = _dev(_nchw(g["heat"]) if layout == "nchw" else g["heat"][None])
    paf = _dev(_nchw(g["paf"]) if layout == "nchw" else g["paf"][None])
    pp.run(heat, paf, layout=layout, frontend="reference")
    res = pp.results(with_peaks=True)
    got = util.peaks_table(res, 0)
    want = g["ref_peaks"]           # reference NMS() with OpenCV's own bicubic code
    assert got.shape == want.shape
    assert np.array_equal(got[:, [0, 1, 3, 4]], want[:, [0, 1, 3, 4]])      # coords, ids, parts: exact
    assert_bits_equal(got[:, 2], want[:, 2], "peak score vs cv2 (IPP off)")
    want_ipp = g["ref_peaks_ipp"]   # cv2 default build (IPP): same coordinates, scores to 2.5e-7
    assert np.array_equal(got[:, [0, 1, 3, 4]], want_ipp[:, [0, 1, 3, 4]])
    if len(want_ipp):
        assert np.abs(got[:, 2] - want_ipp[:, 2]).max() <= 2.5e-7
    n = int(res["num_humans"][0])
    assert n == len(g["ref_subset"])
    assert_bits_equal(res["subset"][0, :n], g["ref_subset"], "subset")
    # person count and part indices also equal the reference run with IPP on
    assert np.array_equal(res["subset"][0, :n, :18], g["ref_subset_ipp"][:, :18])


@pytest.mark.parametrize("scene", util.SCENES)
def test_paf_to_pose_cpp_dropin(ek, scene):
    """The reference-facing function: numpy HWC in, list[Human] out, equal to the reference's humans."""
    g = golden(scene)
    humans = ek.paf_to_pose_cpp(g["heat"], g["paf"], ek.cfg)
    want_parts, want_score = g["ref_humans_parts"], g["ref_humans_score"]
    assert len(humans) == len(want_score)
    for k, hm in enumerate(humans):
        assert hm.score == want_score[k]
        present = {int(i) for i in np.nonzero(want_parts[k, :, 0])[0]}
        assert set(hm.body_parts) == present
        for part, bp in hm.body_parts.items():
            assert bp.uidx == "%d-%d" % (k, part) and bp.part_idx == part
            assert (bp.x, bp.y, bp.score) == tuple(want_parts[k, part, 1:])
    # a transposed view of a CHW array (what estimator.get_outputs returns) takes the no-copy route
    chw_h = np.ascontiguousarray(g["heat"].transpose(2, 0, 1))
    chw_p = np.ascontiguousarray(g["paf"].transpose(2, 0, 1))
    humans2 = ek.paf_to_pose_cpp(chw_h.transpose(1, 2, 0), chw_p.transpose(1, 2, 0), ek.cfg)
    assert [sorted(h.body_parts) for h in humans2] == [sorted(h.body_parts) for h in humans]


def test_nms_dropin(ek):
    g = golden("c2_46x54_p6")
    lists = ek.NMS(g["heat"], upsampFactor=8, config=ek.cfg)
    flat = np.array([tuple(r) + (k,) for k, rows in enumerate(lists) for r in rows], np.float32)
    assert_bits_equal(flat, g["ref_peaks"], "NMS joint list")


@pytest.mark.parametrize("scene", ["border"] + util.SCENES)
def test_nms_with_gaussian_filter_dropin(ek, scene):
    """NMS(bool_gaussian_filt=True) (paf_to_pose.py:111-112: scipy's gaussian_filter(sigma=3) on every upsampled patch,
    double arithmetic, float32 between the two axis passes) against the reference's own Python + SciPy output on the golden
    scenes and on a map with peaks in the corners, on the edges and next to them (clipped 3x3 ... 4x5-cell windows), and
    against the oracle: coordinates, ids and float32 scores bit-identical."""
    g = golden("nms_gauss")
    heat = g["border_heat"] if scene == "border" else golden(scene)["heat"]
    lists = ek.NMS(heat, upsampFactor=8, bool_gaussian_filt=True, config=ek.cfg)
    assert len(lists) == 18 and all(a.dtype == np.float64 and a.shape[1:] == (4,) for a in lists)
    flat = np.array([tuple(r) + (k,) for k, rows in enumerate(lists) for r in rows], np.float64).reshape(-1, 5)
    assert_bits_equal(flat, g[scene + "_peaks"], "NMS(bool_gaussian_filt=True) joint list vs the reference's")
    assert_bits_equal(flat.astype(np.float32), util.frontend().ref_nms(heat, gauss=True), "vs the oracle")
    if scene == "border":   # the same clipped windows through the plain refinement, against the reference's own output
        plain = ek.NMS(heat, upsampFactor=8, config=ek.cfg)
        flat0 = np.array([tuple(r) + (k,) for k, rows in enumerate(plain) for r in rows], np.float64).reshape(-1, 5)
        assert_bits_equal(flat0, g["border_peaks_plain"], "NMS() on the border map vs the reference's")
        assert (flat0[:, :2] != flat[:, :2]).any() or (flat0[:, 2] != flat[:, 2]).any()   # the filter does change something
    # the filter has no effect without refinement (:103-122), as in the reference
    a = ek.NMS(heat, upsampFactor=8, bool_refine_center=False, bool_gaussian_filt=True, config=ek.cfg)
    b = ek.NMS(heat, upsampFactor=8, bool_refine_center=False, config=ek.cfg)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))


def test_gaussian_refinement_in_a_batch_equals_the_oracle(ek):
    """frontend='reference_gauss' through the batched entry (NCHW, 8 images, people included): the peak tables and the
    people are the oracle's for NMS(bool_gaussian_filt=True) peaks."""
    from torch_ekpose_b200 import synthetic
    heat, paf = synthetic.make_batch(8, 46, 82, (2, 8), seed=91)
    p = ek.PostProcessor(device=0, max_batch=8, max_h=46, max_w=82, max_peaks=1024, max_humans=64)
    import torch
    p.run(torch.from_numpy(heat).cuda(), torch.from_numpy(paf).cuda(), frontend="reference_gauss")
    res = p.results(with_peaks=True)
    fe = util.frontend()
    for i in range(8):
        hw = np.ascontiguousarray(heat[i].transpose(1, 2, 0)); pw = np.ascontiguousarray(paf[i].transpose(1, 2, 0))
        peaks = fe.ref_nms(hw, gauss=True)
        sub, line = util.oracle_people(peaks, 368, 656, fe.upsample_nearest(pw))
        n = int(res["num_humans"][i])
        assert n == len(sub) and int(res["n_peaks"][i]) == len(peaks)
        assert_bits_equal(res["subset"][i, :n], sub, f"image {i}")
        rows = res["peaks"][i][:len(peaks)]
        assert np.array_equal(rows["x"], line[0]) and np.array_equal(rows["y"], line[1])
        assert_bits_equal(rows["score"], line[2])
    p.close()


def _find_peaks_reference(param, img):
    """The reference's own expression, paf_to_pose.py:34-36 (SciPy is the primitive it imports, :4-6)."""
    from scipy.ndimage import generate_binary_structure, maximum_filter
    peaks_binary = (maximum_filter(img, footprint=generate_binary_structure(2, 1)) == img) * (img > param)
    return np.array(np.nonzero(peaks_binary)[::-1]).T


def test_find_peaks_dropin(ek):
    """find_peaks (SURVEY 8a row a1): plateaus give several peaks, borders compare with in-bounds neighbours only."""
    rng = np.random.default_rng(3)
    for shape, levels in [((46, 54), None), ((23, 31), 6), ((5, 5), 3), ((92, 164), 40)]:
        img = rng.random(shape).astype(np.float32)
        if levels:
            img = (np.floor(img * levels) / levels).astype(np.float32)   # exact ties, plateaus
        for thr in (0.15, 0.5, -1.0):
            got = ek.find_peaks(thr, img)
            want = _find_peaks_reference(np.float32(thr), img)
            assert got.shape == want.shape and np.array_equal(got, want), (shape, levels, thr)
    assert np.array_equal(ek.compute_resized_coords([1, 2], 2), [2.5, 4.5])     # the example of paf_to_pose.py:43-44


@pytest.mark.parametrize("scene", ["c2_46x54_p6", "c4_crowd_64x96_p24", "empty_46x54"])
def test_nms_without_refinement_and_people(ek, scene):
    """NMS(bool_refine_center=False) (paf_to_pose.py:119-125) and the people stages 4-5 build from those peaks."""
    g = golden(scene)
    heat, paf = g["heat"], g["paf"]
    lists = ek.NMS(heat, upsampFactor=8, bool_refine_center=False, config=ek.cfg)
    want, cnt = [], 0
    for k in range(18):
        pk = _find_peaks_reference(np.float32(0.15), heat[:, :, k])
        arr = np.zeros((len(pk), 4))
        for i, p_ in enumerate(pk):
            arr[i] = tuple(ek.compute_resized_coords(p_, 8)) + (heat[p_[1], p_[0], k], cnt)
            cnt += 1
        want.append(arr)
    for k in range(18):
        assert lists[k].shape == want[k].shape and np.array_equal(lists[k], want[k]), k
    h, w = heat.shape[:2]
    pp2 = ek.PostProcessor(device=0, max_batch=1, max_h=h, max_w=w, max_peaks=2048, max_humans=128)
    pp2.run(heat[None], paf[None], layout="nhwc", frontend="reference_coarse")
    res = pp2.results()
    pp2.close()
    peaks = np.array([tuple(r) + (k,) for k, rows in enumerate(want) for r in rows], np.float32).reshape(-1, 5)
    if len(peaks):
        sub, _ = util.oracle_people(peaks, 8 * h, 8 * w, util.frontend().upsample_nearest(paf))
    else:
        sub = np.zeros((0, 20), np.float32)
    m = int(res["num_humans"][0])
    assert m == len(sub)
    assert_bits_equal(res["subset"][0, :m], sub, "subset")


# ---------------------------------------------------------------------------------------------
# dense front-end (north_star stages 1-3) + stages 4-5
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("materialize", [True, False])
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("scene", util.SCENES)
def test_dense_frontend_golden(pp, scene, layout, materialize):
    g = golden(scene)
    heat = _dev(_nchw(g["heat"]) if layout == "nchw" else g["heat"][None])
    paf = _dev(_nchw(g["paf"]) if layout == "nchw" else g["paf"][None])
    pp.run(heat, paf, layout=layout, frontend="dense", materialize=materialize)
    res = pp.results(with_peaks=True)
    got = util.peaks_table(res, 0)
    assert_bits_equal(got, g["dense_peaks"], "dense peaks")
    n = int(res["num_humans"][0])
    assert n == len(g["dense_subset"])
    assert_bits_equal(res["subset"][0, :n], g["dense_subset"], "dense subset (people from the compiled reference)")
    if materialize:
        ys, xs = g["probe_yx"][:, 0], g["probe_yx"][:, 1]
        assert_bits_equal(pp.paf_mat[0].cpu().numpy()[ys, xs], g["probe_paf_mat"], "paf_mat probes")
        assert_bits_equal(pp.heat_mat[0].cpu().numpy()[ys, xs], g["probe_heat_mat"], "heat_mat probes")


@pytest.mark.parametrize("shape", [(46, 54), (46, 82), (33, 40), (5, 5), (7, 70)])
def test_dense_tensors_vs_oracle(pp, shape):
    """Whole smoothed map and both operator-surface tensors, every element, against the oracle."""
    from torch_ekpose_b200 import synthetic
    h, w = shape
    heat, paf = synthetic.make_scene(h, w, 3, 77 + h * w)
    fe = util.frontend()
    sm = pp.dense_smooth(_dev(_nchw(heat))).cpu().numpy()[0]
    assert_bits_equal(sm, fe.dense_smooth(heat), "smoothed heat map")
    pp.run(_dev(_nchw(heat)), _dev(_nchw(paf)), frontend="dense", materialize=True)
    pp.results()
    assert_bits_equal(pp.paf_mat[0].cpu().numpy(), fe.upsample_bilinear(paf), "paf_mat")
    assert_bits_equal(pp.heat_mat[0].cpu().numpy(), fe.upsample_bilinear(heat), "heat_mat")


def test_nearest_operator_surface(pp):
    """REFERENCE front-end with materialisation: paf_mat / heat_mat == cv2 INTER_NEAREST x8."""
    g = golden("c1_46x54_p3")
    pp.run(_dev(_nchw(g["heat"])), _dev(_nchw(g["paf"])), frontend="reference", materialize=True)
    pp.results()
    assert np.array_equal(pp.paf_mat[0].cpu().numpy(), np.repeat(np.repeat(g["paf"], 8, 0), 8, 1))
    assert np.array_equal(pp.heat_mat[0].cpu().numpy(), np.repeat(np.repeat(g["heat"], 8, 0), 8, 1))


# ---------------------------------------------------------------------------------------------
# BASELINE.json configurations, batched, against the live oracle
# ---------------------------------------------------------------------------------------------
def _check_batch(pp, heat, paf, frontend, materialize, images):
    pp.run(_dev(heat), _dev(paf), frontend=frontend, materialize=materialize)
    res = pp.results(with_peaks=True)
    assert not res["overflow"].any()
    for i in images:
        hw, pw = np.ascontiguousarray(heat[i].transpose(1, 2, 0)), np.ascontiguousarray(paf[i].transpose(1, 2, 0))
        peaks, sub = (util.oracle_dense if frontend == "dense" else util.oracle_reference)(hw, pw)
        assert_bits_equal(util.peaks_table(res, i), peaks, f"image {i} peaks")
        n = int(res["num_humans"][i])
        assert n == len(sub), f"image {i}: {n} humans vs {len(sub)}"
        assert_bits_equal(res["subset"][i, :n], sub, f"image {i} subset")
    return res


@pytest.mark.parametrize("frontend,materialize", [("dense", True), ("dense", False), ("reference", False)])
def test_config2_batch64_368x432(pp, frontend, materialize):
    from torch_ekpose_b200 import synthetic
    heat, paf = synthetic.make_batch(64, 46, 54, (1, 6), seed=2)
    res = _check_batch(pp, heat, paf, frontend, materialize, range(64))   # every image of the batch
    assert res["num_humans"].sum() > 150


@pytest.mark.parametrize("frontend", ["dense", "reference"])
def test_config3_656x368(pp, frontend):
    from torch_ekpose_b200 import synthetic
    heat, paf = synthetic.make_batch(32, 46, 82, (2, 8), seed=3)
    _check_batch(pp, heat, paf, frontend, frontend == "dense", range(32))


@pytest.mark.parametrize("frontend,materialize", [("dense", True), ("dense", False), ("reference", False)])
def test_config3_full_batch_256(ek, frontend, materialize):
    """configs[2] at its full size: 256 frames of 656x368 in ONE batch, every image checked against the oracle."""
    from torch_ekpose_b200 import synthetic
    heat, paf = synthetic.make_batch(256, 46, 82, (2, 8), seed=33)
    big = ek.PostProcessor(device=0, max_batch=256, max_h=46, max_w=82, max_peaks=1024, max_humans=32, max_part=64, max_cand=512)
    res = _check_batch(big, heat, paf, frontend, materialize, range(256))
    assert res["num_humans"].sum() > 1000
    big.close()


@pytest.mark.parametrize("frontend", ["dense", "reference"])
def test_config4_crowded_1312x736(pp, frontend):
    """30-40 people per image: >16 candidates per limb with exact score ties (std::sort emulation)."""
    from torch_ekpose_b200 import synthetic
    heat, paf = synthetic.make_batch(4, 92, 164, (30, 40), seed=4)
    res = _check_batch(pp, heat, paf, frontend, False, range(4))
    assert res["num_humans"].min() >= 25
    ref = util.ref_or_none()
    if ref is not None and frontend == "reference":   # and straight against the compiled reference
        hw, pw = np.ascontiguousarray(heat[0].transpose(1, 2, 0)), np.ascontiguousarray(paf[0].transpose(1, 2, 0))
        fe = util.frontend()
        sub, _ = util.oracle_people(fe.ref_nms(hw), 736, 1312, fe.upsample_nearest(pw), impl=ref)
        assert_bits_equal(res["subset"][0, :len(sub)], sub, "vs compiled reference")


@pytest.mark.parametrize("frontend", ["dense", "reference"])
def test_heavy_crowds_up_to_80_people(ek, frontend):
    """Stage 4 in its one-thread-per-pair regime (two exact passes over thousands of pairs per limb) and the assembly with
    60+ rows, on 1312x736 scenes with 34-38 and 80 people, run three times on the same context (graph replays included),
    against the oracle."""
    from torch_ekpose_b200 import synthetic
    heat, paf = synthetic.make_batch(2, 92, 164, (34, 38), seed=44)
    h80, p80 = synthetic.make_batch(1, 92, 164, (80, 80), seed=45)
    big = ek.PostProcessor(device=0, max_batch=3, max_h=92, max_w=164, max_peaks=4096, max_humans=256, max_part=256, max_cand=4096)
    for _ in range(3):
        res = _check_batch(big, np.concatenate([heat, h80]), np.concatenate([paf, p80]), frontend, False, range(3))
        assert int(res["num_humans"][2]) >= 60
        assert int(res["n_peaks"][2]) >= 900
    big.close()


@pytest.mark.parametrize("materialize", [True, False])
def test_large_map_2624x1472(ek, materialize):
    """A map four times the area of the largest BASELINE shape (184 x 328 stride-8 cells, 12 column tiles): tile
    geometry, halos and the store chunking far from the shapes the kernels were tuned on, against the oracle."""
    from torch_ekpose_b200 import synthetic
    heat, paf = synthetic.make_batch(1, 184, 328, (20, 20), seed=4)
    big = ek.PostProcessor(device=0, max_batch=1, max_h=184, max_w=328, max_peaks=2048, max_humans=128)
    res = _check_batch(big, heat, paf, "dense", materialize, [0])
    assert int(res["num_humans"][0]) >= 18
    if materialize:  # and the operator-surface tensors themselves, whole-tensor bit comparison
        fe = util.frontend()
        pw = np.ascontiguousarray(paf[0].transpose(1, 2, 0))
        assert_bits_equal(big.paf_mat[0].cpu().numpy(), fe.upsample_bilinear(pw), "paf_mat")
    big.close()


# ---------------------------------------------------------------------------------------------
# size-independent properties at full batch sizes
# ---------------------------------------------------------------------------------------------
def test_properties_batch_layout_materialise_invariance(pp):
    from torch_ekpose_b200 import synthetic
    heat, paf = synthetic.make_batch(64, 46, 54, (1, 6), seed=9)
    hd, pd = _dev(heat), _dev(paf)

    def run(hh, ppp, **kw):
        pp.run(hh, ppp, **kw)
        r = pp.results(with_peaks=True)
        return r

    a = run(hd, pd, frontend="dense", materialize=True)
    b = run(hd, pd, frontend="dense", materialize=False)                     # lean == materialised
    c = run(hd.permute(0, 2, 3, 1).contiguous(), pd.permute(0, 2, 3, 1).contiguous(), layout="nhwc", frontend="dense")
    d = run(hd.flip(0).contiguous(), pd.flip(0).contiguous(), frontend="dense", materialize=True)  # batch order
    e = run(hd, pd, frontend="dense", materialize=True)                      # determinism (atomics order)
    for other, flip in ((b, False), (c, False), (d, True), (e, False)):
        for k in ("num_humans", "n_peaks"):
            assert np.array_equal(a[k], other[k][::-1] if flip else other[k])
        sub = other["subset"][::-1] if flip else other["subset"]
        pk = other["peaks"][::-1] if flip else other["peaks"]
        for i in range(64):
            n, m = int(a["num_humans"][i]), int(a["n_peaks"][i])
            assert_bits_equal(a["subset"][i, :n], sub[i, :n])
            assert np.array_equal(a["peaks"][i][:m], pk[i][:m])
    # single-image runs equal the batched result
    for i in (0, 17, 63):
        s = run(hd[i:i + 1], pd[i:i + 1], frontend="dense")
        n = int(a["num_humans"][i])
        assert int(s["num_humans"][0]) == n
        assert_bits_equal(s["subset"][0, :n], a["subset"][i, :n])


def test_run_peaks_random_lists_vs_oracle(pp):
    """Stage 4-5 device entry: unsorted peak lists with duplicates, random PAF."""
    rng = np.random.default_rng(5)
    n, H, W, stride = 6, 96, 128, 160
    paf = rng.normal(0, 0.6, (n, H, W, 38)).astype(np.float32)
    peaks = np.zeros((n, stride, 5), np.float32)
    counts = np.array([0, 1, 40, 90, 160, 120], np.int32)
    for i in range(n):
        k = counts[i]
        peaks[i, :k, 0] = rng.integers(0, W, k)
        peaks[i, :k, 1] = rng.integers(0, H, k)
        peaks[i, :k, 2] = rng.random(k)
        peaks[i, :k, 4] = rng.integers(0, 18, k)
        if k > 10:
            peaks[i, 5:10, :2] = peaks[i, 0:5, :2]   # duplicate coordinates
    pp.run_peaks(_dev(peaks), _dev(counts), _dev(paf), h1=H)
    res = pp.results(with_peaks=True)
    for i in range(n):
        if counts[i] == 0:
            assert res["num_humans"][i] == 0
            continue
        sub, line = util.oracle_people(peaks[i, :counts[i]], H, W, paf[i])
        m = int(res["num_humans"][i])
        assert m == len(sub)
        assert_bits_equal(res["subset"][i, :m], sub, f"image {i}")
        got = res["peaks"][i][:counts[i]]
        assert np.array_equal(got["x"], line[0]) and np.array_equal(got["id"], line[3])


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


@pytest.mark.parametrize("seed", range(6))
def test_stage45_adversarial_fuzz_vs_oracle(ek, seed):
    """Stages 4-5 on scenes built to hit every branch of the assembly and the sort: > 32 connections per
    limb, connections that match two or three rows, merges, exact score ties among > 16 candidates (the
    std::sort replay), unsorted input.  subset rows must equal the oracle's bit for bit."""
    rng = np.random.default_rng(1000 + seed)
    H, W = 128, 192
    cases = []
    for people, drop, block, levels in [(4, 0.0, 8, [0.0, 1.0]), (12, 0.3, 16, [-1.0, 0.0, 0.5, 1.0]), (40, 0.15, 8, [0.0, 0.25, 1.0]),
                                        (60, 0.5, 32, [0.5, 1.0]), (90, 0.2, 4, [-0.5, 0.0, 0.5, 1.0]), (25, 0.6, 64, [1.0])]:
        cases.append(_fuzz_scene(rng, H, W, people, drop, block, levels))
    n = len(cases)
    stride = max(len(c[0]) for c in cases)
    peaks = np.zeros((n, stride, 5), np.float32)
    counts = np.array([len(c[0]) for c in cases], np.int32)
    for i, c in enumerate(cases):
        peaks[i, :counts[i]] = c[0]
    paf = np.stack([c[1] for c in cases])
    big = ek.PostProcessor(device=0, max_batch=n, max_h=16, max_w=24, max_peaks=2048, max_humans=512)
    big.run_peaks(_dev(peaks), _dev(counts), _dev(paf), h1=H)
    res = big.results()
    for i in range(n):
        sub, _ = util.oracle_people(peaks[i, :counts[i]], H, W, paf[i])
        m = int(res["num_humans"][i])
        assert m == len(sub), f"case {i}: {m} people vs {len(sub)}"
        assert_bits_equal(res["subset"][i, :m], sub, f"case {i}")
    big.close()
    # the same scenes through a context with few rows (<= 128): the sequential walk then keeps the two compared
    # columns in registers, merges included
    few = [i for i in range(n) if len(cases[i][0]) < 400]
    small = ek.PostProcessor(device=0, max_batch=len(few), max_h=16, max_w=24, max_peaks=1024, max_humans=128)
    small.run_peaks(_dev(peaks[few]), _dev(counts[few]), _dev(paf[few]), h1=H)
    res2 = small.results()
    for j, i in enumerate(few):
        m = int(res["num_humans"][i])
        assert int(res2["num_humans"][j]) == m
        assert_bits_equal(res2["subset"][j, :m], res["subset"][i, :m], f"case {i}, 128-row context")
    small.close()


@pytest.mark.parametrize("C,offset", [(38, 0), (38, 1), (39, 0), (40, 0), (41, 3)])
def test_run_peaks_channel_counts_and_alignment(ek, C, offset):
    """process_paf indexes paf[ch + f3 * (x + f2 * y)] for any f3 >= 38 (pafprocess.cpp:8): odd channel counts and
    bases that are only 4-byte aligned take the two-load gather, even ones the 8-byte gather; same people."""
    rng = np.random.default_rng(C * 10 + offset)
    H, W = 96, 128
    peaks, paf38 = _fuzz_scene(rng, H, W, 10, 0.2, 8, [0.0, 0.5, 1.0])
    paf = rng.normal(0, 1, (H, W, C)).astype(np.float32)
    paf[:, :, :38] = paf38
    buf = torch.zeros(paf.size + offset, dtype=torch.float32, device="cuda")
    view = buf[offset:].view(1, H, W, C)
    view.copy_(torch.from_numpy(paf)[None])
    pp_ = ek.PostProcessor(device=0, max_batch=1, max_h=12, max_w=16, max_peaks=1024, max_humans=128)
    pp_.run_peaks(_dev(peaks[None]), _dev(np.array([len(peaks)], np.int32)), view, h1=H)
    res = pp_.results()
    sub, _ = util.oracle_people(peaks, H, W, paf)
    m = int(res["num_humans"][0])
    assert m == len(sub) and m > 0
    assert_bits_equal(res["subset"][0, :m], sub, "subset")
    pp_.close()


# ---------------------------------------------------------------------------------------------
# capacity and argument errors are reported, never silent
# ---------------------------------------------------------------------------------------------
def test_overflow_is_reported(ek):
    from torch_ekpose_b200 import synthetic
    heat, paf = synthetic.make_batch(2, 46, 54, (6, 6), seed=1)
    small = ek.PostProcessor(device=0, max_batch=2, max_h=46, max_w=54, max_peaks=16, max_humans=2)
    small.run(_dev(heat), _dev(paf), frontend="dense")
    with pytest.raises(ek._lib.EkpCapacityError):
        small.results()
    small.close()


def test_inputs_that_are_only_4_byte_aligned(ek):
    """Device inputs at an odd float offset (views into a bigger buffer): same people as the aligned tensors."""
    from torch_ekpose_b200 import synthetic
    heat, paf = synthetic.make_batch(3, 46, 54, (2, 4), seed=9)
    pp_ = ek.PostProcessor(device=0, max_batch=3, max_h=46, max_w=54, max_peaks=1024, max_humans=32)
    pp_.run(_dev(heat), _dev(paf), frontend="dense", materialize=True)
    want = pp_.results()
    hb = torch.zeros(heat.size + 3, dtype=torch.float32, device="cuda")
    pb = torch.zeros(paf.size + 1, dtype=torch.float32, device="cuda")
    hv, pv = hb[3:].view(heat.shape), pb[1:].view(paf.shape)
    hv.copy_(torch.from_numpy(heat)); pv.copy_(torch.from_numpy(paf))
    assert hv.data_ptr() % 16 != 0 and pv.data_ptr() % 16 != 0
    for materialize in (True, False):
        pp_.run(hv, pv, frontend="dense", materialize=materialize)
        got = pp_.results()
        assert np.array_equal(got["num_humans"], want["num_humans"])
        assert_bits_equal(got["subset"], want["subset"], "subset")
    pp_.close()


@pytest.mark.parametrize("frontend", ["dense", "reference"])
@pytest.mark.parametrize("shape", [(46, 54), (5, 5), (23, 37), (46, 82), (31, 64)])
def test_operator_surface_writes_stay_inside_their_tensors(ek, frontend, shape):
    """compute-sanitizer is not available on the pool, so: heat_mat / paf_mat sit between guard regions filled with a
    sentinel; after the bulk-store (dense) and nearest-upsample (reference) kernels the guards must be untouched and
    every element of the tensors written."""
    from torch_ekpose_b200 import synthetic
    h, w = shape
    n = 3
    heat, paf = synthetic.make_batch(n, h, w, (1, 3), seed=h * 100 + w)
    G = 4096  # floats per guard, keeps the 16-byte alignment of the tensors
    nh, npf = n * 64 * h * w * 19, n * 64 * h * w * 38
    hbuf = torch.full((G + nh + G,), float("nan"), dtype=torch.float32, device="cuda")
    pbuf = torch.full((G + npf + G,), float("nan"), dtype=torch.float32, device="cuda")
    pp_ = ek.PostProcessor(device=0, max_batch=n, max_h=h, max_w=w, max_peaks=1024, max_humans=64)
    lib = ek._lib.lib
    hd, pd = _dev(heat), _dev(paf)
    rc = lib.ekp_postprocess(pp_._ctx, hd.data_ptr(), pd.data_ptr(), n, h, w, ek._lib.LAYOUT_NCHW, 0.15,
                             ek._lib.FRONTEND_DENSE if frontend == "dense" else ek._lib.FRONTEND_REFERENCE,
                             hbuf.data_ptr() + 4 * G, pbuf.data_ptr() + 4 * G, 0)
    assert rc == 0, lib.ekp_last_error()
    torch.cuda.synchronize()
    for buf, cnt in ((hbuf, nh), (pbuf, npf)):
        assert torch.isnan(buf[:G]).all() and torch.isnan(buf[G + cnt:]).all(), "a guard region was written"
        assert not torch.isnan(buf[G:G + cnt]).any(), "part of the tensor was not written"
    fe = util.frontend()
    pw = np.ascontiguousarray(paf[1].transpose(1, 2, 0))
    want = fe.upsample_bilinear(pw) if frontend == "dense" else fe.upsample_nearest(pw)
    got = pbuf[G:G + npf].view(n, 8 * h, 8 * w, 38)[1].cpu().numpy()
    assert_bits_equal(got, want, "paf_mat of image 1")
    pp_.close()


def test_small_context_does_not_shrink_kernel_limits_of_a_big_one(ek):
    """Kernel attributes (dynamic shared memory limits) are per device, not per context: creating a context
    with small capacities after a big one must leave the big one working."""
    from torch_ekpose_b200 import synthetic
    heat, paf = synthetic.make_batch(2, 46, 54, (2, 3), seed=3)
    big = ek.PostProcessor(device=0, max_batch=2, max_h=46, max_w=54, max_peaks=4096, max_humans=512)
    big.run(_dev(heat), _dev(paf), frontend="dense")
    want = big.results()["num_humans"].copy()
    small = ek.PostProcessor(device=0, max_batch=1, max_h=8, max_w=8, max_peaks=16, max_humans=2)
    big.run(_dev(heat), _dev(paf), frontend="dense")
    assert np.array_equal(big.results()["num_humans"], want) and want.sum() > 0
    small.close()
    big.close()


def test_part_and_candidate_capacities_are_reported(ek):
    """More than EKP_MAX_CAND passing pairs on one limb, more than EKP_MAX_PART peaks of one part: flagged per
    image (EKP_OVF_CANDIDATES / EKP_OVF_PART) and raised, never silently truncated; a clean image in the same
    batch is unaffected."""
    H, W = 64, 768
    paf = np.zeros((3, H, W, 38), np.float32)
    paf[:, :, :, 12] = 1.0                                  # limb 0 (neck -> RShoulder) x channel: every pair to the right passes
    def grid(n_a, n_b):
        rows = [(2 + i, 2 + 2 * (i % 20), 0.9, 0, 1) for i in range(n_a)]           # necks on the left
        rows += [(300 + i, 2 + 2 * (i % 20), 0.9, 0, 2) for i in range(n_b)]        # right shoulders far to the right
        return np.array(rows, np.float32)
    cases = [grid(60, 60), grid(3, 300), grid(2, 2)]      # 3600 candidates; 300 peaks of part 2; fine
    stride = max(len(c) for c in cases)
    peaks = np.zeros((3, stride, 5), np.float32)
    counts = np.array([len(c) for c in cases], np.int32)
    for i, c in enumerate(cases):
        peaks[i, :len(c)] = c
    pp_ = ek.PostProcessor(device=0, max_batch=3, max_h=8, max_w=96, max_peaks=1024, max_humans=512)
    pp_.run_peaks(_dev(peaks), _dev(counts), _dev(paf), h1=H)
    with pytest.raises(ek._lib.EkpCapacityError):
        pp_.results()
    res = pp_.results(raise_on_overflow=False)
    assert res["overflow"][0] & ek._lib.OVF_CANDIDATES and not res["overflow"][0] & ek._lib.OVF_PART
    assert res["overflow"][1] & ek._lib.OVF_PART
    assert res["overflow"][2] == 0
    sub, _ = util.oracle_people(cases[2], H, W, paf[2])
    assert int(res["num_humans"][2]) == len(sub)
    pp_.close()


def test_argument_errors(ek, pp):
    from torch_ekpose_b200 import synthetic
    heat, paf = synthetic.make_batch(1, 46, 54, (1, 1), seed=1)
    with pytest.raises(ValueError):
        pp.run(_dev(heat), _dev(paf[:, :37]), frontend="dense")
    tiny = _dev(np.zeros((1, 19, 4, 4), np.float32)), _dev(np.zeros((1, 38, 4, 4), np.float32))
    with pytest.raises(ek._lib.EkpError):
        pp.run(*tiny, frontend="dense")
    big = _dev(np.zeros((65, 19, 5, 5), np.float32)), _dev(np.zeros((65, 38, 5, 5), np.float32))
    with pytest.raises(ek._lib.EkpError):
        pp.run(*big, frontend="dense")
    # operator-surface tensors that are not 16-byte aligned are refused (they are written with 16-byte bulk copies)
    hd, pd = _dev(heat), _dev(paf)
    hm = torch.empty(368 * 432 * 19 + 4, dtype=torch.float32, device="cuda")
    pm = torch.empty(368 * 432 * 38 + 4, dtype=torch.float32, device="cuda")
    lib = ek._lib.lib
    args = (pp._ctx, hd.data_ptr(), pd.data_ptr(), 1, 46, 54, ek._lib.LAYOUT_NCHW, 0.15, ek._lib.FRONTEND_DENSE)
    rc = lib.ekp_postprocess(*args, hm.data_ptr() + 4, pm.data_ptr() + 4, 0)
    assert rc == ek._lib.ERR_ARG and b"16-byte aligned" in lib.ekp_last_error()
    rc = lib.ekp_postprocess(*args, hm.data_ptr(), pm.data_ptr(), 0)
    assert rc == 0, lib.ekp_last_error()
    torch.cuda.synchronize()


@pytest.mark.parametrize("people", [20, 50, 100, 150])
def test_assembly_paths_by_people_count(ek, people):
    """20 / 50 / 100 / 150 four-part people in one image: one chunk of connections per limb and several (the
    assembly takes one lane per connection, 32 at a time); all must equal the oracle bit for bit."""
    H, W = 32, 40 * people + 24
    paf = np.zeros((1, H, W, 38), np.float32)
    rows = []
    rng = np.random.default_rng(people)
    for i in range(people):
        y, x0 = 8 + (i % 3) * 6, 8 + 40 * i
        for k, part in enumerate((1, 2, 3, 4)):      # neck -> RShoulder -> RElbow -> RWrist, 8 px apart
            rows.append((x0 + 8 * k, y, 0.5 + 0.4 * rng.random(), 0, part))
        paf[0, y - 1:y + 2, x0 - 1:x0 + 26, 12] = 1     # limb 0 (1->2), 2 (2->3), 3 (3->4): x channels 12, 14, 16
        paf[0, y - 1:y + 2, x0 - 1:x0 + 26, 14] = 1
        paf[0, y - 1:y + 2, x0 - 1:x0 + 26, 16] = 1
    peaks = np.array(rows, np.float32)
    peaks = peaks[rng.permutation(len(peaks))][None]            # unsorted input on purpose
    big = ek.PostProcessor(device=0, max_batch=1, max_h=8, max_w=8, max_peaks=1024, max_humans=256)
    big.run_peaks(_dev(peaks), _dev(np.array([peaks.shape[1]], np.int32)), _dev(paf), h1=H)
    res = big.results()
    sub, _ = util.oracle_people(peaks[0], H, W, paf[0])
    assert len(sub) == people == int(res["num_humans"][0])
    assert_bits_equal(res["subset"][0, :people], sub, "subset")
    big.close()


def test_batched_handoff_from_the_network(ek):
    """Row f1: a (fake) network emits CUDA tensors for a batch of frames; infer_humans must give the
    people paf_to_pose_cpp gives frame by frame on host copies."""
    from torch_ekpose_b200 import estimator, synthetic
    heat, paf = synthetic.make_batch(3, 46, 54, (2, 4), seed=21)

    class FakeNet(torch.nn.Module):
        def forward(self, x):
            # get_outputs scales the LONG side to 368 (estimator.py:59,73): 368x432 -> 313x368 -> padded 320x368
            assert x.shape == (3, 3, 320, 368) and x.is_cuda
            return (torch.from_numpy(paf).to(x.device), torch.from_numpy(heat).to(x.device)), None

    frames = [np.zeros((368, 432, 3), np.uint8) for _ in range(3)]
    dev = torch.device("cuda", torch.cuda.device_count() - 1)   # the tensors' device decides, not device 0
    got = estimator.infer_humans(frames, FakeNet(), "vgg", dev)
    assert estimator.last_postprocessor().device == dev.index
    fe = util.frontend()
    for i in range(3):
        # the ORACLE on the same maps: reference front-end restatement + the compiled reference process_paf, then the
        # getter loop of paf_to_pose_cpp (paf_to_pose.py:361-377) restated on its tables
        hw, pw = np.ascontiguousarray(heat[i].transpose(1, 2, 0)), np.ascontiguousarray(paf[i].transpose(1, 2, 0))
        peaks = fe.ref_nms(hw)
        sub, line = util.oracle_people(peaks, 368, 432, fe.upsample_nearest(pw))
        assert len(got[i]) == len(sub) > 0
        for hm, row in zip(got[i], sub):
            assert np.float32(hm.score) == np.float32(row[18]) / np.float32(row[19])
            cids = {k: int(row[k]) for k in range(18) if int(row[k]) >= 0}
            assert sorted(hm.body_parts) == sorted(cids)
            for k, cid in cids.items():
                bp = hm.body_parts[k]
                assert (bp.x, bp.y) == (float(line[0][cid]) / 432, float(line[1][cid]) / 368)
                assert np.float32(bp.score) == line[2][cid] and bp.uidx == "%d-%d" % (got[i].index(hm), k)


@pytest.mark.parametrize("scene", util.SCENES)
def test_coco_results_equal_the_reference_append_result(ek, pp, scene):
    """Row f3 end to end on the GPU: maps -> CUDA post-processing (reference front-end) -> vectorised COCO conversion must
    equal what the reference's own append_result (eval.py:93-125, executed unmodified by make_golden.py) produced from the
    reference's paf_to_pose_cpp humans."""
    from torch_ekpose_b200 import coco
    fx = golden("coco_append_result")
    g = golden(scene)
    h, w = g["heat"].shape[:2]
    pp.run(_dev(_nchw(g["heat"])), _dev(_nchw(g["paf"])), frontend="reference")
    num, parts, _ = pp.human_tables()
    got = coco.coco_results([int(fx[scene + "_image_id"])], num, parts, (8 * h, 8 * w), tuple(fx[scene + "_upsample_keypoints"]))
    want = fx[scene + "_keypoints"]
    assert len(got) == len(want)
    for a, b in zip(got, want):
        assert np.array_equal(np.asarray(a["keypoints"], np.float64).view(np.uint64), b.view(np.uint64))
        assert a["score"] == 1.0 and a["category_id"] == 1


def test_repeated_batches_replay_as_cuda_graphs(ek):
    """A batch with the same pointers, shape and flags as an earlier one is one graph launch; results equal the eager
    first submission bit for bit, on the device entry and on the host entry (one pinned block, one copy)."""
    from torch_ekpose_b200 import synthetic
    heat, paf = synthetic.make_batch(8, 46, 54, (2, 5), seed=77)
    p = ek.PostProcessor(device=0, max_batch=8, max_h=46, max_w=54, max_peaks=1024, max_humans=32)
    hd, pd = _dev(heat), _dev(paf)
    outs = []
    for rep in range(3):
        for frontend, mat in (("dense", True), ("dense", False), ("reference", False)):
            p.run(hd, pd, frontend=frontend, materialize=mat)
            outs.append((rep, frontend, mat, p.results(with_peaks=True)))
    assert p.graph_launches() >= 6   # the second and third round at least (the first captures)
    pb = ek.PinnedBatch(8, 46, 54)
    np.copyto(pb.heat, heat); np.copyto(pb.paf, paf)
    for rep in range(3):
        p.run(pb.heat, pb.paf, frontend="dense", materialize=True)
        outs.append((rep, "dense", True, p.results(with_peaks=True)))
    first = {}
    for rep, frontend, mat, res in outs:
        ref = first.setdefault((frontend, mat), res)
        for key in ("num_humans", "n_peaks", "overflow"):
            assert np.array_equal(ref[key], res[key])
        assert_bits_equal(ref["subset"], res["subset"], f"{frontend} {mat} rep {rep}")
        assert np.array_equal(ref["peaks"], res["peaks"])
    _check_batch(p, heat, paf, "dense", True, range(8))
    pb.close()
    p.close()


def test_graph_replay_reads_the_buffers_current_content(ek):
    """A replayed batch must see what the caller's buffers hold NOW: the same pageable NumPy arrays, the same pinned
    block and the same device tensors are refilled between submissions (a stream of frames through fixed buffers)."""
    from torch_ekpose_b200 import synthetic
    scenes = [synthetic.make_batch(4, 46, 54, (p, p + 2), seed=300 + p) for p in (1, 3, 5)]
    p = ek.PostProcessor(device=0, max_batch=4, max_h=46, max_w=54, max_peaks=1024, max_humans=32)
    host_h, host_p = np.empty_like(scenes[0][0]), np.empty_like(scenes[0][1])          # pageable host memory
    pb = ek.PinnedBatch(4, 46, 54)
    dev_h, dev_p = torch.empty(host_h.shape, device="cuda"), torch.empty(host_p.shape, device="cuda")
    for rounds in range(2):
        for heat, paf in scenes:
            want = None
            for kind in ("pageable", "pinned", "device"):
                if kind == "pageable":
                    host_h[...] = heat; host_p[...] = paf
                    p.run(host_h, host_p, frontend="reference")
                elif kind == "pinned":
                    np.copyto(pb.heat, heat); np.copyto(pb.paf, paf)
                    p.run(pb.heat, pb.paf, frontend="reference")
                else:
                    dev_h.copy_(torch.from_numpy(heat)); dev_p.copy_(torch.from_numpy(paf))
                    p.run(dev_h, dev_p, frontend="reference")
                res = p.results()
                if want is None:
                    want = res
                    for i in range(4):
                        hw, pw = np.ascontiguousarray(heat[i].transpose(1, 2, 0)), np.ascontiguousarray(paf[i].transpose(1, 2, 0))
                        _, sub = util.oracle_reference(hw, pw)
                        n = int(res["num_humans"][i])
                        assert n == len(sub)
                        assert_bits_equal(res["subset"][i, :n], sub, f"{kind} image {i}")
                else:
                    assert np.array_equal(want["num_humans"], res["num_humans"])
                    assert_bits_equal(want["subset"], res["subset"], kind)
    assert p.graph_launches() >= 6
    pb.close()
    p.close()


def test_context_capacities_and_growth(ek):
    """max_part / max_cand are per-context capacities (ekp_create_ex): a crowd overflows a small context (reported,
    never silent) and fits a big one; postprocess_batch grows the capacities that overflowed and retries, within the
    library's limits."""
    from torch_ekpose_b200 import _lib, synthetic
    heat, paf = synthetic.make_batch(1, 92, 164, (35, 35), seed=9)
    small = ek.PostProcessor(device=0, max_batch=1, max_h=92, max_w=164, max_peaks=2048, max_humans=128, max_part=16, max_cand=64)
    assert (small.max_part, small.max_cand) == (16, 64)
    small.run(_dev(heat), _dev(paf), frontend="reference")
    res = small.results(raise_on_overflow=False)
    assert int(res["overflow"][0]) & _lib.OVF_PART
    with pytest.raises(_lib.EkpCapacityError):
        small.results()
    small.close()
    big = ek.PostProcessor(device=0, max_batch=1, max_h=92, max_w=164, max_peaks=2048, max_humans=128, max_part=512, max_cand=4096)
    _check_batch(big, heat, paf, "reference", False, [0])
    big.close()
    for bad in (dict(max_part=2048), dict(max_cand=16), dict(max_humans=2048), dict(max_peaks=100000), dict(max_batch=70000)):
        kw = dict(device=0, max_batch=1, max_h=8, max_w=8, max_peaks=64, max_humans=8)
        kw.update(bad)
        with pytest.raises(_lib.EkpError):
            ek.PostProcessor(**kw)
    # the convenience API starts small and grows what overflowed
    from torch_ekpose_b200 import paf_to_pose
    paf_to_pose._cache.clear()
    humans = ek.postprocess_batch(heat, paf, frontend="reference", max_peaks=256, max_humans=8, max_part=8, max_cand=64)
    hw, pw = np.ascontiguousarray(heat[0].transpose(1, 2, 0)), np.ascontiguousarray(paf[0].transpose(1, 2, 0))
    _, sub = util.oracle_reference(hw, pw)
    assert len(humans[0]) == len(sub) >= 30
    paf_to_pose._cache.clear()


def test_random_shapes_layouts_thresholds_vs_oracle(ek):
    """Fuzz: random map sizes (incl. odd / tiny / wide), layouts, thresholds, random fields instead of
    person-like scenes; both front-ends; peaks and people must equal the oracle bit for bit."""
    rng = np.random.default_rng(2024)
    pp = ek.PostProcessor(device=0, max_batch=3, max_h=48, max_w=80, max_peaks=8192, max_humans=512)
    fe = util.frontend()
    for trial in range(12):
        h, w = int(rng.integers(5, 48)), int(rng.integers(5, 80))
        n = int(rng.integers(1, 4))
        layout = "nchw" if trial % 2 else "nhwc"
        thr = float(rng.choice([0.22, 0.3, 0.6]))
        # a random background below every threshold plus a few sharp spikes (so that peaks stay sparse)
        heat = rng.random((n, h, w, 19)).astype(np.float32) * 0.2
        for _ in range(int(rng.integers(0, 60))):
            heat[rng.integers(0, n), rng.integers(0, h), rng.integers(0, w), rng.integers(0, 18)] = rng.random() * 0.9 + 0.2
        paf = rng.normal(0, 0.5, (n, h, w, 38)).astype(np.float32)
        hin = heat if layout == "nhwc" else np.ascontiguousarray(heat.transpose(0, 3, 1, 2))
        pin = paf if layout == "nhwc" else np.ascontiguousarray(paf.transpose(0, 3, 1, 2))
        for frontend in ("dense", "reference"):
            pp.run(_dev(hin), _dev(pin), layout=layout, frontend=frontend, thr=thr, materialize=bool(trial % 3 == 0))
            res = pp.results(with_peaks=True)
            assert not res["overflow"].any(), (trial, frontend)
            for i in range(n):
                if frontend == "dense":
                    peaks = fe.dense_nms(fe.dense_smooth(heat[i]), np.float32(thr))
                    paf_mat = fe.upsample_bilinear(paf[i])
                else:
                    peaks = fe.ref_nms(heat[i], np.float32(thr))
                    paf_mat = fe.upsample_nearest(paf[i])
                assert_bits_equal(util.peaks_table(res, i), peaks, f"trial {trial} {frontend} {h}x{w} {layout} image {i} peaks")
                sub, _ = util.oracle_people(peaks, 8 * h, 8 * w, paf_mat)
                m = int(res["num_humans"][i])
                assert m == len(sub), (trial, frontend, i, m, len(sub))
                assert_bits_equal(res["subset"][i, :m], sub, f"trial {trial} {frontend} image {i} subset")
    pp.close()


@pytest.mark.parametrize("mode", ["vgg", "rtpose"])
@pytest.mark.parametrize("shape", [(480, 640), (300, 500), (101, 77), (720, 1280)])
def test_input_side_kernel_vs_oracle(pp, shape, mode):
    """Row f4: padding + normalisation kernel == the oracle (== cv2 + the reference's Python) bit for bit."""
    rng = np.random.default_rng(shape[0])
    frames = rng.integers(0, 256, (3,) + shape + (3,), dtype=np.uint8)
    out, scale = pp.preprocess(torch.from_numpy(frames).cuda(), mode=mode)
    fe = util.frontend()
    assert scale == fe.preprocess_dims(*shape)[4]
    got = out.cpu().numpy()
    for i in range(3):
        assert_bits_equal(got[i], fe.preprocess(frames[i], mode), f"frame {i}")


def test_device_std_sort_replay_equals_libstdcxx(ek, pp):
    """The device replay of libstdc++'s std::sort (used when >16 candidates tie) against the oracle's
    restatement, itself pinned to the compiled reference's std::sort -- incl. median-of-3 killer
    inputs that reach the heapsort fallback, which real scenes never do."""
    port = util.port()
    rng = np.random.default_rng(0)

    def killer(n):
        k = n // 2
        a = np.zeros(n)
        for i in range(k):
            a[i] = i + 1 if i % 2 == 0 else k + i + 1
            a[k + i] = 2 * (i + 1)
        return (-a).astype(np.float32)

    before = port.heapsort_hits()
    for n in [0, 1, 2, 15, 16, 17, 18, 33, 64, 100, 257, 1000, 2048]:
        for v in (rng.random(n), rng.integers(0, 3, n), np.zeros(n), np.sort(rng.integers(0, 9, n)), killer(n) if n > 1 else np.zeros(n)):
            v = np.asarray(v, np.float32)
            s = torch.from_numpy(v.copy()).cuda()
            t = torch.arange(n, dtype=torch.int32).cuda()
            ek._lib.check(ek._lib.lib.ekp_debug_std_sort(pp._ctx, s.data_ptr(), t.data_ptr(), n, 0))
            torch.cuda.synchronize()
            want_s, want_t = port.sort_scores(v)
            assert np.array_equal(t.cpu().numpy(), want_t) and np.array_equal(s.cpu().numpy(), want_s), n
    assert port.heapsort_hits() > before
    ref = util.ref_or_none()
    if ref is not None:   # and the oracle's restatement against the real std::sort on the same inputs
        for n in (17, 100, 2048):
            v = killer(n)
            assert np.array_equal(port.sort_scores(v)[1], ref.sort_scores(v)[1])


def test_host_entry_equals_device_entry(ek):
    """ekp_postprocess_host (pinned / pageable host buffers, the e2e path of bench.py) must give exactly
    what ekp_postprocess gives on device tensors, with and without materialisation."""
    from torch_ekpose_b200 import synthetic
    heat, paf = synthetic.make_batch(8, 46, 54, (1, 6), seed=31)
    a = ek.PostProcessor(device=0, max_batch=8, max_h=46, max_w=54, max_peaks=512, max_humans=32)
    b = ek.PostProcessor(device=0, max_batch=8, max_h=46, max_w=54, max_peaks=512, max_humans=32)
    for frontend in ("dense", "reference"):
        for mat in (True, False):
            a.run(_dev(heat), _dev(paf), frontend=frontend, materialize=mat)
            b.run(torch.from_numpy(heat).pin_memory(), torch.from_numpy(paf).pin_memory(), frontend=frontend, materialize=mat)
            ra, rb = a.results(with_peaks=True), b.results(with_peaks=True)
            for k in ("num_humans", "n_peaks", "overflow", "part_off"):
                assert np.array_equal(ra[k], rb[k]), (frontend, mat, k)
            assert np.array_equal(ra["subset"].view(np.uint32), rb["subset"].view(np.uint32))
            assert np.array_equal(ra["peaks"], rb["peaks"])
            ha, hb = a.human_tables(), b.human_tables()
            assert all(np.array_equal(x, y) for x, y in zip(ha, hb))
    a.close(); b.close()


def _nccl_worker(rank, world, port, out_dir):
    import os
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from torch_ekpose_b200 import synthetic
    from torch_ekpose_b200.sharding import postprocess_sharded
    heat, paf = synthetic.make_batch(9, 46, 54, (1, 4), seed=41)
    num, sub = postprocess_sharded(heat, paf, frontend="dense", max_humans=32, max_peaks=512)
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), num=num, sub=sub)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_two_gpus_nccl(ek, tmp_path):
    """One process per GPU, images sharded, final gather over NCCL == single-GPU result."""
    import socket
    import torch.multiprocessing as mp
    from torch_ekpose_b200 import synthetic
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_nccl_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    heat, paf = synthetic.make_batch(9, 46, 54, (1, 4), seed=41)
    one = ek.PostProcessor(device=0, max_batch=9, max_h=46, max_w=54, max_peaks=512, max_humans=32)
    one.run(_dev(heat), _dev(paf), frontend="dense")
    want = one.results()
    one.close()
    for r in range(2):
        z = np.load(tmp_path / f"rank{r}.npz")
        assert np.array_equal(z["num"], want["num_humans"])
        assert np.array_equal(z["sub"].view(np.uint32), want["subset"].view(np.uint32))
