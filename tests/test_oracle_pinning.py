"""CPU: pin the oracle against the real code it restates: libstdc++'s std::sort, OpenCV and SciPy (the libraries the
reference's Python side calls, paf_to_pose.py:1-6).  Its comparisons with the reference itself are the golden fixtures
(tests/test_oracle_golden.py)."""
import os

import numpy as np
import pytest

import oracle
from tests import util
from tests.util import assert_bits_equal
from torch_ekpose_b200 import synthetic

# std::sort exactly as pafprocess.cpp:97 calls it: the element type of pafprocess.h:38-43 and the comparator of
# pafprocess.cpp:244-246, compiled against the host's libstdc++ (the ordering the reference's results inherit)
_STD_SORT_CPP = r"""
#include <algorithm>
#include <vector>
struct ConnectionCandidate { int idx1; int idx2; float score; float etc; };
static bool comp_candidate(ConnectionCandidate a, ConnectionCandidate b) { return a.score > b.score; }
extern "C" void std_sort(int n, float *score, int *tag) {
    std::vector<ConnectionCandidate> v(n);
    for (int i = 0; i < n; i++) { v[i].idx1 = tag[i]; v[i].idx2 = 0; v[i].score = score[i]; v[i].etc = 0; }
    std::sort(v.begin(), v.end(), comp_candidate);
    for (int i = 0; i < n; i++) { score[i] = v[i].score; tag[i] = v[i].idx1; }
}
"""


class _LibstdcxxSort:
    def __init__(self, tmp_dir):
        import ctypes
        import subprocess
        src, so = os.path.join(tmp_dir, "std_sort.cpp"), os.path.join(tmp_dir, "libstd_sort.so")
        with open(src, "w") as f:
            f.write(_STD_SORT_CPP)
        subprocess.run([os.environ.get("CXX", "g++"), "-O2", "-fPIC", "-shared", "-o", so, src], check=True)
        self.fn = ctypes.CDLL(so).std_sort
        self.fn.argtypes = [ctypes.c_int, np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS"),
                            np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")]
        self.fn.restype = None

    def sort_scores(self, scores):
        s = np.ascontiguousarray(scores, np.float32).copy()
        t = np.arange(len(s), dtype=np.int32)
        self.fn(len(s), s, t)
        return s, t


def test_sort_port_equals_libstdcxx_incl_heapsort_fallback(tmp_path):
    """The restated introsort (oracle/paf_oracle.c) against libstdc++'s own std::sort with the reference's comparator,
    and against the compiled reference where it was built."""
    port = util.port()
    sorts = [_LibstdcxxSort(str(tmp_path))] + ([util.ref_or_none()] if oracle.have_ref() else [])
    rng = np.random.default_rng(0)

    def killer(n):  # median-of-3 killer: drives introsort into its heapsort fallback
        k = n // 2
        a = np.zeros(n)
        for i in range(k):
            a[i] = i + 1 if i % 2 == 0 else k + i + 1
            a[k + i] = 2 * (i + 1)
        return (-a).astype(np.float32)

    before = port.heapsort_hits()
    for n in list(range(0, 40)) + [64, 100, 500, 2048]:
        for v in (rng.random(n), rng.integers(0, 3, n), np.zeros(n), np.sort(rng.integers(0, 9, n)), killer(n) if n > 1 else np.zeros(n)):
            v = np.asarray(v, np.float32)
            b = port.sort_scores(v)
            for ref in sorts:
                a = ref.sort_scores(v)
                assert np.array_equal(a[1], b[1]) and np.array_equal(a[0], b[0])
    assert port.heapsort_hits() > before   # the fallback really ran


def test_bicubic_restatement_equals_opencv_own_code():
    cv2 = pytest.importorskip("cv2")
    fe = util.frontend()
    rng = np.random.default_rng(3)
    was = cv2.ipp.useIPP()
    try:
        for _ in range(40):
            ph, pw = rng.integers(3, 6, 2)
            patch = rng.random((ph, pw)).astype(np.float32)
            mine = fe.resize_cubic(patch)
            cv2.ipp.setUseIPP(False)
            assert_bits_equal(mine, cv2.resize(patch, None, fx=8, fy=8, interpolation=cv2.INTER_CUBIC), "vs cv2 (IPP off)")
            cv2.ipp.setUseIPP(True)
            ipp = cv2.resize(patch, None, fx=8, fy=8, interpolation=cv2.INTER_CUBIC)
            assert np.abs(mine - ipp).max() <= 2.5e-7 and mine.argmax() == ipp.argmax()
    finally:
        cv2.ipp.setUseIPP(was)


def _library_dense_peaks(heat, thr=0.15):
    """Stages 1-3 with the library primitives the reference imports (paf_to_pose.py:1-6): cv2.resize(INTER_LINEAR) x8,
    scipy.ndimage.gaussian_filter(sigma=3), maximum_filter(size=3) == value & value > thr."""
    import cv2
    from scipy import ndimage as ndi
    up = cv2.resize(heat, None, fx=8, fy=8, interpolation=cv2.INTER_LINEAR)
    lib = np.stack([ndi.gaussian_filter(up[:, :, k], sigma=3) for k in range(18)], -1)
    peaks = set()
    for k in range(18):
        m = (ndi.maximum_filter(lib[:, :, k], size=3, mode="constant", cval=-np.inf) == lib[:, :, k]) & (lib[:, :, k] > np.float32(thr))
        peaks |= {(int(x), int(y), k) for y, x in zip(*np.nonzero(m))}
    return peaks, lib, up


def _oracle_dense_peaks(fe, heat, sequential=False):
    S = fe.dense_smooth(heat, sequential=sequential)
    return {(int(r[0]), int(r[1]), int(r[4])) for r in fe.dense_nms(S, cap=400000)}, S


_PIN_CASES = [("golden:" + n, None) for n in util.SCENES] + [
    ("46x54 4 people", (46, 54, 4, 21)), ("46x82 8 people (configs[2] shape)", (46, 82, 8, 31)),
    ("92x164 36 people (configs[3] shape)", (92, 164, 36, 41)), ("92x164 40 people (configs[3] shape)", (92, 164, 40, 42))]


@pytest.mark.parametrize("name,spec", _PIN_CASES, ids=[c[0] for c in _PIN_CASES])
def test_dense_definition_close_to_library_primitives(name, spec):
    """The dense front-end's arithmetic is defined by our oracle (the reference has none).  Pin of that definition: on
    every golden scene and on the real configs[2] / configs[3] shapes (30-40 people) the smoothed map is within 1e-6
    of the library composition, and BOTH forms of the oracle (5-tap polyphase = what the GPU runs; literal upsample ->
    25-tap Gaussian) produce exactly the library's peak SET: 0 disagreeing peaks."""
    pytest.importorskip("cv2")
    pytest.importorskip("scipy.ndimage")
    fe = util.frontend()
    heat = util.golden(name.split(":")[1])["heat"] if spec is None else synthetic.make_scene(*spec)[0]
    want, lib, up = _library_dense_peaks(heat)
    assert np.abs(up - fe.upsample_bilinear(heat)).max() <= 1e-6
    got, S = _oracle_dense_peaks(fe, heat)
    got_seq, S_seq = _oracle_dense_peaks(fe, heat, sequential=True)
    assert np.abs(S - lib).max() <= 1e-6 and np.abs(S_seq - lib).max() <= 1e-6 and np.abs(S - S_seq).max() <= 1e-6
    assert len(got ^ want) == 0, f"{len(got - want)} peaks only in the oracle, {len(want - got)} only in the library form"
    assert len(got_seq ^ want) == 0 and len(got ^ got_seq) == 0
    if spec is not None:
        assert len(want) >= 17 * spec[2] * 0.8   # a real scene, not an empty map


def test_dense_definition_on_exact_plateaus_is_arithmetic_defined():
    """Peaks are defined by float equality (`value == max3x3(value)`), so on EXACT plateaus -- constant regions, flat blocks:
    inputs a network never produces -- which members of a plateau count as peaks depends on the last bit of the
    smoothing arithmetic (SciPy accumulates in double, the oracle / GPU in float32 polyphase form).  What holds, and
    is checked: (1) isolated and mirror-symmetric maxima agree exactly; (2) the oracle never reports a peak the
    library form does not (oracle peaks are a subset); (3) every library-only peak is a plateau member (it ties bit for
    bit with a 3x3 neighbour in the library map), i.e. the disagreement is confined to plateaus."""
    pytest.importorskip("cv2")
    fe = util.frontend()
    pl = np.zeros((46, 54, 19), np.float32)
    pl[10:14, 10:14, 0] = 0.8                      # flat 4x4 block
    pl[20, 20, 1] = pl[20, 21, 1] = 0.9            # two equal neighbours
    pl[30:33, 30:33, 2] = 1.0                      # saturated 3x3 block
    pl[5, 5, 3] = pl[5, 9, 3] = 0.7                # mirror-symmetric pair of blobs
    pl[:, :, 4] = 0.5                              # a constant map: one plateau above the threshold
    pl[15:30, 15:40, 5] = np.float32(0.6)          # a large flat region
    pl[25, 25, 6] = 0.9                            # an ordinary isolated maximum
    want, lib, _ = _library_dense_peaks(pl)
    got, S = _oracle_dense_peaks(fe, pl)
    assert np.abs(S - lib).max() <= 1e-6
    by = lambda P, k: {q for q in P if q[2] == k}
    for k in (1, 2, 3, 6):
        assert by(got, k) == by(want, k) and len(by(want, k)) >= 1
    assert not (got - want), "an oracle peak that the library form does not have"
    only_lib = want - got
    assert only_lib and {q[2] for q in only_lib} <= {0, 4, 5}
    H, W = lib.shape[:2]
    for x, y, k in list(only_lib)[:2000]:
        v = lib[y, x, k]
        ties = [lib[j, i, k] == v for j in range(max(y - 1, 0), min(y + 2, H)) for i in range(max(x - 1, 0), min(x + 2, W)) if (j, i) != (y, x)]
        assert any(ties), f"library-only peak at {(x, y, k)} is not on a plateau"


def test_gaussian_restatement_equals_scipy_own_code():
    """NMS(bool_gaussian_filt=True): okp_scipy_gauss3 == scipy.ndimage.gaussian_filter(sigma=3) bit for bit on float32
    patches of every size a clipped window gives (3..5 cells x 8), its weights == scipy's own kernel array, and the
    product library's host-side copy of the weights (what a context uploads) == both."""
    from scipy.ndimage import gaussian_filter
    from scipy.ndimage._filters import _gaussian_kernel1d
    fe = util.frontend()
    w = _gaussian_kernel1d(3.0, 0, 12)[::-1]
    assert np.array_equal(w, w[::-1])
    assert np.array_equal(fe.scipy_gauss3_weights(), w[:13])
    import ctypes
    from torch_ekpose_b200 import _lib
    mine = np.zeros(13, np.float64)
    assert _lib.lib.ekp_scipy_gauss3_weights(mine.ctypes.data_as(ctypes.c_void_p)) == 0
    assert np.array_equal(mine, w[:13])
    rng = np.random.default_rng(5)
    for hh in (24, 32, 40):
        for ww in (24, 32, 40):
            for k in range(4):
                patch = (rng.random((hh, ww)) ** (1 + k)).astype(np.float32) * np.float32(10.0 ** (k - 2))
                assert_bits_equal(fe.scipy_gauss3(patch), gaussian_filter(patch, sigma=3), f"{hh}x{ww}")


def test_input_side_restatement_equals_cv2_and_reference_python():
    """Row f4 oracle: padding() + vgg/rtpose_preprocess restated in C == cv2 (8-bit INTER_LINEAR is OpenCV's own
    fixed-point code, no IPP for 8UC3) and == the REFERENCE'S OWN padding (lib/evaluate/estimator.py:52-68) and
    vgg_preprocess / rtpose_preprocess (lib/datasets/preprocessing.py:16-43), imported unmodified (source tree here,
    byte-compiled oracle/_ref/py on the GPU box)."""
    cv2 = pytest.importorskip("cv2")
    fe = util.frontend()
    rng = np.random.default_rng(1)
    try:
        ref_est = oracle.reference_module("lib.evaluate.estimator")
        ref_prep = oracle.reference_module("lib.datasets.preprocessing")
    except FileNotFoundError:
        ref_est = ref_prep = None
    for (h, w) in [(480, 640), (720, 1280), (300, 500), (368, 432), (101, 77), (640, 480), (50, 50), (333, 555)]:
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        rh, rw, ph, pw, scale = fe.preprocess_dims(h, w)
        assert np.array_equal(fe.resize_linear_u8(img, scale), cv2.resize(img, None, fx=scale, fy=scale))
        if ref_est is None:
            continue
        pad, s2, shp = ref_est.padding(img, 368, factor=8, is_ceil=True)
        assert s2 == scale and pad.shape == (ph, pw, 3) and tuple(shp) == (rh, rw, 3)
        assert_bits_equal(fe.preprocess(img, "vgg"), ref_prep.vgg_preprocess(pad), "vs the reference's vgg_preprocess")
        assert_bits_equal(fe.preprocess(img, "rtpose"), ref_prep.rtpose_preprocess(pad), "vs the reference's rtpose_preprocess")
    assert ref_est is not None or not os.path.isdir(oracle.REF_ROOT)
