"""ekp_draw_humans / PostProcessor.draw_humans / estimator.infer_and_draw: the people of a run painted onto device
frames must be byte for byte what the reference's draw_humans (lib/utils/common.py:252-275) paints with cv2.

The CPU tests pin the rasteriser itself (the same __host__ __device__ code, through the library's host test hooks) to
cv2: the part marker stamp, thick lines, whole human tables.  The GPU tests compare every drawn frame with the checker
applied to pp.humans() of the same run, on a copy of the same random-content frame."""
import os

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")
torch = pytest.importorskip("torch")

import oracle  # noqa: E402
from tests import draw_check  # noqa: E402
from torch_ekpose_b200 import _lib  # noqa: E402
from torch_ekpose_b200.common import CocoPairsRender  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _raster(kind, x0, y0, x1, y1, H, W):
    m = np.zeros((H, W), np.uint8)
    _lib.check(_lib.lib.ekp_debug_raster_host(kind, x0, y0, x1, y1, H, W, m.ctypes.data))
    return m


def _cv2_line(p0, p1, H, W):
    m = np.zeros((H, W), np.uint8)
    cv2.line(m, p0, p1, 1, 3)
    return m


def _draw_host(num, parts, map_h, map_w, frames):
    out = np.array(frames, copy=True)
    num = np.ascontiguousarray(num, np.int32)
    parts = np.ascontiguousarray(parts)
    n, H, W, _ = out.shape
    _lib.check(_lib.lib.ekp_debug_draw_host(num.ctypes.data, parts.ctypes.data, parts.shape[1], map_h, map_w,
                                            out.ctypes.data, n, H, W))
    return out


def _random_tables(rng, n, max_humans, map_h, map_w, present=0.8):
    num = rng.integers(0, max_humans + 1, n).astype(np.int32)
    parts = np.zeros((n, max_humans, 18), draw_check.PEAK_DT)
    parts["x"] = rng.integers(0, map_w, parts.shape)
    parts["y"] = rng.integers(0, map_h, parts.shape)
    parts["score"] = rng.random(parts.shape)
    parts["id"] = np.where(rng.random(parts.shape) < present, rng.integers(0, 1000, parts.shape), -1)
    return num, parts


# ---- CPU: the rasteriser against cv2 ---------------------------------------------------------------------------------
def test_render_tables_are_the_reference_tables():
    assert len(CocoPairsRender) == 17
    try:
        ref = oracle.reference_module("lib.utils.common")
    except FileNotFoundError:
        ref = None
    if ref is not None:
        assert [list(c) for c in ref.CocoColors] == draw_check.CocoColors
        assert [tuple(p) for p in ref.CocoPairsRender] == list(CocoPairsRender)
    assert ref is not None or not os.path.isdir(oracle.REF_ROOT)


@pytest.mark.parametrize("H,W", [(1, 1), (1, 2), (2, 1), (2, 2), (3, 7), (11, 11), (24, 31)])
def test_part_marker_stamp_equals_cv2_circle(H, W):
    """cv2.circle(c, 3, thickness=3, lineType=8) for EVERY centre in [-1, W] x [-1, H] (draw_humans' range plus one)."""
    for y in range(-1, H + 1):
        for x in range(-1, W + 1):
            want = np.zeros((H, W), np.uint8)
            cv2.circle(want, (x, y), 3, 1, thickness=3, lineType=8, shift=0)
            assert np.array_equal(_raster(1, x, y, 0, 0, H, W), want), (H, W, x, y)


def test_part_marker_is_a_96_pixel_ring():
    m = _raster(1, 10, 10, 0, 0, 21, 21)
    assert m.sum() == 96 and m[10, 10] == 0 and m[5:16, 5:16].sum() == 96


def _line_cases(rng):
    sizes = [(1, 1), (1, 2), (2, 1), (3, 3), (5, 9), (17, 12), (30, 40), (48, 64), (61, 83)]
    for k in range(100_000):
        H, W = sizes[k % len(sizes)]
        x0, x1 = (int(v) for v in rng.integers(0, W + 1, 2))
        y0, y1 = (int(v) for v in rng.integers(0, H + 1, 2))
        kind = k % 10
        if kind == 0:            # zero length: only the caps
            x1, y1 = x0, y0
        elif kind == 1:          # along a border
            side = (k // 10) % 4
            if side == 0:
                x0 = x1 = 0
            elif side == 1:
                x0 = x1 = W
            elif side == 2:
                y0 = y1 = 0
            else:
                y0 = y1 = H
        elif kind == 2:          # through / from the corners
            corners = [(0, 0), (W, 0), (0, H), (W, H)]
            (x0, y0), (x1, y1) = corners[(k // 10) % 4], corners[(k // 40) % 4]
        elif kind == 3:          # one endpoint on a corner
            x0, y0 = [(0, 0), (W, 0), (0, H), (W, H)][(k // 10) % 4]
        yield (x0, y0), (x1, y1), H, W


def test_thick_lines_equal_cv2_line():
    """10^5 seeded cv2.line(..., 3) with endpoints in draw_humans' range [0, W] x [0, H]: zero-length lines, lines along
    each border, lines through the frame's corners and random ones, on frames from 1x1 to 61x83."""
    rng = np.random.default_rng(2026)
    bad = []
    for p0, p1, H, W in _line_cases(rng):
        if not np.array_equal(_raster(2, *p0, *p1, H, W), _cv2_line(p0, p1, H, W)):
            bad.append((p0, p1, H, W))
    assert not bad, f"{len(bad)} lines differ from cv2, first {bad[:5]}"


@pytest.mark.parametrize("H,W", [(480, 640), (736, 1312), (77, 100)])
def test_long_thick_lines_equal_cv2_line(H, W):
    rng = np.random.default_rng(H * W)
    for k in range(1500):
        p0 = (int(rng.integers(0, W + 1)), int(rng.integers(0, H + 1)))
        p1 = (int(rng.integers(0, W + 1)), int(rng.integers(0, H + 1)))
        if k % 5 == 1:
            p0, p1 = (0, p0[1]), (W, p1[1])
        elif k % 5 == 2:
            p0, p1 = (p0[0], 0), (p1[0], H)
        assert np.array_equal(_raster(2, *p0, *p1, H, W), _cv2_line(p0, p1, H, W)), (p0, p1)


@pytest.mark.parametrize("H,W,map_hw", [(368, 432, (368, 432)), (77, 100, (368, 432)), (480, 640, (368, 432)),
                                        (2, 1, (64, 48)), (736, 1312, (736, 1312))])
def test_whole_tables_equal_restated_draw_humans(H, W, map_hw):
    """Random human tables (overlapping people, absent parts, empty rows) on random frames: the host hook draws what
    the restated draw_humans draws, and what the reference's own one draws where it can be imported."""
    rng = np.random.default_rng(H + W)
    map_h, map_w = map_hw
    n = 3
    num, parts = _random_tables(rng, n, 12, map_h, map_w)
    num[0] = 0
    parts["id"][1, 0] = -1                    # a row with no parts draws nothing
    frames = rng.integers(0, 256, (n, H, W, 3), dtype=np.uint8)
    humans = draw_check.humans_of(num, parts, map_h, map_w)
    want = draw_check.draw_batch(frames, humans)
    assert np.array_equal(_draw_host(num, parts, map_h, map_w, frames), want)
    try:
        ref = oracle.reference_module("lib.utils.common")
    except FileNotFoundError:
        return
    assert np.array_equal(draw_check.draw_batch(frames, humans, ref.draw_humans), want)


def test_host_hooks_reject_bad_arguments():
    m = np.zeros((4, 4), np.uint8)
    assert _lib.lib.ekp_debug_raster_host(3, 0, 0, 0, 0, 4, 4, m.ctypes.data) == _lib.ERR_ARG
    assert _lib.lib.ekp_debug_raster_host(1, 0, 0, 0, 0, 0, 4, m.ctypes.data) == _lib.ERR_ARG
    assert _lib.lib.ekp_debug_raster_host(1, 0, 0, 0, 0, 4, 4, None) == _lib.ERR_ARG
    num = np.zeros(1, np.int32)
    parts = np.zeros((1, 1, 18), draw_check.PEAK_DT)
    fr = np.zeros((1, 4, 4, 3), np.uint8)
    assert _lib.lib.ekp_debug_draw_host(num.ctypes.data, parts.ctypes.data, 1, 0, 8, fr.ctypes.data, 1, 4, 4) == _lib.ERR_ARG
    assert _lib.lib.ekp_debug_draw_host(num.ctypes.data, parts.ctypes.data, 1, 8, 8, fr.ctypes.data, 1, 4, 16385) == _lib.ERR_ARG


def test_package_does_not_import_cv2():
    pkg = os.path.join(ROOT, "torch_ekpose_b200")
    for name in os.listdir(pkg):
        if name.endswith(".py"):
            with open(os.path.join(pkg, name)) as f:
                assert "import cv2" not in f.read(), name


# ---- GPU: the device draw against the checker ------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ek():
    import torch_ekpose_b200 as ek
    return ek


def _frames(rng, n, H, W):
    return rng.integers(0, 256, (n, H, W, 3), dtype=np.uint8)


def _check_draw(pp, host_frames, stream=None):
    """Draws pp's last run onto a device copy of host_frames and compares with the checker on pp.humans()."""
    t = torch
    dev = t.from_numpy(host_frames).cuda(pp.device)
    out = pp.draw_humans(dev, stream=stream)
    assert out is dev
    got = dev.cpu().numpy()
    want = draw_check.draw_batch(host_frames, pp.humans())
    if not np.array_equal(got, want):
        idx = np.argwhere(got != want)
        raise AssertionError(f"{len(idx)} bytes differ, first at {idx[:5].tolist()}")
    return got


def _batch(n, h, w, people, seed):
    from torch_ekpose_b200 import synthetic
    heat, paf = synthetic.make_batch(n, h, w, people, seed=seed)
    t = torch
    return t.from_numpy(heat).cuda(), t.from_numpy(paf).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("frontend", ["dense", "reference"])
@pytest.mark.parametrize("H,W", [(368, 432), (480, 640), (77, 100)])
def test_scenes(ek, frontend, H, W):
    pp = ek.PostProcessor(device=0, max_batch=16, max_h=46, max_w=54, max_peaks=1024, max_humans=64)
    heat, paf = _batch(16, 46, 54, (1, 6), 5)
    pp.run(heat, paf, frontend=frontend)
    rng = np.random.default_rng(H)
    _check_draw(pp, _frames(rng, 16, H, W))
    assert sum(len(h) for h in pp.humans()) > 16
    pp.close()


@pytest.mark.gpu
def test_crowded_scenes(ek):
    """16 crowded 92x164 scenes (30-40 people) onto 736x1312 frames: heavy overlap tests the drawing order."""
    pp = ek.PostProcessor(device=0, max_batch=16, max_h=92, max_w=164, max_peaks=4096, max_humans=128, max_part=512,
                          max_cand=4096)
    heat, paf = _batch(16, 92, 164, (30, 40), 9)
    pp.run(heat, paf, frontend="reference")
    assert not pp.results()["overflow"].any()
    _check_draw(pp, _frames(np.random.default_rng(3), 16, 736, 1312))
    assert min(len(h) for h in pp.humans()) >= 20
    pp.close()


def _edge_person(map_h, map_w):
    """One person stretched over the whole map: wrists on the left and right edges, eyes on the top, ankles on the
    bottom row; a constant PAF along every limb, so all of it connects."""
    from torch_ekpose_b200.synthetic import COCOPAIRS, COCOPAIRS_NET, _TPL
    t = _TPL.copy()
    t[:, 0] = (t[:, 0] - t[:, 0].min()) / (t[:, 0].max() - t[:, 0].min()) * (map_w - 1)
    t[:, 1] = (t[:, 1] - t[:, 1].min()) / (t[:, 1].max() - t[:, 1].min()) * (map_h - 1)
    pts = np.rint(t).astype(np.int64)
    peaks = np.zeros((18, 5), np.float32)
    peaks[:, 0], peaks[:, 1], peaks[:, 2], peaks[:, 4] = pts[:, 0], pts[:, 1], 1.0, np.arange(18)
    peaks[:, 3] = np.arange(18)
    paf = np.zeros((map_h, map_w, 38), np.float32)
    for (a, b), (cx, cy) in zip(COCOPAIRS, COCOPAIRS_NET):
        v = (pts[b] - pts[a]).astype(np.float64)
        v /= np.hypot(*v)
        paf[:, :, cx], paf[:, :, cy] = v[0], v[1]
    return peaks, paf


@pytest.mark.gpu
def test_people_touching_the_frame_edges(ek):
    """Hand-placed peaks through ekp_process_paf_dev: centres at x = W and y = H occur (the marker and the limbs there
    are clipped as cv2 clips them), on small, odd and 1-2 px frames."""
    t = torch
    map_h, map_w = 368, 432
    peaks, paf = _edge_person(map_h, map_w)
    n = 2
    pk = t.from_numpy(np.stack([peaks] * n)).cuda()
    npk = t.full((n,), 18, dtype=t.int32, device="cuda")
    pm = t.from_numpy(np.stack([paf] * n)).cuda()
    pp = ek.PostProcessor(device=0, max_batch=n, max_h=46, max_w=54, max_peaks=64, max_humans=8)
    pp.run_peaks(pk, npk, pm, h1=map_h)
    humans = pp.humans()
    assert all(len(h) == 1 and len(h[0].body_parts) == 18 for h in humans)
    rng = np.random.default_rng(0)
    at_edge = set()
    for H, W in [(77, 100), (368, 432), (41, 33), (5, 3), (2, 2), (1, 1), (2, 1)]:
        _check_draw(pp, _frames(rng, n, H, W))
        for bp in humans[0][0].body_parts.values():
            cx, cy = int(bp.x * W + 0.5), int(bp.y * H + 0.5)
            at_edge |= {"x=W"} if cx == W else set()
            at_edge |= {"y=H"} if cy == H else set()
            at_edge |= {"x=0"} if cx == 0 else set()
            at_edge |= {"y=0"} if cy == 0 else set()
    assert at_edge == {"x=W", "y=H", "x=0", "y=0"}
    pp.close()


@pytest.mark.gpu
def test_consecutive_draws_onto_one_reused_buffer(ek):
    """Different people and frame sizes, one frames allocation reused: no key of an earlier draw leaks into a later one."""
    t = torch
    pp = ek.PostProcessor(device=0, max_batch=8, max_h=46, max_w=82, max_peaks=1024, max_humans=64)
    buf = t.empty(8 * 480 * 640 * 3, dtype=t.uint8, device="cuda")
    rng = np.random.default_rng(11)
    cases = [(8, 46, 54, 480, 640), (5, 46, 82, 368, 656), (8, 46, 54, 480, 640), (3, 46, 54, 200, 300),
             (8, 46, 82, 100, 77), (8, 46, 54, 480, 640)]
    for k, (n, h, w, H, W) in enumerate(cases):
        heat, paf = _batch(n, h, w, (1, 6), 100 + k)
        pp.run(heat, paf, frontend="dense" if k % 2 else "reference")
        host = _frames(rng, n, H, W)
        frames = buf[:n * H * W * 3].view(n, H, W, 3)
        frames.copy_(t.from_numpy(host))
        pp.draw_humans(frames)
        want = draw_check.draw_batch(host, pp.humans())
        assert np.array_equal(frames.cpu().numpy(), want), k
        pp.draw_humans(frames)          # drawing the same people again changes nothing
        assert np.array_equal(frames.cpu().numpy(), want), k
    pp.close()


@pytest.mark.gpu
def test_key_epoch_wraparound(ek):
    """The keys are cleared when the draw counter wraps (65535 draws): draws on both sides of it stay exact."""
    t = torch
    pp = ek.PostProcessor(device=0, max_batch=2, max_h=46, max_w=54, max_peaks=512, max_humans=32)
    heat, paf = _batch(2, 46, 54, (3, 5), 4)
    pp.run(heat, paf)
    host = _frames(np.random.default_rng(5), 2, 24, 32)
    dev = t.from_numpy(host).cuda()
    want = draw_check.draw_batch(host, pp.humans())
    st = t.cuda.current_stream().cuda_stream
    for _ in range(65540):
        assert _lib.lib.ekp_draw_humans(pp._ctx, dev.data_ptr(), 2, 24, 32, st) == 0
    assert np.array_equal(dev.cpu().numpy(), want)
    dev.copy_(t.from_numpy(host))
    pp.draw_humans(dev)
    assert np.array_equal(dev.cpu().numpy(), want)
    pp.close()


@pytest.mark.gpu
def test_draw_on_another_stream_then_an_immediate_run(ek):
    """Run on s1, draw on s2, then at once the next run on s1: the draw still paints the first run's people, and the
    second run's results are its own."""
    t = torch
    kw = dict(device=0, max_batch=16, max_h=46, max_w=54, max_peaks=1024, max_humans=64)
    pp, ref = ek.PostProcessor(**kw), ek.PostProcessor(**kw)
    b1, b2 = _batch(16, 46, 54, (1, 6), 31), _batch(16, 46, 54, (4, 6), 32)
    ref.run(*b1)
    want_humans = ref.humans()
    ref.run(*b2)
    want_tables2 = ref.human_tables()
    host = _frames(np.random.default_rng(7), 16, 480, 640)
    want = draw_check.draw_batch(host, want_humans)
    s1, s2 = t.cuda.Stream(), t.cuda.Stream()
    dev = t.from_numpy(host).cuda()
    t.cuda.synchronize()
    with t.cuda.stream(s1):
        pp.run(*b1, stream=s1)
    pp.draw_humans(dev, stream=s2)
    pp.run(*b2, stream=s1)
    t.cuda.synchronize()
    assert np.array_equal(dev.cpu().numpy(), want)
    got_tables2 = pp.human_tables()
    for a, b in zip(got_tables2, want_tables2):
        assert np.array_equal(a, b)
    pp.close()
    ref.close()


@pytest.mark.gpu
def test_draw_has_no_side_effects_on_results_graphs_or_counts(ek):
    pp = ek.PostProcessor(device=0, max_batch=8, max_h=46, max_w=54, max_peaks=1024, max_humans=64)
    heat, paf = _batch(8, 46, 54, (1, 6), 41)
    pp.run(heat, paf)
    pp.run(heat, paf)                                 # second submission of the same batch: a graph replay
    res0, tab0 = pp.results(with_peaks=True), pp.human_tables()
    launches, graphs = pp.kernel_launches(), pp.graph_launches()
    _check_draw(pp, _frames(np.random.default_rng(1), 8, 240, 320))
    assert pp.kernel_launches() == launches + 2       # cover + paint
    res1, tab1 = pp.results(with_peaks=True), pp.human_tables()
    for k in res0:
        assert np.array_equal(res0[k], res1[k]), k
    for a, b in zip(tab0, tab1):
        assert np.array_equal(a, b)
    pp.run(heat, paf)
    assert pp.graph_launches() == graphs + 1          # later batches still replay their graph
    _check_draw(pp, _frames(np.random.default_rng(2), 8, 240, 320))
    pp.close()


@pytest.mark.gpu
def test_errors(ek):
    t = torch
    pp = ek.PostProcessor(device=0, max_batch=4, max_h=46, max_w=54, max_peaks=512, max_humans=32)
    frames = t.zeros((4, 32, 32, 3), dtype=t.uint8, device="cuda")
    with pytest.raises(_lib.EkpError) as e:              # no run yet
        pp.draw_humans(frames)
    assert e.value.code == _lib.ERR_STATE
    L = _lib.lib
    assert L.ekp_draw_humans(pp._ctx, frames.data_ptr(), 4, 32, 32, None) == _lib.ERR_STATE
    heat, paf = _batch(4, 46, 54, (1, 3), 1)
    pp.run(heat, paf)
    ptr = frames.data_ptr()
    assert L.ekp_draw_humans(None, ptr, 4, 32, 32, None) == _lib.ERR_ARG
    assert L.ekp_draw_humans(pp._ctx, None, 4, 32, 32, None) == _lib.ERR_ARG
    assert L.ekp_draw_humans(pp._ctx, ptr, 3, 32, 32, None) == _lib.ERR_ARG
    assert L.ekp_draw_humans(pp._ctx, ptr, 5, 32, 32, None) == _lib.ERR_ARG
    assert L.ekp_draw_humans(pp._ctx, ptr, 4, 0, 32, None) == _lib.ERR_ARG
    assert L.ekp_draw_humans(pp._ctx, ptr, 4, 32, 0, None) == _lib.ERR_ARG
    assert L.ekp_draw_humans(pp._ctx, ptr, 4, _lib.DRAW_MAX_SIDE + 1, 1, None) == _lib.ERR_ARG
    assert L.ekp_draw_humans(pp._ctx, ptr, 4, 1, _lib.DRAW_MAX_SIDE + 1, None) == _lib.ERR_ARG
    for bad in (frames.cpu(), frames.float(), frames[:, :, :16], frames.permute(0, 2, 1, 3), frames[:3],
                frames[..., :2].contiguous(), frames[0], np.zeros((4, 32, 32, 3), np.uint8)):
        with pytest.raises(ValueError):
            pp.draw_humans(bad)
    with pytest.raises(ValueError):
        pp.draw_humans(t.zeros((4, 1, _lib.DRAW_MAX_SIDE + 1, 3), dtype=t.uint8, device="cuda"))
    _check_draw(pp, np.zeros((4, 32, 32, 3), np.uint8))   # the failed calls left the context usable
    pp.close()


@pytest.mark.gpu
def test_infer_and_draw_equals_infer_humans_plus_the_checker(ek):
    t = torch
    from torch_ekpose_b200 import estimator
    heat, paf = _batch(3, 46, 54, (2, 5), 21)

    class FakeNet(t.nn.Module):
        def forward(self, x):
            return (paf, heat), None

    rng = np.random.default_rng(8)
    host = _frames(rng, 3, 368, 432)
    want = draw_check.draw_batch(host, estimator.infer_humans(list(host), FakeNet(), "vgg", t.device("cuda", 0)))
    got = estimator.infer_and_draw(list(host), FakeNet(), "vgg", t.device("cuda", 0))
    assert got.is_cuda and got.dtype == t.uint8 and tuple(got.shape) == host.shape
    assert np.array_equal(got.cpu().numpy(), want)
    assert sum(len(h) for h in estimator.last_postprocessor().humans()) > 0
    dev = t.from_numpy(host).cuda()                       # a CUDA tensor is drawn in place
    assert estimator.infer_and_draw(dev, FakeNet(), "vgg", t.device("cuda", 0)) is dev
    assert np.array_equal(dev.cpu().numpy(), want)
    got = estimator.infer_and_draw(t.from_numpy(host), FakeNet(), "vgg", t.device("cuda", 0))   # a CPU tensor: its copy
    assert np.array_equal(got.cpu().numpy(), want)
