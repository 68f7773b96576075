"""ekp_results_device / PostProcessor.result_tensors / estimator.infer_human_tensors: the last run's tables written into
device tensors, ordered after the run, with no host wait.  Copied to the host, every tensor must equal the host
readers' table (results(), human_tables()) byte for byte, padding rows included."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from torch_ekpose_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PEAK_DT = np.dtype([("x", np.int32), ("y", np.int32), ("score", np.float32), ("id", np.int32)])
FIELDS = ("num_humans", "overflow", "n_peaks", "subset", "parts", "scores")


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_struct_layout_equals_the_c_compilers(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ekpose_b200.h"\nint main(void) {\n'
                   '    printf("%lu", (unsigned long) sizeof(ekp_device_results));\n' +
                   "".join(f'    printf(" %lu", (unsigned long) offsetof(ekp_device_results, {f}));\n' for f in FIELDS) +
                   '    printf("\\n");\n    return 0;\n}\n')
    exe = str(tmp_path / "layout")
    cc = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                         str(src), "-o", exe], capture_output=True, text=True)
    assert cc.returncode == 0, cc.stderr
    got = [int(v) for v in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    want = [ctypes.sizeof(_lib.DeviceResults)] + [getattr(_lib.DeviceResults, f).offset for f in FIELDS]
    assert got == want


def test_null_context_or_out_is_an_argument_error_without_a_device():
    tabs = _lib.DeviceResults()
    assert _lib.lib.ekp_results_device(None, 1, ctypes.byref(tabs), None) == _lib.ERR_ARG
    assert _lib.lib.ekp_results_device(None, 1, None, None) == _lib.ERR_ARG
    # the NULL `out` is rejected before anything reads the context, so any non-NULL handle shows it
    stand_in = ctypes.create_string_buffer(64)
    assert _lib.lib.ekp_results_device(ctypes.addressof(stand_in), 1, None, None) == _lib.ERR_ARG
    assert "NULL out" in _lib.last_error()


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


@pytest.fixture(scope="module")
def ek():
    import torch_ekpose_b200 as ek
    return ek


def _batch(torch, n, h, w, people, seed, layout="nchw"):
    from torch_ekpose_b200 import synthetic
    heat, paf = synthetic.make_batch(n, h, w, people, seed=seed, layout=layout)
    return torch.from_numpy(heat).cuda(), torch.from_numpy(paf).cuda()


def _np(t):
    return t.cpu().numpy()


def _same_bytes(a, b):
    return a.shape == b.shape and np.ascontiguousarray(a).tobytes() == np.ascontiguousarray(b).tobytes()


def _host_tables(pp):
    """What the two host C calls write, overflow or not (the Python readers raise on it)."""
    n, mh = pp._rows(), pp.max_humans
    num, npk, ovf = np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.uint32)
    subset = np.zeros((n, mh, 20), np.float32)
    parts = np.zeros((n, mh, 18), PEAK_DT)
    scores = np.zeros((n, mh), np.float32)
    L = _lib.lib
    assert L.ekp_results(pp._ctx, num.ctypes.data, subset.ctypes.data, npk.ctypes.data, None, ovf.ctypes.data) in (0, _lib.ERR_CAPACITY)
    num2 = np.zeros(n, np.int32)
    assert L.ekp_results_humans(pp._ctx, num2.ctypes.data, parts.ctypes.data, scores.ctypes.data, None) in (0, _lib.ERR_CAPACITY)
    assert np.array_equal(num, num2)
    return dict(num_humans=num, n_peaks=npk, overflow=ovf, subset=subset, parts=parts, scores=scores)


def _check(got, want_res, want_tabs):
    """got: result_tensors(subset=True); want_res: results(); want_tabs: human_tables()."""
    num, parts, scores = want_tabs
    assert _same_bytes(_np(got["num_humans"]), want_res["num_humans"])
    assert _same_bytes(_np(got["num_humans"]), num)
    assert _same_bytes(_np(got["n_peaks"]), want_res["n_peaks"])
    assert _same_bytes(_np(got["overflow"]).view(np.uint32), want_res["overflow"])
    assert _same_bytes(_np(got["subset"]), want_res["subset"])
    p = _np(got["parts"])
    assert _same_bytes(p.view(PEAK_DT)[..., 0], parts)
    assert _same_bytes(_np(got["part_score"]), parts["score"])
    assert _same_bytes(_np(got["scores"]), scores)


def _check_pp(pp, got):
    _check(got, pp.results(raise_on_overflow=False), pp.human_tables())


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("frontend", ["dense", "reference", "reference_coarse", "reference_gauss"])
def test_tables_equal_the_host_readers(torch, ek, frontend, layout):
    pp = ek.PostProcessor(device=0, max_batch=16, max_h=46, max_w=54, max_peaks=1024, max_humans=32)
    heat, paf = _batch(torch, 16, 46, 54, (1, 6), 3, layout)
    pp.run(heat, paf, layout=layout, frontend=frontend)
    got = pp.result_tensors(subset=True)
    assert {k: (str(v.dtype), tuple(v.shape)) for k, v in got.items()} == {
        "num_humans": ("torch.int32", (16,)), "overflow": ("torch.int32", (16,)), "n_peaks": ("torch.int32", (16,)),
        "parts": ("torch.int32", (16, 32, 18, 4)), "part_score": ("torch.float32", (16, 32, 18)),
        "scores": ("torch.float32", (16, 32)), "subset": ("torch.float32", (16, 32, 20))}
    assert all(v.is_cuda and v.device.index == 0 for v in got.values())
    assert got["part_score"].data_ptr() == got["parts"].data_ptr() + 8     # a view of the score column
    _check_pp(pp, got)
    assert int(got["num_humans"].sum()) > 16
    assert "subset" not in pp.result_tensors()
    pp.close()


@pytest.mark.gpu
def test_bf16_host_run_peaks_and_crowded_batches(torch, ek):
    pp = ek.PostProcessor(device=0, max_batch=16, max_h=92, max_w=164, max_peaks=4096, max_humans=128, max_part=512,
                          max_cand=4096)
    heat, paf = _batch(torch, 16, 46, 54, (1, 6), 5)
    pp.run(heat.bfloat16(), paf.bfloat16())                              # 16-bit inputs
    _check_pp(pp, pp.result_tensors(subset=True))
    pb = ek.PinnedBatch(16, 46, 54)                                       # host inputs
    np.copyto(pb.heat, _np(heat)); np.copyto(pb.paf, _np(paf))
    pp.run(pb.heat, pb.paf, frontend="dense")
    _check_pp(pp, pp.result_tensors(subset=True))
    pb.close()
    rng = np.random.default_rng(5)                                        # ekp_process_paf_dev
    n, H, W, stride = 6, 96, 128, 160
    pafm = rng.normal(0, 0.6, (n, H, W, 38)).astype(np.float32)
    peaks = np.zeros((n, stride, 5), np.float32)
    counts = np.array([0, 1, 40, 90, 160, 120], np.int32)
    for i, k in enumerate(counts):
        peaks[i, :k, 0], peaks[i, :k, 1] = rng.integers(0, W, k), rng.integers(0, H, k)
        peaks[i, :k, 2], peaks[i, :k, 4] = rng.random(k), rng.integers(0, 18, k)
    pp.run_peaks(torch.from_numpy(peaks).cuda(), torch.from_numpy(counts).cuda(), torch.from_numpy(pafm).cuda(), h1=H)
    got = pp.result_tensors(subset=True)
    assert got["num_humans"].shape == (n,)
    _check_pp(pp, got)
    heat, paf = _batch(torch, 16, 92, 164, (30, 40), 9)                    # 16 crowded scenes
    pp.run(heat, paf)
    got = pp.result_tensors(subset=True)
    _check_pp(pp, got)
    assert int(got["num_humans"].min()) >= 20 and not got["overflow"].any()
    pp.close()


def _filled(torch, pp, subset=True, offset=0):
    """An out= dict of the right shapes whose every byte is 0x7f; offset > 0 places each tensor that many 4-byte words
    into a buffer (so it is not 16-byte aligned)."""
    n, mh = pp._rows(), pp.max_humans
    specs = dict(num_humans=((n,), torch.int32), overflow=((n,), torch.int32), n_peaks=((n,), torch.int32),
                 parts=((n, mh, 18, 4), torch.int32), scores=((n, mh), torch.float32))
    if subset:
        specs["subset"] = ((n, mh, 20), torch.float32)
    out = {}
    for k, (shape, dt) in specs.items():
        buf = torch.empty(int(np.prod(shape)) + offset, dtype=dt, device="cuda")
        buf.view(torch.uint8).fill_(0x7f)
        out[k] = buf[offset:].view(shape)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("max_humans,offset", [(32, 0), (31, 0), (32, 1)])   # 31 / offset 1: not all in 16-byte units
def test_zero_padding_is_written(torch, ek, max_humans, offset):
    pp = ek.PostProcessor(device=0, max_batch=8, max_h=46, max_w=54, max_peaks=1024, max_humans=max_humans)
    heat, paf = _batch(torch, 8, 46, 54, (0, 6), 12)
    pp.run(heat, paf)
    out = _filled(torch, pp, offset=offset)
    assert all(t.data_ptr() % 16 for t in out.values()) if offset else True
    got = pp.result_tensors(subset=True, out=out)
    assert got is out
    num = _np(got["num_humans"])
    assert num.min() == 0 and num.max() > 0
    for name in ("subset", "parts", "scores"):
        a = _np(got[name])
        for i, k in enumerate(num):
            assert not a[i, k:].any(), (name, i)
    _check_pp(pp, got)
    pp.close()


@pytest.mark.gpu
def test_overflow_is_reported_not_raised(torch, ek):
    pp = ek.PostProcessor(device=0, max_batch=8, max_h=46, max_w=54, max_peaks=1024, max_humans=2)
    heat, paf = _batch(torch, 8, 46, 54, (1, 6), 13)
    pp.run(heat, paf)
    got = pp.result_tensors(subset=True, out=_filled(torch, pp))
    want = _host_tables(pp)
    ovf = _np(got["overflow"]).view(np.uint32)
    assert np.array_equal(ovf, want["overflow"])
    assert (ovf & _lib.OVF_HUMANS).any()
    with pytest.raises(_lib.EkpCapacityError):
        pp.human_tables()
    for k in ("num_humans", "n_peaks", "subset", "scores"):
        assert _same_bytes(_np(got[k]), want[k]), k
    assert _same_bytes(_np(got["parts"]).view(PEAK_DT)[..., 0], want["parts"])
    pp.close()


@pytest.mark.gpu
def test_no_host_wait(torch, ek):
    pp = ek.PostProcessor(device=0, max_batch=16, max_h=46, max_w=54, max_peaks=1024, max_humans=32)
    heat, paf = _batch(torch, 16, 46, 54, (1, 6), 14)
    s = torch.cuda.Stream()
    ring = []
    for _ in range(2):   # first use of the shape: tables, graph capture; and the out= buffers
        pp.run(heat, paf, stream=s)
        ring.append(pp.result_tensors(subset=True, stream=s))
    torch.cuda.synchronize()
    want = (pp.results(), pp.human_tables())
    for out in ring:
        for t in out.values():
            t.zero_()
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(50_000_000)        # tens of ms
    pp.run(heat, paf, stream=s)
    got = pp.result_tensors(subset=True, stream=s, out=ring[0])
    fresh = pp.result_tensors(subset=True, stream=s)
    assert not s.query()
    torch.cuda.synchronize()
    _check(got, *want)
    _check(fresh, *want)
    pp.close()


@pytest.mark.gpu
def test_export_on_another_stream_then_an_immediate_run(torch, ek):
    kw = dict(device=0, max_batch=16, max_h=46, max_w=54, max_peaks=1024, max_humans=64)
    pp, ref = ek.PostProcessor(**kw), ek.PostProcessor(**kw)
    b1, b2 = _batch(torch, 16, 46, 54, (1, 6), 31), _batch(torch, 16, 46, 54, (4, 6), 32)
    ref.run(*b1)
    want1 = (ref.results(), ref.human_tables())
    ref.run(*b2)
    want2 = (ref.results(), ref.human_tables())
    s1, s2, s3 = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    pp.run(*b1, stream=s1)
    got1 = pp.result_tensors(subset=True, stream=s2)
    pp.run(*b2, stream=s1)
    got2 = pp.result_tensors(subset=True, stream=s3)
    torch.cuda.synchronize()
    _check(got1, *want1)
    _check(got2, *want2)
    _check_pp(pp, got2)
    pp.close()
    ref.close()


@pytest.mark.gpu
def test_export_has_no_side_effects(torch, ek):
    from tests import draw_check
    pp = ek.PostProcessor(device=0, max_batch=8, max_h=46, max_w=54, max_peaks=1024, max_humans=64)
    heat, paf = _batch(torch, 8, 46, 54, (1, 6), 41)
    pp.run(heat, paf)
    pp.run(heat, paf)                                    # a graph replay
    res0, tab0 = pp.results(with_peaks=True), pp.human_tables()
    launches, graphs = pp.kernel_launches(), pp.graph_launches()
    got = pp.result_tensors(subset=True)
    assert pp.kernel_launches() == launches + 1
    assert pp.graph_launches() == graphs
    res1, tab1 = pp.results(with_peaks=True), pp.human_tables()
    for k in res0:
        assert np.array_equal(res0[k], res1[k]), k
    for a, b in zip(tab0, tab1):
        assert np.array_equal(a, b)
    _check(got, res1, tab1)
    host = np.random.default_rng(1).integers(0, 256, (8, 240, 320, 3), dtype=np.uint8)
    frames = torch.from_numpy(host).cuda()
    pp.draw_humans(frames)                               # a draw after an export
    assert np.array_equal(_np(frames), draw_check.draw_batch(host, pp.humans()))
    pp.run(heat, paf)
    assert pp.graph_launches() == graphs + 1             # the batch still replays its graph
    before = pp.kernel_launches()
    assert _lib.lib.ekp_results_device(pp._ctx, 8, ctypes.byref(_lib.DeviceResults()), None) == 0
    assert pp.kernel_launches() == before                # all pointers NULL: nothing launched
    pp.close()


@pytest.mark.gpu
def test_errors(torch, ek):
    pp = ek.PostProcessor(device=0, max_batch=4, max_h=46, max_w=54, max_peaks=512, max_humans=32)
    L = _lib.lib
    num = torch.zeros(4, dtype=torch.int32, device="cuda")
    tabs = _lib.DeviceResults(num_humans=num.data_ptr())
    with pytest.raises(_lib.EkpError) as e:              # no run yet
        pp.result_tensors()
    assert e.value.code == _lib.ERR_STATE
    assert L.ekp_results_device(pp._ctx, 4, ctypes.byref(tabs), None) == _lib.ERR_STATE
    heat, paf = _batch(torch, 4, 46, 54, (1, 3), 1)
    pp.run(heat, paf)
    assert L.ekp_results_device(None, 4, ctypes.byref(tabs), None) == _lib.ERR_ARG
    assert L.ekp_results_device(pp._ctx, 4, None, None) == _lib.ERR_ARG
    assert L.ekp_results_device(pp._ctx, 3, ctypes.byref(tabs), None) == _lib.ERR_ARG
    assert L.ekp_results_device(pp._ctx, 5, ctypes.byref(tabs), None) == _lib.ERR_ARG
    buf = torch.zeros(4 * 32 * 20 + 4, dtype=torch.int32, device="cuda")
    for field in FIELDS:
        bad = _lib.DeviceResults(**{field: buf.data_ptr() + 2})
        assert L.ekp_results_device(pp._ctx, 4, ctypes.byref(bad), None) == _lib.ERR_ARG, field
        assert "aligned" in _lib.last_error()
    good = pp.result_tensors(subset=True)
    cases = []
    for k in ("num_humans", "parts", "scores", "subset"):
        v = good[k]
        cases += [(k, v[:-1]), (k, v.float() if v.dtype == torch.int32 else v.int()), (k, v.cpu()),
                  (k, v.transpose(0, 1).contiguous().transpose(0, 1) if v.dim() > 1 else v[::2])]
    for k, bad in cases:
        out = dict(good)
        out[k] = bad
        with pytest.raises(ValueError):
            pp.result_tensors(subset=True, out=out)
    out = dict(good)
    del out["overflow"]
    with pytest.raises(ValueError):
        pp.result_tensors(out=out)
    with pytest.raises(ValueError):
        pp.result_tensors(out=[good[k] for k in good])
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            pp.result_tensors(out={k: v.to("cuda:1") for k, v in good.items()})
    _check_pp(pp, pp.result_tensors(subset=True, out=_filled(torch, pp)))   # the context stays usable
    pp.close()


@pytest.mark.gpu
def test_infer_human_tensors_equals_infer_humans(torch, ek):
    from torch_ekpose_b200 import estimator
    heat, paf = _batch(torch, 3, 46, 54, (2, 5), 21)

    class FakeNet(torch.nn.Module):
        def forward(self, x):
            return (paf, heat), None

    rng = np.random.default_rng(8)
    host = rng.integers(0, 256, (3, 368, 432, 3), dtype=np.uint8)
    dev = torch.device("cuda", 0)
    estimator.infer_humans(list(host), FakeNet(), "vgg", dev)
    want_tabs = estimator.last_postprocessor().human_tables()
    want_res = estimator.last_postprocessor().results()
    _, _, want_scale = estimator.get_outputs_batched(list(host), FakeNet(), "vgg", dev)
    got, scale = estimator.infer_human_tensors(list(host), FakeNet(), "vgg", dev, subset=True)
    assert scale == want_scale
    _check(got, want_res, want_tabs)
    assert int(got["num_humans"].sum()) > 0
    got, _ = estimator.infer_human_tensors(torch.from_numpy(host).cuda(), FakeNet(), "vgg", dev)
    assert "subset" not in got
    assert _same_bytes(_np(got["parts"]).view(PEAK_DT)[..., 0], want_tabs[1])
