"""Device-only runs and the peak table on the device: ekp_set_host_copy / PostProcessor.set_host_copy, which leaves a
batch's result records on the device, and ekp_results_device_peaks / result_tensors(peaks=True), which exports the
part-sorted peak table into device tensors.  In both modes the device tables copied back must equal the host readers'
tables byte for byte, the host readers must still work after a device-only run, and a device-only batch must issue no
device-to-host copy."""
import ctypes
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from tests import util
from tests.util import assert_bits_equal
from torch_ekpose_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PEAK_DT = np.dtype([("x", np.int32), ("y", np.int32), ("score", np.float32), ("id", np.int32)])
PEAK_FIELDS = ("n_peaks", "peaks", "part_off")


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_peaks_struct_layout_equals_the_c_compilers(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ekpose_b200.h"\nint main(void) {\n'
                   '    printf("%lu", (unsigned long) sizeof(ekp_device_peaks));\n' +
                   "".join(f'    printf(" %lu", (unsigned long) offsetof(ekp_device_peaks, {f}));\n' for f in PEAK_FIELDS) +
                   '    printf("\\n");\n    return 0;\n}\n')
    exe = str(tmp_path / "layout")
    cc = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                         str(src), "-o", exe], capture_output=True, text=True)
    assert cc.returncode == 0, cc.stderr
    got = [int(v) for v in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    want = [ctypes.sizeof(_lib.DevicePeaks)] + [getattr(_lib.DevicePeaks, f).offset for f in PEAK_FIELDS]
    assert got == want


def test_null_context_or_out_is_an_argument_error_without_a_device():
    tabs = _lib.DevicePeaks()
    assert _lib.lib.ekp_results_device_peaks(None, 1, ctypes.byref(tabs), None) == _lib.ERR_ARG
    assert _lib.lib.ekp_results_device_peaks(None, 1, None, None) == _lib.ERR_ARG
    stand_in = ctypes.create_string_buffer(64)   # the NULL `out` is rejected before anything reads the context
    assert _lib.lib.ekp_results_device_peaks(ctypes.addressof(stand_in), 1, None, None) == _lib.ERR_ARG
    assert "NULL out" in _lib.last_error()
    for enable in (0, 1):
        assert _lib.lib.ekp_set_host_copy(None, enable) == _lib.ERR_ARG
        assert "NULL context" in _lib.last_error()


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


@pytest.fixture(scope="module")
def ek():
    import torch_ekpose_b200 as ek
    return ek


def _np(t):
    return t.cpu().numpy()


def _same_bytes(a, b):
    return a.shape == b.shape and np.ascontiguousarray(a).tobytes() == np.ascontiguousarray(b).tobytes()


def _host(pp):
    """Every host table of the last run: results(with_peaks=True) and human_tables(), overflow or not."""
    res = pp.results(with_peaks=True, raise_on_overflow=False)
    n, mh = pp._rows(), pp.max_humans
    num, parts, scores = np.zeros(n, np.int32), np.zeros((n, mh, 18), PEAK_DT), np.zeros((n, mh), np.float32)
    assert _lib.lib.ekp_results_humans(pp._ctx, num.ctypes.data, parts.ctypes.data, scores.ctypes.data, None) in (0, _lib.ERR_CAPACITY)
    return dict(res, hnum=num, hparts=parts, hscores=scores)


def _check(got, want):
    """got: result_tensors(subset=True, peaks=True); want: _host() of the same run."""
    for k in ("num_humans", "n_peaks", "subset", "part_off"):
        assert _same_bytes(_np(got[k]), want[k]), k
    assert _same_bytes(_np(got["overflow"]).view(np.uint32), want["overflow"])
    assert _same_bytes(_np(got["num_humans"]), want["hnum"])
    assert _same_bytes(_np(got["parts"]).view(PEAK_DT)[..., 0], want["hparts"])
    assert _same_bytes(_np(got["part_score"]), want["hparts"]["score"])
    assert _same_bytes(_np(got["scores"]), want["hscores"])
    assert _same_bytes(_np(got["peaks"]).view(PEAK_DT)[..., 0], want["peaks"])
    assert _same_bytes(_np(got["peak_score"]), want["peaks"]["score"])


def _same_host(a, b):
    for k in a:
        assert _same_bytes(np.asarray(a[k]), np.asarray(b[k])), k


def _batch(n, h, w, people, seed, layout="nchw"):
    from torch_ekpose_b200 import synthetic
    return synthetic.make_batch(n, h, w, people, seed=seed, layout=layout)


def _peaks_batch(seed):
    rng = np.random.default_rng(seed)
    n, H, W, stride = 6, 96, 128, 160
    pafm = rng.normal(0, 0.6, (n, H, W, 38)).astype(np.float32)
    peaks = np.zeros((n, stride, 5), np.float32)
    counts = np.array([0, 1, 40, 90, 160, 120], np.int32)
    for i, k in enumerate(counts):
        peaks[i, :k, 0], peaks[i, :k, 1] = rng.integers(0, W, k), rng.integers(0, H, k)
        peaks[i, :k, 2], peaks[i, :k, 4] = rng.random(k), rng.integers(0, 18, k)
    return peaks, counts, pafm, H


def _submit(torch, ek, pp, kind, frontend, seed):
    """One batch through the entry point `kind`; returns what must stay alive until the run has finished."""
    if kind == "run_peaks":
        peaks, counts, pafm, H = _peaks_batch(seed)
        keep = tuple(torch.from_numpy(a).cuda() for a in (peaks, counts, pafm))
        pp.run_peaks(*keep, h1=H)
        return keep
    layout = "nhwc" if kind == "dev_f32_nhwc" else "nchw"
    heat, paf = _batch(16, 46, 54, (1, 6), seed, layout)
    if kind.startswith("pinned"):
        pb = ek.PinnedBatch(16, 46, 54, dtype="float16" if kind == "pinned_f16" else "float32")
        np.copyto(pb.heat, heat.astype(pb.heat.dtype)); np.copyto(pb.paf, paf.astype(pb.paf.dtype))
        pp.run(pb.heat, pb.paf, frontend=frontend)
        return pb
    hd, pd = torch.from_numpy(heat).cuda(), torch.from_numpy(paf).cuda()
    if kind == "dev_bf16":
        hd, pd = hd.bfloat16(), pd.bfloat16()
    pp.run(hd, pd, layout=layout, frontend=frontend)
    return hd, pd


# every map entry point with both front-ends, and run_peaks (which takes peaks: it has no front-end)
CASES = [(fe, kind) for fe in ("reference", "dense")
         for kind in ("dev_f32_nchw", "dev_f32_nhwc", "dev_bf16", "pinned_f32", "pinned_f16")] + [("none", "run_peaks")]


@pytest.mark.gpu
@pytest.mark.parametrize("frontend,kind", CASES)
def test_tables_equal_in_both_modes(torch, ek, frontend, kind):
    kw = dict(device=0, max_batch=16, max_h=46, max_w=54, max_peaks=1024, max_humans=32)
    if kind == "run_peaks":
        kw.update(max_h=12, max_w=16, max_peaks=256, max_humans=128)
    host_pp, dev_pp = ek.PostProcessor(**kw), ek.PostProcessor(**kw)
    dev_pp.set_host_copy(False)
    assert host_pp.host_copy and not dev_pp.host_copy
    for rep in range(2):   # the second batch of each context replays its graph
        keep = [_submit(torch, ek, pp, kind, frontend, 40 + rep) for pp in (host_pp, dev_pp)]
        got = [pp.result_tensors(subset=True, peaks=True) for pp in (host_pp, dev_pp)]
        torch.cuda.synchronize()
        for t in got:   # the device tables come before any host read of the run
            assert {k: (str(v.dtype), tuple(v.shape)) for k, v in t.items() if k in ("peaks", "peak_score", "part_off")} == {
                "peaks": ("torch.int32", (len(t["n_peaks"]), kw["max_peaks"], 4)),
                "peak_score": ("torch.float32", (len(t["n_peaks"]), kw["max_peaks"])),
                "part_off": ("torch.int32", (len(t["n_peaks"]), 19))}
            assert t["peak_score"].data_ptr() == t["peaks"].data_ptr() + 8
        want_host, want_dev = _host(host_pp), _host(dev_pp)
        _same_host(want_dev, want_host)                   # host tables after a device-only run == host-copy run's
        _same_host(_host(dev_pp), want_dev)               # a second read (no second download) reads the same
        _check(got[0], want_host)
        _check(got[1], want_dev)
        assert int(want_host["n_peaks"].sum()) > 0 and (kind == "run_peaks" or int(want_host["num_humans"].sum()) > 0)
        del keep
    assert host_pp.graph_launches() == dev_pp.graph_launches()
    host_pp.close()
    dev_pp.close()


@pytest.mark.gpu
@pytest.mark.parametrize("frontend", ["reference", "dense"])
def test_full_batch_equals_the_oracle_device_only(torch, ek, frontend):
    """configs[1]: 64 x 46x54 at full batch, host copy off, the device tables against the oracle."""
    pp = ek.PostProcessor(device=0, max_batch=64, max_h=46, max_w=54, max_peaks=1024, max_humans=32)
    pp.set_host_copy(False)
    heat, paf = _batch(64, 46, 54, (1, 6), 7)
    pp.run(torch.from_numpy(heat).cuda(), torch.from_numpy(paf).cuda(), frontend=frontend)
    got = pp.result_tensors(subset=True, peaks=True)
    dev = dict(n_peaks=_np(got["n_peaks"]), peaks=_np(got["peaks"]).view(PEAK_DT)[..., 0], part_off=_np(got["part_off"]))
    assert not got["overflow"].any()
    subset, num = _np(got["subset"]), _np(got["num_humans"])
    for i in range(64):
        hw, pw = np.ascontiguousarray(heat[i].transpose(1, 2, 0)), np.ascontiguousarray(paf[i].transpose(1, 2, 0))
        peaks, sub = (util.oracle_dense if frontend == "dense" else util.oracle_reference)(hw, pw)
        assert_bits_equal(util.peaks_table(dev, i), peaks, f"image {i} peaks")
        assert int(num[i]) == len(sub), (i, int(num[i]), len(sub))
        assert_bits_equal(subset[i, :len(sub)], sub, f"image {i} subset")
    _check(got, _host(pp))
    pp.close()


@pytest.mark.gpu
def test_switching_modes_on_the_same_buffers(torch, ek):
    """Every batch goes through the same input tensors, with new contents and the mode flipped in a fixed pattern.  A
    host-copy batch that replayed a device-only graph would leave the previous batch's records in the host mirror, and a
    device-only batch that replayed a host-copy graph would take the host readers' stale-records path: either shows up as
    tables that differ from a context that always copies."""
    kw = dict(device=0, max_batch=16, max_h=46, max_w=54, max_peaks=1024, max_humans=32)
    pp, ref = ek.PostProcessor(**kw), ek.PostProcessor(**kw)
    sets = [_batch(16, 46, 54, (1, 6), 60 + s) for s in range(3)]
    hd, pd = torch.from_numpy(sets[0][0]).cuda(), torch.from_numpy(sets[0][1]).cuda()
    pattern = [True, False, False, True, False, True, True, False]
    graphs = pp.graph_launches()
    for b, mode in enumerate(pattern):
        heat, paf = sets[b % 3]
        hd.copy_(torch.from_numpy(heat)); pd.copy_(torch.from_numpy(paf))
        pp.set_host_copy(mode)
        pp.run(hd, pd)
        got = pp.result_tensors(subset=True, peaks=True)
        ref.run(hd, pd)
        want = _host(ref)
        if b % 2:   # device tables first, then the host readers; and the other way round
            torch.cuda.synchronize()
            _check(got, want)
            _same_host(_host(pp), want)
        else:
            _same_host(_host(pp), want)
            _check(got, want)
    assert pp.graph_launches() == graphs + len(pattern)
    pp.close()
    ref.close()


def _filled(torch, n, shape_of, offset):
    """out= tensors for result_tensors(subset=True, peaks=True) whose every byte is 0xff; offset > 0 places each that many
    4-byte words into a buffer (so it is not 16-byte aligned)."""
    out = {}
    for k, shape in shape_of.items():
        dt = torch.float32 if k in ("subset", "scores") else torch.int32
        buf = torch.empty(int(np.prod(shape)) + offset, dtype=dt, device="cuda")
        buf.view(torch.uint8).fill_(0xff)
        out[k] = buf[offset:].view(shape)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("host_copy", [True, False])
@pytest.mark.parametrize("offset", [0, 1])
def test_stale_rows_are_zeroed(torch, ek, host_copy, offset):
    n, mh, mp = 16, 128, 2048
    pp = ek.PostProcessor(device=0, max_batch=n, max_h=92, max_w=164, max_peaks=mp, max_humans=mh, max_part=512, max_cand=4096)
    pp.set_host_copy(host_copy)
    shapes = dict(num_humans=(n,), overflow=(n,), n_peaks=(n,), parts=(n, mh, 18, 4), scores=(n, mh), subset=(n, mh, 20),
                  peaks=(n, mp, 4), part_off=(n, 19))
    out = _filled(torch, n, shapes, offset)
    if offset:
        assert all(t.data_ptr() % 16 for t in out.values())
    crowd = _batch(n, 92, 164, (30, 40), 9)
    sparse = _batch(n, 46, 54, (0, 1), 10)
    for heat, paf in (crowd, sparse):
        pp.run(torch.from_numpy(heat).cuda(), torch.from_numpy(paf).cuda())
        got = pp.result_tensors(subset=True, peaks=True, out=out)
        assert got is out
        torch.cuda.synchronize()
        num, npk = _np(got["num_humans"]), _np(got["n_peaks"])
        assert not got["overflow"].any()
        for i in range(n):
            for k in ("subset", "parts", "scores"):
                assert not _np(got[k])[i, num[i]:].any(), (k, i)
            assert not _np(got["peaks"])[i, npk[i]:].any(), i
        _check(got, _host(pp))
    assert int(npk.min()) == 0 and int(num.min()) == 0   # the sparse batch's empty images, after a crowd
    pp.close()


@pytest.mark.gpu
@pytest.mark.parametrize("host_copy", [True, False])
def test_peak_overflow_exports_what_the_host_returns(torch, ek, host_copy):
    n, mp = 8, 64
    pp = ek.PostProcessor(device=0, max_batch=n, max_h=46, max_w=54, max_peaks=mp, max_humans=128)
    pp.set_host_copy(host_copy)
    heat, paf = _batch(n, 46, 54, (0, 7), 11)   # 0 .. 7 people: the crowded half has more than 64 peaks
    pp.run(torch.from_numpy(heat).cuda(), torch.from_numpy(paf).cuda())
    shapes = dict(num_humans=(n,), overflow=(n,), n_peaks=(n,), parts=(n, 128, 18, 4), scores=(n, 128), subset=(n, 128, 20),
                  peaks=(n, mp, 4), part_off=(n, 19))
    got = pp.result_tensors(subset=True, peaks=True, out=_filled(torch, n, shapes, 0))
    want = _host(pp)
    ovf = _np(got["overflow"]).view(np.uint32)
    npk = _np(got["n_peaks"])
    over = (ovf & _lib.OVF_PEAKS) != 0
    assert over.any() and not over.all(), (ovf, npk)
    assert (npk[over] == mp).all() and (npk[~over] <= mp).all()   # an overflowing image reports a full table
    with pytest.raises(_lib.EkpCapacityError):
        pp.results()
    _check(got, want)
    pp.close()


@pytest.mark.gpu
@pytest.mark.parametrize("host_copy", [True, False])
def test_export_on_a_second_stream_then_an_immediate_run(torch, ek, host_copy):
    """The export waits for the run on another stream, and the next run (submitted at once on the first stream) waits
    for the export: the exported tables are the first run's, by the oracle."""
    pp = ek.PostProcessor(device=0, max_batch=16, max_h=46, max_w=54, max_peaks=1024, max_humans=32)
    pp.set_host_copy(host_copy)
    b1, b2 = _batch(16, 46, 54, (1, 6), 71), _batch(16, 46, 54, (3, 6), 72)
    d1 = tuple(torch.from_numpy(a).cuda() for a in b1)
    d2 = tuple(torch.from_numpy(a).cuda() for a in b2)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    pp.run(*d1, stream=s1)
    with torch.cuda.stream(s2):
        torch.cuda._sleep(50_000_000)        # tens of ms: the export is still queued when the next run is submitted
    got = pp.result_tensors(subset=True, peaks=True, stream=s2)
    pp.run(*d2, stream=s1)
    torch.cuda.synchronize()
    dev = dict(n_peaks=_np(got["n_peaks"]), peaks=_np(got["peaks"]).view(PEAK_DT)[..., 0], part_off=_np(got["part_off"]))
    num, subset = _np(got["num_humans"]), _np(got["subset"])
    heat, paf = b1
    for i in range(16):
        hw, pw = np.ascontiguousarray(heat[i].transpose(1, 2, 0)), np.ascontiguousarray(paf[i].transpose(1, 2, 0))
        peaks, sub = util.oracle_reference(hw, pw)
        assert_bits_equal(util.peaks_table(dev, i), peaks, f"image {i} peaks")
        assert int(num[i]) == len(sub)
        assert_bits_equal(subset[i, :len(sub)], sub, f"image {i} subset")
    res2 = pp.results(with_peaks=True)                    # and the second run is intact
    heat, paf = b2
    for i in range(16):
        hw, pw = np.ascontiguousarray(heat[i].transpose(1, 2, 0)), np.ascontiguousarray(paf[i].transpose(1, 2, 0))
        peaks, sub = util.oracle_reference(hw, pw)
        assert_bits_equal(util.peaks_table(res2, i), peaks, f"run 2 image {i} peaks")
        assert int(res2["num_humans"][i]) == len(sub)
    pp.close()


@pytest.mark.gpu
def test_errors_and_launch_counts(torch, ek):
    pp = ek.PostProcessor(device=0, max_batch=4, max_h=46, max_w=54, max_peaks=512, max_humans=32)
    L = _lib.lib
    npk = torch.zeros(4, dtype=torch.int32, device="cuda")
    tabs = _lib.DevicePeaks(n_peaks=npk.data_ptr())
    assert L.ekp_results_device_peaks(pp._ctx, 4, ctypes.byref(tabs), None) == _lib.ERR_STATE   # no run yet
    assert "no run" in _lib.last_error()
    heat, paf = _batch(4, 46, 54, (1, 3), 1)
    pp.set_host_copy(False)
    pp.run(torch.from_numpy(heat).cuda(), torch.from_numpy(paf).cuda())
    assert L.ekp_results_device_peaks(None, 4, ctypes.byref(tabs), None) == _lib.ERR_ARG
    assert L.ekp_results_device_peaks(pp._ctx, 4, None, None) == _lib.ERR_ARG
    assert L.ekp_results_device_peaks(pp._ctx, 3, ctypes.byref(tabs), None) == _lib.ERR_ARG
    assert L.ekp_results_device_peaks(pp._ctx, 5, ctypes.byref(tabs), None) == _lib.ERR_ARG
    buf = torch.zeros(4 * 512 * 4 + 4, dtype=torch.int32, device="cuda")
    for field in PEAK_FIELDS:
        bad = _lib.DevicePeaks(**{field: buf.data_ptr() + 2})
        assert L.ekp_results_device_peaks(pp._ctx, 4, ctypes.byref(bad), None) == _lib.ERR_ARG, field
        assert "aligned" in _lib.last_error()
    before = pp.kernel_launches()
    assert L.ekp_results_device_peaks(pp._ctx, 4, ctypes.byref(_lib.DevicePeaks()), None) == 0
    assert pp.kernel_launches() == before                 # all pointers NULL: nothing launched
    good = pp.result_tensors(subset=True, peaks=True)
    assert pp.kernel_launches() == before + 2             # the people's export and the peaks' export
    for k in ("peaks", "part_off"):
        v = good[k]
        for bad in (v[:-1], v.float(), v.cpu(), v.transpose(0, 1).contiguous().transpose(0, 1)):
            out = dict(good)
            out[k] = bad
            with pytest.raises(ValueError):
                pp.result_tensors(peaks=True, out=out)
    out = dict(good)
    del out["part_off"]
    with pytest.raises(ValueError):
        pp.result_tensors(peaks=True, out=out)
    pp.result_tensors(out=out)                            # without peaks=True the peak tensors are not needed
    _check(pp.result_tensors(subset=True, peaks=True, out=good), _host(pp))
    pp.close()


@pytest.mark.gpu
def test_growing_keeps_the_mode(torch, ek):
    from torch_ekpose_b200 import paf_to_pose
    paf_to_pose._cache.clear()
    heat, paf = _batch(2, 46, 54, (3, 4), 2)
    pp = paf_to_pose._processor(0, 2, 46, 54, max_peaks=1024, max_humans=1)
    pp.set_host_copy(False)
    grown = paf_to_pose._run_growing(0, torch.from_numpy(heat).cuda(), torch.from_numpy(paf).cuda(), 2, 46, 54,
                                     dict(max_peaks=1024, max_humans=1), _lib.OVF_HUMANS)
    assert grown is not pp and grown.max_humans > 1
    assert grown.host_copy is False
    paf_to_pose._cache.clear()


# ---- device-to-host copies, from a profiler trace in a fresh process -------------------------------------------------
def _trace_worker(out_path):
    import torch
    from torch.profiler import ProfilerActivity, profile

    import torch_ekpose_b200 as ek
    from torch_ekpose_b200 import estimator

    def trace(fn):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        names = [e.name for e in prof.events()]
        return dict(dtoh=sum(bool(re.search(r"memcpy.*dtoh", e, re.I)) for e in names),
                    assemble=sum("assemble_kernel" in e for e in names))

    out = {}
    n = 64
    pp = ek.PostProcessor(device=0, max_batch=n, max_h=46, max_w=54, max_peaks=1024, max_humans=32)
    sets = [_batch(n, 46, 54, (1, 6), 80 + s) for s in range(2)]
    hd, pd = torch.from_numpy(sets[0][0]).cuda(), torch.from_numpy(sets[0][1]).cuda()
    ring = None
    for mode in (True, False, True, False):   # tables, graph capture of each mode, the out= buffers
        pp.set_host_copy(mode)
        pp.run(hd, pd)
        ring = pp.result_tensors(subset=True, peaks=True, out=ring)
    pp.results()

    def batches(pattern):
        def fn():
            for b, mode in enumerate(pattern):
                hd.copy_(torch.from_numpy(sets[b % 2][0]), non_blocking=False)
                pp.set_host_copy(mode)
                pp.run(hd, pd)
                pp.result_tensors(subset=True, peaks=True, out=ring)
        return fn

    for name, pattern in (("off", [False] * 4), ("on", [True] * 4), ("mixed", [True, False, False, True, False, True])):
        g0 = pp.graph_launches()
        out[name] = dict(trace(batches(pattern)), batches=len(pattern), on=sum(pattern), graphs=pp.graph_launches() - g0)
    pp.close()

    heat, paf = (torch.from_numpy(a).cuda() for a in _batch(3, 46, 54, (2, 5), 21))

    class FakeNet(torch.nn.Module):
        def forward(self, x):
            return (paf, heat), None

    frames = torch.from_numpy(np.random.default_rng(8).integers(0, 256, (3, 368, 432, 3), dtype=np.uint8)).cuda()
    dev = torch.device("cuda", 0)
    estimator.infer_humans(frames, FakeNet(), "vgg", dev)
    want = estimator.last_postprocessor().human_tables()
    for _ in range(2):
        estimator.infer_human_tensors(frames, FakeNet(), "vgg", dev, peaks=True)
        estimator.infer_and_draw(frames.clone(), FakeNet(), "vgg", dev)
    drawn = frames.clone()
    got = {}
    out["infer_human_tensors"] = trace(lambda: got.update(t=estimator.infer_human_tensors(frames, FakeNet(), "vgg", dev, peaks=True)[0]))
    out["infer_and_draw"] = trace(lambda: estimator.infer_and_draw(drawn, FakeNet(), "vgg", dev))
    after = estimator.last_postprocessor().human_tables()
    out["humans_equal"] = all(np.array_equal(a, b) for a, b in zip(want, after))
    t = got["t"]
    out["tensors_equal"] = bool(np.array_equal(t["num_humans"].cpu().numpy(), want[0]) and
                                np.array_equal(t["parts"].cpu().numpy().view(PEAK_DT)[..., 0], want[1]))
    out["peaks_rows"] = int(t["n_peaks"].sum())
    with open(out_path, "w") as f:
        json.dump(out, f)


_WORKER = "import sys; from tests.test_device_only import _trace_worker; _trace_worker(sys.argv[1])"


@pytest.fixture(scope="module")
def traces(tmp_path_factory):
    done = {}

    def run(graphs):
        if graphs not in done:
            path = tmp_path_factory.mktemp("trace") / "out.json"
            env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
            env.pop("EKP_GRAPHS", None)
            if not graphs:
                env["EKP_GRAPHS"] = "0"
            r = subprocess.run([sys.executable, "-c", _WORKER, str(path)], capture_output=True, text=True, env=env, cwd=ROOT,
                               timeout=1200)
            assert r.returncode == 0, f"worker exited {r.returncode}:\n{r.stderr[-3000:]}"
            with open(path) as f:
                done[graphs] = json.load(f)
        return done[graphs]
    return run


@pytest.mark.gpu
def test_eager_device_only_batches_copy_nothing_to_the_host(traces):
    t = traces(False)
    for name in ("off", "on", "mixed"):
        c = t[name]
        assert c["graphs"] == 0, c
        assert c["assemble"] == c["batches"], c      # the trace sees every batch's kernels
        assert c["dtoh"] == c["on"], c               # one records copy per host-copy batch, none otherwise
    for name in ("infer_human_tensors", "infer_and_draw"):
        assert t[name]["dtoh"] == 0 and t[name]["assemble"] == 1, t[name]
    assert t["humans_equal"] and t["tensors_equal"] and t["peaks_rows"] > 0


@pytest.mark.gpu
def test_graph_replays_of_device_only_batches_copy_nothing_to_the_host(traces):
    t = traces(True)
    for name in ("off", "on", "mixed"):
        c = t[name]
        assert c["graphs"] == c["batches"], c        # every batch replayed a graph
        assert c["assemble"] == c["batches"], c      # and the trace lists the nodes of graph replays
        assert c["dtoh"] == c["on"], c
    for name in ("infer_human_tensors", "infer_and_draw"):
        assert t[name]["dtoh"] == 0 and t[name]["assemble"] == 1, t[name]
    assert t["humans_equal"] and t["tensors_equal"] and t["peaks_rows"] > 0
