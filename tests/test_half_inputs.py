"""bf16 / fp16 heat and PAF maps (what a network returns under torch.autocast): widened to float32 on the device, they
must give bit for bit what the float32 path gives on x16.float() -- people, peaks, human tables and, where
materialised, the operator-surface tensors -- through every entry point, layout, front-end, alignment and graph
replay."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import util
from tests.util import assert_bits_equal

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DTYPES = {"bf16": torch.bfloat16, "fp16": torch.float16}
FRONTENDS = ["dense", "reference", "reference_coarse", "reference_gauss"]


@pytest.fixture(scope="module")
def ek():
    import torch_ekpose_b200 as ek
    return ek


@pytest.fixture(scope="module")
def pair(ek):
    """Two contexts of equal capacity: the float32 reference run and the 16-bit run, each with its own buffers."""
    kw = dict(device=0, max_batch=64, max_h=92, max_w=164, max_peaks=4096, max_humans=128, max_part=512, max_cand=4096)
    a, b = ek.PostProcessor(**kw), ek.PostProcessor(**kw)
    yield a, b
    a.close()
    b.close()


@functools.lru_cache(maxsize=None)
def _batch(n, h, w, people, seed, layout="nchw"):
    from torch_ekpose_b200 import synthetic
    return synthetic.make_batch(n, h, w, people, seed=seed, layout=layout)


def _dev16(a, dt):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda().to(dt)


def _outputs(pp, materialize=False):
    res = pp.results(with_peaks=True, raise_on_overflow=False)
    num, parts, scores = pp.human_tables() if not res["overflow"].any() else (None, None, None)
    out = dict(res, h_num=num, h_parts=parts, h_scores=scores)
    if materialize:
        out["heat_mat"], out["paf_mat"] = pp.heat_mat.clone(), pp.paf_mat.clone()
    return out


def _assert_same(want, got, what):
    for k in ("num_humans", "n_peaks", "overflow", "part_off"):
        assert np.array_equal(want[k], got[k]), f"{what}: {k}"
    assert_bits_equal(want["subset"], got["subset"], f"{what}: subset")
    assert np.array_equal(want["peaks"].view(np.int32), got["peaks"].view(np.int32)), f"{what}: peak table"
    if want["h_num"] is not None:
        assert np.array_equal(want["h_num"], got["h_num"]), f"{what}: human count"
        assert np.array_equal(want["h_parts"].view(np.int32), got["h_parts"].view(np.int32)), f"{what}: human parts"
        assert_bits_equal(want["h_scores"], got["h_scores"], f"{what}: human scores")
    for k in ("heat_mat", "paf_mat"):
        if k in want and k in got:
            assert torch.equal(want[k].view(torch.int32), got[k].view(torch.int32)), f"{what}: {k}"


def _run_pair(pair, heat, paf, dt, **kw):
    """The float32 run on x16.float() and the 16-bit run on x16 (device entry); returns both outputs."""
    a, b = pair
    h16, p16 = _dev16(heat, dt), _dev16(paf, dt)
    mat = kw.get("materialize", False)
    a.run(h16.float(), p16.float(), **kw)
    want = _outputs(a, mat)
    b.run(h16, p16, **kw)
    got = _outputs(b, mat)
    return want, got


# 1. device entry, every front-end x layout x materialisation ----------------------------------------------------
@pytest.mark.parametrize("materialize", [False, True])
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("frontend", FRONTENDS)
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_device_entry_equals_float32(pair, dtype, frontend, layout, materialize):
    heat, paf = _batch(6, 46, 54, (1, 6), 40, layout)
    want, got = _run_pair(pair, heat, paf, DTYPES[dtype], layout=layout, frontend=frontend, materialize=materialize)
    assert want["num_humans"].sum() > 0
    _assert_same(want, got, f"{dtype} {frontend} {layout} mat={materialize}")


# 2. shapes that take the other code paths -------------------------------------------------------------------------
SHAPES = {
    "c2_64x46x54": (64, 46, 54, (1, 6), 41),
    "single_46x54": (1, 46, 54, (3, 3), 42),       # the sliced plane kernel
    "crowd_16x92x164": (16, 92, 164, (30, 40), 43),
    "odd_3x5x5": (3, 5, 5, (1, 2), 44),           # plane sizes that are not multiples of 8 elements
    "odd_3x23x37": (3, 23, 37, (1, 4), 45),
    "odd_2x46x82": (2, 46, 82, (2, 8), 46),
}


@pytest.mark.parametrize("frontend", ["dense", "reference"])
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_shapes_equal_float32(pair, dtype, shape, frontend):
    n, h, w, people, seed = SHAPES[shape]
    heat, paf = _batch(n, h, w, people, seed)
    want, got = _run_pair(pair, heat, paf, DTYPES[dtype], frontend=frontend)
    _assert_same(want, got, f"{dtype} {shape} {frontend}")


# 3. against the oracle on the widened maps -------------------------------------------------------------------------
@pytest.mark.parametrize("frontend", ["dense", "reference"])
def test_bf16_batch_against_the_oracle(pair, frontend):
    heat, paf = _batch(4, 46, 54, (2, 5), 47)
    h16, p16 = _dev16(heat, torch.bfloat16), _dev16(paf, torch.bfloat16)
    hw32, pw32 = h16.float().cpu().numpy(), p16.float().cpu().numpy()
    pp = pair[1]
    pp.run(h16, p16, frontend=frontend)
    res = pp.results(with_peaks=True)
    for i in range(4):
        hw, pw = np.ascontiguousarray(hw32[i].transpose(1, 2, 0)), np.ascontiguousarray(pw32[i].transpose(1, 2, 0))
        peaks, sub = (util.oracle_dense if frontend == "dense" else util.oracle_reference)(hw, pw)
        assert_bits_equal(util.peaks_table(res, i), peaks, f"image {i} peaks")
        m = int(res["num_humans"][i])
        assert m == len(sub) > 0, (i, m, len(sub))
        assert_bits_equal(res["subset"][i, :m], sub, f"image {i} subset")


# 4. alignment ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_inputs_that_are_only_2_byte_aligned(pair, dtype):
    dt = DTYPES[dtype]
    heat, paf = _batch(3, 46, 54, (2, 4), 48)
    a, b = pair
    h16, p16 = _dev16(heat, dt), _dev16(paf, dt)
    hb = torch.zeros(heat.size + 3, dtype=dt, device="cuda")
    pb = torch.zeros(paf.size + 1, dtype=dt, device="cuda")
    hv, pv = hb[3:].view(heat.shape), pb[1:].view(paf.shape)
    hv.copy_(h16); pv.copy_(p16)
    assert hv.data_ptr() % 16 != 0 and pv.data_ptr() % 16 != 0 and hv.data_ptr() % 2 == 0
    for frontend, mat in (("dense", True), ("dense", False), ("reference", False)):
        a.run(h16.float(), p16.float(), frontend=frontend, materialize=mat)
        want = _outputs(a, mat)
        b.run(hv, pv, frontend=frontend, materialize=mat)
        _assert_same(want, _outputs(b, mat), f"{dtype} offset views {frontend} mat={mat}")


def test_misaligned_pointers_and_unknown_dtypes_are_rejected(ek, pair):
    _lib = ek._lib
    pp = pair[1]
    h16 = torch.zeros((1, 19, 8, 8), dtype=torch.bfloat16, device="cuda")
    p16 = torch.zeros((1, 38, 8, 8), dtype=torch.bfloat16, device="cuda")
    rc = _lib.lib.ekp_postprocess_typed(pp._ctx, h16.data_ptr() + 1, p16.data_ptr(), _lib.DTYPE_BF16, 1, 8, 8, 0, 0.15, 0,
                                        None, None, None)
    assert rc == _lib.ERR_ARG and "2-byte" in _lib.last_error()
    rc = _lib.lib.ekp_postprocess_typed(pp._ctx, h16.data_ptr(), p16.data_ptr() + 1, _lib.DTYPE_F16, 1, 8, 8, 0, 0.15, 0,
                                        None, None, None)
    assert rc == _lib.ERR_ARG
    for bad in (3, -1):
        rc = _lib.lib.ekp_postprocess_typed(pp._ctx, h16.data_ptr(), p16.data_ptr(), bad, 1, 8, 8, 0, 0.15, 0, None, None, None)
        assert rc == _lib.ERR_ARG and "dtype" in _lib.last_error()
        hh, ph = np.zeros(19 * 64, np.float16), np.zeros(38 * 64, np.float16)
        rc = _lib.lib.ekp_postprocess_host_typed(pp._ctx, hh.ctypes.data, ph.ctypes.data, bad, 1, 8, 8, 0, 0.15, 0, 0, None)
        assert rc == _lib.ERR_ARG and "dtype" in _lib.last_error()


# 5. host entry -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("frontend", ["dense", "reference"])
def test_host_entry_equals_device_entry(ek, pair, frontend):
    heat, paf = _batch(8, 46, 54, (1, 6), 49)
    a, b = pair
    for mat in (False, True):
        for dtype, dt in DTYPES.items():
            h16, p16 = _dev16(heat, dt), _dev16(paf, dt)
            a.run(h16, p16, frontend=frontend, materialize=mat)
            want = _outputs(a)
            hc, pc = h16.cpu(), p16.cpu()
            inputs = {"pageable torch": (hc, pc)}
            if dtype == "fp16":
                inputs["pageable numpy"] = (hc.numpy(), pc.numpy())
            pinned = ek.PinnedBatch(8, 46, 54, dtype={"bf16": "bfloat16", "fp16": "float16"}[dtype])
            assert pinned.nbytes == 2 * 8 * 46 * 54 * 57
            if dtype == "fp16":
                assert pinned.heat.dtype == np.float16
                np.copyto(pinned.heat, hc.numpy()); np.copyto(pinned.paf, pc.numpy())
            else:
                assert pinned.heat.dtype == torch.bfloat16 and not pinned.heat.is_cuda
                pinned.heat.copy_(hc); pinned.paf.copy_(pc)
            inputs["pinned block"] = (pinned.heat, pinned.paf)
            for kind, (hh, ph) in inputs.items():
                b.run(hh, ph, frontend=frontend, materialize=mat)
                _assert_same(want, _outputs(b), f"{dtype} {kind} {frontend} mat={mat}")
            pinned.close()


def test_pinned_batch_dtypes(ek):
    for dtype, item in (("float32", 4), ("float16", 2), ("bfloat16", 2)):
        for layout in ("nchw", "nhwc"):
            pb = ek.PinnedBatch(2, 6, 7, layout, dtype=dtype)
            assert pb.nbytes == item * 2 * 6 * 7 * 57
            want_h = (2, 19, 6, 7) if layout == "nchw" else (2, 6, 7, 19)
            assert tuple(pb.heat.shape) == want_h
            # heat directly followed by paf: the library moves the block with one copy
            ptr = (lambda x: x.data_ptr()) if dtype == "bfloat16" else (lambda x: x.ctypes.data)
            assert ptr(pb.paf) == ptr(pb.heat) + item * 2 * 6 * 7 * 19
            pb.close()
    with pytest.raises(ValueError):
        ek.PinnedBatch(1, 5, 5, dtype="float64")


# 6. graphs ---------------------------------------------------------------------------------------------------------
def test_repeated_16bit_batches_replay_as_graphs(ek, pair):
    heat, paf = _batch(8, 46, 54, (2, 5), 50)
    a, b = pair
    h16, p16 = _dev16(heat, torch.bfloat16), _dev16(paf, torch.bfloat16)
    a.run(h16.float(), p16.float(), frontend="dense", materialize=True)
    want = _outputs(a, True)
    pb = ek.PinnedBatch(8, 46, 54, dtype="float16")
    np.copyto(pb.heat, heat.astype(np.float16)); np.copyto(pb.paf, paf.astype(np.float16))
    a.run(torch.from_numpy(pb.heat).cuda().float(), torch.from_numpy(pb.paf).cuda().float(), frontend="reference")
    want_host = _outputs(a)
    for rep in range(4):
        g0 = b.graph_launches()
        b.run(h16, p16, frontend="dense", materialize=True)
        assert b.graph_launches() == g0 + 1
        _assert_same(want, _outputs(b, True), f"device rep {rep}")
        g0 = b.graph_launches()
        b.run(pb.heat, pb.paf, frontend="reference")
        assert b.graph_launches() == g0 + 1
        _assert_same(want_host, _outputs(b), f"pinned rep {rep}")
    pb.close()


def test_graph_replay_reads_the_16bit_buffers_current_content(ek, pair):
    scenes = [_batch(4, 46, 54, (p, p + 2), 300 + p) for p in (1, 3, 5)]
    a, b = pair
    dev_h = torch.empty(scenes[0][0].shape, dtype=torch.bfloat16, device="cuda")
    dev_p = torch.empty(scenes[0][1].shape, dtype=torch.bfloat16, device="cuda")
    host_h, host_p = np.empty(scenes[0][0].shape, np.float16), np.empty(scenes[0][1].shape, np.float16)
    pb = ek.PinnedBatch(4, 46, 54, dtype="bfloat16")
    g0 = b.graph_launches()
    for rounds in range(2):
        for heat, paf in scenes:
            dev_h.copy_(torch.from_numpy(heat)); dev_p.copy_(torch.from_numpy(paf))
            a.run(dev_h.float(), dev_p.float(), frontend="reference")
            want = _outputs(a)
            b.run(dev_h, dev_p, frontend="reference")
            _assert_same(want, _outputs(b), f"device bf16 round {rounds}")
            pb.heat.copy_(dev_h.cpu()); pb.paf.copy_(dev_p.cpu())
            b.run(pb.heat, pb.paf, frontend="reference")
            _assert_same(want, _outputs(b), f"pinned bf16 round {rounds}")
            host_h[...] = heat; host_p[...] = paf
            a.run(torch.from_numpy(host_h).cuda().float(), torch.from_numpy(host_p).cuda().float(), frontend="reference")
            want = _outputs(a)
            b.run(host_h, host_p, frontend="reference")
            _assert_same(want, _outputs(b), f"pageable fp16 round {rounds}")
    assert b.graph_launches() - g0 == 18
    pb.close()


def test_same_pointer_and_shape_with_another_dtype_is_another_graph(pair):
    """One device buffer viewed as float32, bf16 and fp16 at the same data_ptr() and shape: none may replay another's
    graph (bf16 and fp16 views differ in nothing else)."""
    heat_a, paf_a = _batch(4, 46, 54, (2, 4), 51)
    heat_b, paf_b = _batch(4, 46, 54, (3, 5), 52)
    a, b = pair
    hbuf = torch.empty(heat_a.size, dtype=torch.float32, device="cuda")
    pbuf = torch.empty(paf_a.size, dtype=torch.float32, device="cuda")
    views = {torch.float32: (hbuf.view(heat_a.shape), pbuf.view(paf_a.shape))}
    for dt in DTYPES.values():
        views[dt] = (hbuf.view(dt)[:heat_a.size].view(heat_a.shape), pbuf.view(dt)[:paf_a.size].view(paf_a.shape))
        assert views[dt][0].data_ptr() == hbuf.data_ptr() and views[dt][0].shape == views[torch.float32][0].shape
    data = {torch.float32: (heat_a, paf_a), torch.bfloat16: (heat_b, paf_b), torch.float16: (heat_b, paf_b)}
    want = {}
    for dt, (heat, paf) in data.items():
        a.run(_dev16(heat, dt).float(), _dev16(paf, dt).float(), frontend="dense")
        want[dt] = _outputs(a)
    for rep in range(2):
        for dt, (hv, pv) in views.items():
            hv.copy_(torch.from_numpy(data[dt][0])); pv.copy_(torch.from_numpy(data[dt][1]))
            b.run(hv, pv, frontend="dense")
            _assert_same(want[dt], _outputs(b), f"{dt} view rep {rep}")


# 7. launch count ---------------------------------------------------------------------------------------------------
_LAUNCH_SCRIPT = r"""
import json, sys, numpy as np, torch
import torch_ekpose_b200 as ek
from torch_ekpose_b200 import synthetic
heat, paf = synthetic.make_batch(4, 46, 54, (2, 4), seed=53)
pp = ek.PostProcessor(device=0, max_batch=4, max_h=46, max_w=54, max_peaks=1024, max_humans=32)
out = {}
for frontend in ("dense", "reference", "reference_coarse", "reference_gauss"):
    for mat in (False, True):
        for dt in (torch.float32, torch.bfloat16, torch.float16):
            h, p = torch.from_numpy(heat).cuda().to(dt), torch.from_numpy(paf).cuda().to(dt)
            for src in ("device", "host"):
                x, y = (h, p) if src == "device" else (h.cpu(), p.cpu())
                k0 = pp.kernel_launches()
                pp.run(x, y, frontend=frontend, materialize=mat and src == "device")
                pp.results()
                out[f"{frontend}/{mat}/{str(dt)[6:]}/{src}"] = pp.kernel_launches() - k0
assert pp.graph_launches() == 0
print(json.dumps(out))
"""


def test_a_16bit_batch_launches_one_kernel_more(ek, pair):
    env = dict(os.environ, EKP_GRAPHS="0", PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    run = subprocess.run([sys.executable, "-c", _LAUNCH_SCRIPT], capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert run.returncode == 0, run.stderr[-2000:]
    import json
    counts = json.loads(run.stdout.strip().splitlines()[-1])
    for key, k in counts.items():
        frontend, mat, dt, src = key.split("/")
        if dt != "float32":
            assert k == counts[f"{frontend}/{mat}/float32/{src}"] + 1, (key, counts)
    # the same count with graphs on: the captured graph holds the widening kernel too
    heat, paf = _batch(4, 46, 54, (2, 4), 53)
    b = pair[1]
    for dt in (torch.float32, torch.bfloat16):
        ks = []
        for rep in range(2):
            k0 = b.kernel_launches()
            b.run(_dev16(heat, dt), _dev16(paf, dt), frontend="reference")
            ks.append(b.kernel_launches() - k0)
        assert ks[0] == ks[1] == counts[f"reference/False/{str(dt)[6:]}/device"], (dt, ks)


# 8. streams --------------------------------------------------------------------------------------------------------
def test_16bit_run_on_a_side_stream(pair):
    heat, paf = _batch(8, 46, 54, (1, 6), 54)
    a, b = pair
    a.run(_dev16(heat, torch.bfloat16).float(), _dev16(paf, torch.bfloat16).float(), frontend="dense")
    want = _outputs(a)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        h = torch.empty(heat.shape, dtype=torch.bfloat16, device="cuda")
        p = torch.empty(paf.shape, dtype=torch.bfloat16, device="cuda")
        h.copy_(torch.from_numpy(heat).pin_memory(), non_blocking=True)   # written on s, read on s
        p.copy_(torch.from_numpy(paf).pin_memory(), non_blocking=True)
        b.run(h, p, frontend="dense")
    _assert_same(want, _outputs(b), "side stream")


# 9. the hand-off from the network -----------------------------------------------------------------------------------
def _humans_equal(x, y):
    assert len(x) == len(y)
    for hx, hy in zip(x, y):
        assert np.float32(hx.score) == np.float32(hy.score)
        assert sorted(hx.body_parts) == sorted(hy.body_parts)
        for k, bx in hx.body_parts.items():
            by = hy.body_parts[k]
            assert (bx.uidx, bx.part_idx, bx.x, bx.y, np.float32(bx.score)) == (by.uidx, by.part_idx, by.x, by.y, np.float32(by.score))


def test_autocast_outputs_through_infer_humans(ek):
    from torch_ekpose_b200 import estimator
    heat, paf = _batch(3, 46, 54, (2, 4), 21)

    class FakeNet(torch.nn.Module):
        """bf16 outputs as under autocast, or their .float()"""
        def __init__(self, widened):
            super().__init__()
            self.widened = widened

        def forward(self, x):
            h16, p16 = torch.from_numpy(heat).to(x.device).to(torch.bfloat16), torch.from_numpy(paf).to(x.device).to(torch.bfloat16)
            return ((p16.float(), h16.float()) if self.widened else (p16, h16)), None

    frames = [np.zeros((368, 432, 3), np.uint8) for _ in range(3)]
    got16 = estimator.infer_humans(frames, FakeNet(False), "vgg", torch.device("cuda", 0))
    got32 = estimator.infer_humans(frames, FakeNet(True), "vgg", torch.device("cuda", 0))
    assert sum(len(g) for g in got32) > 0
    for a, b in zip(got16, got32):
        _humans_equal(a, b)


# 10. growth, sharding: 16-bit tensors are forwarded as they are ------------------------------------------------------
def test_growth_with_a_crowded_bf16_batch(ek):
    from torch_ekpose_b200 import paf_to_pose
    heat, paf = _batch(1, 92, 164, (35, 35), 9)
    h16, p16 = _dev16(heat, torch.bfloat16), _dev16(paf, torch.bfloat16)
    small = dict(frontend="reference", max_peaks=256, max_humans=8, max_part=8, max_cand=64)
    paf_to_pose._cache.clear()
    want = ek.postprocess_batch(h16.float(), p16.float(), **small)
    paf_to_pose._cache.clear()
    got = ek.postprocess_batch(h16, p16, **small)
    grown = paf_to_pose._cache[(0,)]
    assert grown.max_part > 8 and grown.max_humans > 8
    paf_to_pose._cache.clear()
    assert len(want[0]) >= 30
    _humans_equal(want[0], got[0])
    # the host path of postprocess_batch with CPU bf16 tensors
    got_host = ek.postprocess_batch(h16.cpu(), p16.cpu(), **small)
    paf_to_pose._cache.clear()
    _humans_equal(want[0], got_host[0])


def test_sharded_bf16_equals_float32(ek):
    from torch_ekpose_b200 import sharding
    heat, paf = _batch(5, 46, 54, (1, 6), 55)
    h16, p16 = torch.from_numpy(heat).to(torch.bfloat16), torch.from_numpy(paf).to(torch.bfloat16)
    n32, s32 = sharding.postprocess_sharded(h16.float(), p16.float(), frontend="reference")
    n16, s16 = sharding.postprocess_sharded(h16, p16, frontend="reference")
    assert np.array_equal(n32, n16) and n32.sum() > 0
    assert_bits_equal(s32, s16, "sharded subset")
