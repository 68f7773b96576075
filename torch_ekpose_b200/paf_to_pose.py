"""Host side of the post-processing path: the reference's ``paf_to_pose`` interface on top of
libekpose_b200.so.

Mirrors /root/reference/lib/utils/paf_to_pose.py for the functions the inference scripts call
(run_image.py:59, run_video.py:61, run_webcam.py:47, eval.py:156):

* ``paf_to_pose_cpp(heatmaps, pafs, config)`` (:346-380)  numpy HWC in, ``list[Human]`` out;
* ``NMS(heatmaps, upsampFactor, ..., config)``  (:60-133)  list of 18 ``[n_k, 4]`` arrays;

and adds the batched entry points the B200 path is built around:

* ``PostProcessor``      one context (= one GPU, one stream of work) with fixed-capacity buffers;
* ``postprocess_batch``  heat / PAF tensors of a whole batch (CUDA tensors as the network emits
                         them, or host arrays) -> per-image ``list[Human]``.

Everything numerical happens in the CUDA library; this module converts arguments and builds
``Human`` / ``BodyPart`` objects from the result tables.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np

from . import _lib
from .common import BodyPart, Human
from .config import cfg as default_cfg

try:  # torch is plumbing here (device memory and streams), not a requirement of the host path
    import torch
except Exception:  # pragma: no cover
    torch = None

_PEAK_DT = np.dtype([("x", np.int32), ("y", np.int32), ("score", np.float32), ("id", np.int32)])
_FRONTENDS = {"dense": _lib.FRONTEND_DENSE, "reference": _lib.FRONTEND_REFERENCE,
              "reference_coarse": _lib.FRONTEND_REFERENCE_COARSE, "reference_gauss": _lib.FRONTEND_REFERENCE_GAUSS}
_LAYOUTS = {"nchw": _lib.LAYOUT_NCHW, "nhwc": _lib.LAYOUT_NHWC}


def _is_tensor(x) -> bool:
    return torch is not None and isinstance(x, torch.Tensor)


def _dtype16(heat, paf) -> int:
    """The library's 16-bit dtype code when heat and paf are both bf16 / fp16 tensors, or both NumPy float16 arrays, of
    the same dtype; else 0 (EKP_DTYPE_F32: the float32 path, with a conversion for anything that is not float32)."""
    if _is_tensor(heat) and _is_tensor(paf) and heat.dtype == paf.dtype:
        return {torch.bfloat16: _lib.DTYPE_BF16, torch.float16: _lib.DTYPE_F16}.get(heat.dtype, 0)
    if isinstance(heat, np.ndarray) and isinstance(paf, np.ndarray) and heat.dtype == paf.dtype == np.float16:
        return _lib.DTYPE_F16
    return 0


def _torch_stream(dev, stream):
    """``stream`` (None: the current stream of ``dev``; a torch stream; or a raw cudaStream_t) as a torch stream, for
    allocating tensors under the stream that will use them."""
    if stream is None:
        return torch.cuda.current_stream(dev)
    if isinstance(stream, torch.cuda.Stream):
        return stream
    return torch.cuda.ExternalStream(int(getattr(stream, "cuda_stream", stream)), device=dev)


def _check_out(t, what: str, shape, dt, dev) -> None:
    """ValueError unless ``t`` is a contiguous ``dt`` tensor of ``shape`` on ``dev`` (the ``out=`` buffers)."""
    if not (_is_tensor(t) and t.device == dev and t.dtype == dt and tuple(t.shape) == tuple(shape) and t.is_contiguous()):
        raise ValueError(f"{what} must be a contiguous {dt} tensor {list(shape)} on {dev}")


class PostProcessor:
    """A libekpose_b200 context: stages 1-5 for batches of up to ``max_batch`` images.

    ``run`` is asynchronous on the current CUDA stream of ``device``; ``results`` / ``humans`` /
    ``peaks`` wait for it.  Inputs are float32, bfloat16 or float16 stride-8 maps, ``heat`` with 19 and
    ``paf`` with 38 channels, layout ``'nchw'`` (lib/network/vgg2016.py:105) or ``'nhwc'``
    (lib/evaluate/estimator.py:85-86).
    """

    def __init__(self, device: int = 0, max_batch: int = 64, max_h: int = 46, max_w: int = 54, max_peaks: int = 1024,
                 max_humans: int = 64, max_part: int = 0, max_cand: int = 0):
        """max_part / max_cand: peaks of one part / passing candidates of one limb per image (0 = the library
        defaults EKP_MAX_PART 256 / EKP_MAX_CAND 2048); a scene beyond any capacity raises EkpCapacityError."""
        self.device = int(device)
        self._ctx = C.c_void_p()
        _lib.check(_lib.lib.ekp_create_ex(C.byref(self._ctx), self.device, max_batch, max_h, max_w, max_peaks, max_humans,
                                          max_part, max_cand))
        self.max_batch, self.max_h, self.max_w = max_batch, max_h, max_w
        self.max_peaks, self.max_humans = max_peaks, max_humans
        self.max_part, self.max_cand = int(_lib.lib.ekp_max_part(self._ctx)), int(_lib.lib.ekp_max_cand(self._ctx))
        self.host_copy = True  # ekp_set_host_copy
        self._keep = None      # inputs of the in-flight run
        self._n = 0
        self._hw = (0, 0)
        self.heat_mat = None   # operator-surface tensors of the last materialising device run
        self.paf_mat = None

    def close(self):
        if getattr(self, "_ctx", None) and self._ctx.value:
            _lib.lib.ekp_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------------------------------
    def _stream(self, stream) -> int:
        if stream is not None:
            return int(getattr(stream, "cuda_stream", stream))
        if torch is not None and torch.cuda.is_available():
            return int(torch.cuda.current_stream(self.device).cuda_stream)
        return 0

    def _dims(self, heat_shape, paf_shape, layout):
        if len(heat_shape) != 4 or len(paf_shape) != 4:
            raise ValueError(f"heat / paf must be 4-D, got {tuple(heat_shape)} / {tuple(paf_shape)}")
        if layout == "nchw":
            n, ch, h, w = heat_shape
            pn, pc, ph, pw = paf_shape
        elif layout == "nhwc":
            n, h, w, ch = heat_shape
            pn, ph, pw, pc = paf_shape
        else:
            raise ValueError("layout must be 'nchw' or 'nhwc'")
        if ch != _lib.HEAT_CH or pc != _lib.PAF_CH or (pn, ph, pw) != (n, h, w):
            raise ValueError(f"expected heat with 19 and paf with 38 channels of equal batch/size, got "
                             f"{tuple(heat_shape)} / {tuple(paf_shape)} ({layout})")
        return int(n), int(h), int(w)

    def run(self, heat, paf, *, layout: str = "nchw", frontend: str = "reference", thr: float = 0.15,
            materialize: bool = False, stream=None) -> None:
        """Submit one batch (n <= max_batch).  CUDA tensors take the device entry point; NumPy
        arrays / CPU tensors take the host entry point (H2D copies on the same stream).
        heat and paf of the same 16-bit dtype (torch.bfloat16 / torch.float16 tensors, NumPy float16 arrays: what a
        network returns under torch.autocast) are handed over as they are and widened to float32 on the device, which
        gives exactly the results of their .float(); on the host entry only half the bytes cross the bus.  Any other
        dtype (mixed, float64, ...) is converted to float32 here.
        frontend: 'reference' (default: the reference's own stride-8 NMS + bicubic refinement, i.e. the people
        paf_to_pose_cpp returns), 'dense' (the north_star formulation), 'reference_coarse' (NMS(bool_refine_center=False))
        or 'reference_gauss' (NMS(bool_gaussian_filt=True))."""
        if frontend not in _FRONTENDS:
            raise ValueError("frontend must be 'dense', 'reference', 'reference_coarse' or 'reference_gauss'")
        n, h, w = self._dims(heat.shape, paf.shape, layout)
        st = self._stream(stream)
        thr = float(np.float32(thr))
        if _is_tensor(heat) and heat.is_cuda:
            if not (_is_tensor(paf) and paf.is_cuda and paf.device == heat.device):
                raise ValueError("heat and paf must live on the same device")
            if heat.device.index != self.device:
                raise ValueError(f"tensors are on cuda:{heat.device.index}, context on cuda:{self.device}")
            dtype = _dtype16(heat, paf)
            if dtype:
                heat, paf = heat.contiguous(), paf.contiguous()
            else:
                heat, paf = heat.contiguous().float(), paf.contiguous().float()
            hm = pm = None
            if materialize:
                H, W = 8 * h, 8 * w
                if self.paf_mat is None or self.paf_mat.shape != (n, H, W, _lib.PAF_CH):
                    self.heat_mat = torch.empty((n, H, W, _lib.HEAT_CH), dtype=torch.float32, device=heat.device)
                    self.paf_mat = torch.empty((n, H, W, _lib.PAF_CH), dtype=torch.float32, device=heat.device)
                hm, pm = self.heat_mat.data_ptr(), self.paf_mat.data_ptr()
            rc = _lib.lib.ekp_postprocess_typed(self._ctx, heat.data_ptr(), paf.data_ptr(), dtype, n, h, w, _LAYOUTS[layout],
                                                thr, _FRONTENDS[frontend], hm, pm, st)
            self._keep = (heat, paf)
        else:
            dtype = _dtype16(heat, paf)
            if _is_tensor(heat):
                heat_p, paf_p = (heat.contiguous(), paf.contiguous()) if dtype else (heat.contiguous().float(), paf.contiguous().float())
                ptrs = (heat_p.data_ptr(), paf_p.data_ptr())
            else:
                want = np.float16 if dtype else np.float32
                heat_p = np.ascontiguousarray(heat, want)
                paf_p = np.ascontiguousarray(paf, want)
                ptrs = (heat_p.ctypes.data, paf_p.ctypes.data)
            rc = _lib.lib.ekp_postprocess_host_typed(self._ctx, ptrs[0], ptrs[1], dtype, n, h, w, _LAYOUTS[layout], thr,
                                                     _FRONTENDS[frontend], int(bool(materialize)), st)
            self._keep = (heat_p, paf_p)
        _lib.check(rc)
        self._n, self._hw = n, (h, w)

    def run_peaks(self, peaks, n_peaks, paf_mat, h1: int, stream=None) -> None:
        """Stages 4-5 only on DEVICE tensors: peaks float32 [n, stride, 5], n_peaks int32 [n],
        paf_mat float32 [n, H, W, C] (the reference's process_paf arguments, batched)."""
        n, stride, five = peaks.shape
        if five != 5 or paf_mat.dim() != 4 or paf_mat.shape[0] != n:
            raise ValueError("peaks must be [n, stride, 5] and paf_mat [n, H, W, C]")
        peaks, paf_mat = peaks.contiguous().float(), paf_mat.contiguous().float()
        n_peaks = n_peaks.contiguous().to(torch.int32)
        _, H, W, Cc = paf_mat.shape
        _lib.check(_lib.lib.ekp_process_paf_dev(self._ctx, peaks.data_ptr(), n_peaks.data_ptr(), stride, n, int(h1),
                                                paf_mat.data_ptr(), H, W, Cc, self._stream(stream)))
        self._keep = (peaks, n_peaks, paf_mat)
        self._n, self._hw = n, (H // 8, W // 8)

    # ------------------------------------------------------------------------------------------
    def _rows(self) -> int:
        """Images the library will write results for (its own count of the last run, so that the arrays handed to
        it can never be too small, whoever submitted that run)."""
        return int(_lib.lib.ekp_last_batch(self._ctx))

    def results(self, with_peaks: bool = False, raise_on_overflow: bool = True) -> dict:
        """Wait and return numpy tables: num_humans [n], subset [n, max_humans, 20] (float32, the
        reference's rows), n_peaks [n], overflow [n] and optionally peaks [n, max_peaks]
        (structured x, y, score, id) + part_off [n, 19]."""
        n = self._rows()
        num = np.zeros(n, np.int32)
        npk = np.zeros(n, np.int32)
        ovf = np.zeros(n, np.uint32)
        subset = np.zeros((n, self.max_humans, 20), np.float32)
        line = np.zeros((n, self.max_peaks), _PEAK_DT) if with_peaks else None
        rc = _lib.lib.ekp_results(self._ctx, num.ctypes.data, subset.ctypes.data, npk.ctypes.data,
                                  line.ctypes.data if with_peaks else None, ovf.ctypes.data)
        if rc != _lib.ERR_CAPACITY or raise_on_overflow:   # the tables are written either way; `overflow` says what was cut
            _lib.check(rc)
        out = dict(num_humans=num, subset=subset, n_peaks=npk, overflow=ovf)
        if with_peaks:
            po = np.zeros((n, 19), np.int32)
            _lib.check(_lib.lib.ekp_results_parts(self._ctx, po.ctypes.data))
            out["peaks"] = line
            out["part_off"] = po
        return out

    def human_tables(self):
        """(num_humans [n], parts [n, max_humans, 18] structured (x, y, score, id; id -1 = absent),
        scores [n, max_humans]) -- the whole getter loop of paf_to_pose_cpp in three arrays."""
        n = self._rows()
        num = np.zeros(n, np.int32)
        parts = np.zeros((n, self.max_humans, _lib.NUM_PART), _PEAK_DT)
        scores = np.zeros((n, self.max_humans), np.float32)
        _lib.check(_lib.lib.ekp_results_humans(self._ctx, num.ctypes.data, parts.ctypes.data, scores.ctypes.data, None))
        return num, parts, scores

    def set_host_copy(self, enable: bool) -> None:
        """Whether the batches submitted from now on end with the device-to-host copy of their result records (the
        default: on).  Off suits a caller who reads the results only on the device (``result_tensors``,
        ``draw_humans``) and saves the copy on every batch; ``results`` / ``human_tables`` / ``humans`` still work
        after such a run (the first of them downloads the records)."""
        _lib.check(_lib.lib.ekp_set_host_copy(self._ctx, int(bool(enable))))
        self.host_copy = bool(enable)

    def _result_specs(self, n: int, subset: bool, peaks: bool):
        mh = self.max_humans
        specs = [("num_humans", (n,), torch.int32), ("overflow", (n,), torch.int32), ("n_peaks", (n,), torch.int32),
                 ("parts", (n, mh, _lib.NUM_PART, 4), torch.int32), ("scores", (n, mh), torch.float32)]
        if subset:
            specs.append(("subset", (n, mh, _lib.SUBSET_COLS), torch.float32))
        if peaks:
            specs += [("peaks", (n, self.max_peaks, 4), torch.int32), ("part_off", (n, _lib.NUM_PART + 1), torch.int32)]
        return specs

    def result_tensors(self, *, subset: bool = False, peaks: bool = False, out: Optional[dict] = None, stream=None) -> dict:
        """The tables of the last run as CUDA tensors on this context's device, without waiting for the device: the
        export is one kernel on ``stream`` (default: the current stream), ordered after the run and before this
        context's next run on any stream.

        Returns a dict of ``num_humans`` int32 [n], ``overflow`` int32 [n] (EKP_OVF_* bits), ``n_peaks`` int32 [n],
        ``parts`` int32 [n, max_humans, 18, 4] (x, y, score bits, id; id -1 = absent, as ``human_tables``),
        ``part_score`` float32 [n, max_humans, 18] (the view ``parts[..., 2].view(torch.float32)``), ``scores``
        float32 [n, max_humans] and, with ``subset=True``, ``subset`` float32 [n, max_humans, 20] (as ``results``).
        ``peaks=True`` adds the part-sorted peak table of ``results(with_peaks=True)``: ``peaks`` int32
        [n, max_peaks, 4] (x, y, score bits, id), its ``peak_score`` float32 view and ``part_off`` int32 [n, 19].
        Rows from ``num_humans[i]`` (people) and ``n_peaks[i]`` (peaks) on are zero, so each tensor copied to the host
        equals the host table byte for byte.

        This never raises on a capacity overflow (nothing is known about it when the call returns): the caller checks
        ``overflow``, where a non-zero entry means that image's tables were cut.  New tensors are allocated under the
        export's stream; ``out=`` takes the dict of an earlier call and writes into its tensors instead (ValueError if
        their shape, dtype, device or contiguity does not fit this run), e.g. to keep a ring of buffers with no
        allocation per batch."""
        n = self._rows()
        if not n:
            raise _lib.EkpError(_lib.ERR_STATE, "result_tensors: no run has been submitted on this context")
        dev = torch.device("cuda", self.device)
        specs = self._result_specs(n, subset, peaks)
        if out is None:
            stream = _torch_stream(dev, stream)
            with torch.cuda.device(dev), torch.cuda.stream(stream):
                out = {name: torch.empty(shape, dtype=dt, device=dev) for name, shape, dt in specs}
        else:
            for name, shape, dt in specs:
                _check_out(out.get(name) if isinstance(out, dict) else None, f"out[{name!r}]", shape, dt, dev)
        tabs = _lib.DeviceResults(*(out[k].data_ptr() if k in out and (k != "subset" or subset) else None
                                    for k in ("num_humans", "overflow", "n_peaks", "subset", "parts", "scores")))
        st = self._stream(stream)
        _lib.check(_lib.lib.ekp_results_device(self._ctx, n, C.byref(tabs), st))
        out["part_score"] = out["parts"][..., 2].view(torch.float32)
        if peaks:   # n_peaks came with the people
            pk = _lib.DevicePeaks(None, out["peaks"].data_ptr(), out["part_off"].data_ptr())
            _lib.check(_lib.lib.ekp_results_device_peaks(self._ctx, n, C.byref(pk), st))
            out["peak_score"] = out["peaks"][..., 2].view(torch.float32)
        return out

    def humans(self) -> List[List[Human]]:
        """Per image the list[Human] the reference builds at paf_to_pose.py:361-378."""
        num, parts, scores = self.human_tables()
        h, w = self._hw
        H, W = 8 * h, 8 * w
        out = []
        for i in range(len(num)):
            humans = []
            for k in range(int(num[i])):
                human = Human([])
                row = parts[i, k]
                for part_idx in np.nonzero(row["id"] >= 0)[0]:
                    p = row[part_idx]
                    human.body_parts[int(part_idx)] = BodyPart("%d-%d" % (k, part_idx), int(part_idx),
                                                               float(p["x"]) / W, float(p["y"]) / H, float(p["score"]))
                if human.body_parts:
                    human.score = float(scores[i, k])
                    humans.append(human)
            out.append(humans)
        return out

    def draw_humans(self, frames, stream=None):
        """Paints the people of the last run onto ``frames``, a contiguous CUDA uint8 tensor [n, H, W, 3] on this
        context's device with one frame per image of the run, in place, and returns it: byte for byte what the
        reference's ``draw_humans(frame, humans)`` (lib/utils/common.py:252-275, imgcopy=False) paints with the
        people ``humans()`` returns.  Frames of any size work (coordinates are normalised by the run's map, as in
        the reference).  Asynchronous on ``stream`` (default: the current stream), ordered after the run."""
        if not (_is_tensor(frames) and frames.is_cuda and frames.dtype == torch.uint8 and frames.dim() == 4 and
                frames.shape[3] == 3 and frames.is_contiguous()):
            raise ValueError("frames must be a contiguous CUDA uint8 tensor [n, H, W, 3]")
        if frames.device.index != self.device:
            raise ValueError(f"frames are on cuda:{frames.device.index}, context on cuda:{self.device}")
        n, H, W, _ = frames.shape
        rows = self._rows()
        if rows and n != rows:
            raise ValueError(f"{n} frames for a run of {rows} images")
        if not (1 <= H <= _lib.DRAW_MAX_SIDE and 1 <= W <= _lib.DRAW_MAX_SIDE):
            raise ValueError(f"frames of {H}x{W} outside [1x1, {_lib.DRAW_MAX_SIDE}x{_lib.DRAW_MAX_SIDE}]")
        _lib.check(_lib.lib.ekp_draw_humans(self._ctx, frames.data_ptr(), n, H, W, self._stream(stream)))
        return frames

    def set_timing(self, enable: bool) -> None:
        _lib.check(_lib.lib.ekp_set_timing(self._ctx, int(bool(enable))))

    def stage_times(self):
        """Mean device milliseconds per stage over the recorded runs: dict + number of runs."""
        ms = (C.c_float * 4)()
        runs = C.c_int(0)
        _lib.check(_lib.lib.ekp_stage_times(self._ctx, ms, C.byref(runs)))
        return dict(frontend=ms[0], peak_sort=ms[1], connect=ms[2], assemble=ms[3]), runs.value

    def preprocess(self, frames, mode: str = "vgg", dest_size: int = 368, factor: int = 8, stream=None):
        """Input side (row f4): uint8 BGR frames [n, H, W, 3] as a CUDA tensor -> the network input
        float32 [n, 3, padded_h, padded_w] on the same device, bit-identical to the reference's
        padding() + vgg_preprocess()/rtpose_preprocess() (estimator.py:52-68, preprocessing.py:16-43).
        Returns (tensor, im_scale)."""
        if not (_is_tensor(frames) and frames.is_cuda and frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[3] == 3):
            raise ValueError("frames must be a CUDA uint8 tensor [n, H, W, 3] (BGR)")
        frames = frames.contiguous()
        n, sh, sw, _ = frames.shape
        v = [C.c_int() for _ in range(4)]
        scale = C.c_double()
        _lib.check(_lib.lib.ekp_preprocess_dims(sh, sw, dest_size, factor, *[C.addressof(x) for x in v], C.addressof(scale)))
        out = torch.empty((n, 3, v[2].value, v[3].value), dtype=torch.float32, device=frames.device)
        _lib.check(_lib.lib.ekp_preprocess(self._ctx, frames.data_ptr(), n, sh, sw, dest_size, factor,
                                           {"vgg": 0, "rtpose": 1}[mode], out.data_ptr(), self._stream(stream)))
        return out, scale.value

    def kernel_launches(self) -> int:
        return int(_lib.lib.ekp_kernel_launches(self._ctx))

    def graph_launches(self) -> int:
        """Batches replayed as a CUDA graph (same pointers, shape and flags as an earlier batch)."""
        return int(_lib.lib.ekp_graph_launches(self._ctx))

    def dense_smooth(self, heat, layout: str = "nchw"):
        """Test hook: the dense front-end's smoothed map, CUDA tensor [n, 8h, 8w, 18]."""
        if layout == "nchw":
            n, _, h, w = heat.shape
        else:
            n, h, w, _ = heat.shape
        heat = heat.contiguous().float()
        out = torch.empty((n, 8 * h, 8 * w, _lib.NUM_PART), dtype=torch.float32, device=heat.device)
        _lib.check(_lib.lib.ekp_dense_smooth_debug(self._ctx, heat.data_ptr(), n, h, w, _LAYOUTS[layout], out.data_ptr(),
                                                   self._stream(None)))
        return out


class PinnedBatch:
    """One pinned host block holding a batch's heat tensor directly followed by its PAF tensor (NCHW or NHWC):
    ``PostProcessor.run(b.heat, b.paf, ...)`` then moves both with a single host-to-device copy.
    ``heat`` / ``paf`` are views to fill in place: NumPy arrays for ``dtype`` 'float32' and 'float16', torch.bfloat16
    CPU tensors for 'bfloat16' (NumPy has no bfloat16).  The 16-bit blocks are half the size and are widened to float32
    on the device."""

    _ITEMSIZE = {"float32": 4, "float16": 2, "bfloat16": 2}

    def __init__(self, n: int, h: int, w: int, layout: str = "nchw", write_combined: bool = False, dtype: str = "float32"):
        if dtype not in self._ITEMSIZE:
            raise ValueError("dtype must be 'float32', 'float16' or 'bfloat16'")
        if dtype == "bfloat16" and torch is None:
            raise ValueError("a bfloat16 PinnedBatch needs torch (NumPy has no bfloat16)")
        self._ptr = C.c_void_p()
        nh, npf = n * h * w * _lib.HEAT_CH, n * h * w * _lib.PAF_CH
        item = self._ITEMSIZE[dtype]
        _lib.check(_lib.lib.ekp_host_alloc(C.byref(self._ptr), item * (nh + npf), int(bool(write_combined))))
        buf = (C.c_uint8 * (item * (nh + npf))).from_address(self._ptr.value)
        if dtype == "bfloat16":
            flat = torch.frombuffer(buf, dtype=torch.bfloat16)
        else:
            flat = np.frombuffer(buf, dtype=np.float32 if dtype == "float32" else np.float16)
        shp = (lambda c: (n, c, h, w)) if layout == "nchw" else (lambda c: (n, h, w, c))
        self.heat = flat[:nh].reshape(shp(_lib.HEAT_CH))
        self.paf = flat[nh:].reshape(shp(_lib.PAF_CH))
        self.dtype = dtype
        self.nbytes = item * (nh + npf)

    def close(self):
        if getattr(self, "_ptr", None) and self._ptr.value:
            self.heat = self.paf = None
            _lib.lib.ekp_host_free(self._ptr)
            self._ptr = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- module-level convenience API ---------------------------------------------------------------
_cache: dict = {}


def _default_device() -> int:
    """EKP_DEVICE (the same variable the C operator surface reads) or 0."""
    import os
    return int(os.environ.get("EKP_DEVICE", "0"))


def _processor(device: int, n: int, h: int, w: int, max_peaks: int, max_humans: int, max_part: int = 0, max_cand: int = 0) -> PostProcessor:
    """The cached context of ``device``, re-created (new one first, then the old one closed) when a dimension or a
    capacity is too small; a failed creation leaves no stale entry behind."""
    key = (device,)
    pp = _cache.get(key)
    want_part, want_cand = max_part or _lib.MAX_PART, max_cand or _lib.MAX_CAND
    if pp is not None and pp.max_batch >= n and pp.max_h >= h and pp.max_w >= w and pp.max_peaks >= max_peaks and \
            pp.max_humans >= max_humans and pp.max_part >= want_part and pp.max_cand >= want_cand:
        return pp
    if pp is not None:
        max_peaks, max_humans = max(max_peaks, pp.max_peaks), max(max_humans, pp.max_humans)
        want_part, want_cand = max(want_part, pp.max_part), max(want_cand, pp.max_cand)
        n, h, w = max(n, pp.max_batch), max(h, pp.max_h), max(w, pp.max_w)
    try:
        new = PostProcessor(device, n, h, w, max_peaks, max_humans, want_part, want_cand)
    except Exception:
        _cache.pop(key, None)
        if pp is not None:
            pp.close()
        raise
    if pp is not None:
        new.set_host_copy(pp.host_copy)   # the grown context keeps the caller's mode
        pp.close()
    _cache[key] = new
    return new


def _grow(pp: PostProcessor, bits: int):
    """Capacities for a retry after the overflow ``bits``: only what overflowed grows (x4), clamped to the library's
    limits; None when nothing that overflowed can still grow."""
    caps = dict(max_peaks=pp.max_peaks, max_humans=pp.max_humans, max_part=pp.max_part, max_cand=pp.max_cand)
    lim = dict(max_peaks=_lib.LIMIT_PEAKS, max_humans=_lib.LIMIT_HUMANS, max_part=_lib.LIMIT_PART, max_cand=_lib.LIMIT_CAND)
    grew = False
    for bit, name in ((_lib.OVF_PEAKS, "max_peaks"), (_lib.OVF_HUMANS, "max_humans"), (_lib.OVF_PART, "max_part"),
                      (_lib.OVF_CANDIDATES, "max_cand")):
        if bits & bit:
            if caps[name] >= lim[name]:
                return None
            caps[name] = min(caps[name] * 4, lim[name])
            grew = True
    return caps if grew else None


def _run_growing(device, heat, paf, n, h, w, caps, fatal_bits, **run_kw) -> PostProcessor:
    """Run one batch on the cached context of ``device``, growing the capacities named by the overflow bits in
    ``fatal_bits`` until the batch fits (other bits are the caller's business)."""
    while True:
        pp = _processor(device, n, h, w, **caps)
        pp.run(heat, paf, **run_kw)
        res = pp.results(raise_on_overflow=False)
        bits = int(np.bitwise_or.reduce(res["overflow"])) if len(res["overflow"]) else 0
        if bits & _lib.OVF_BADPEAK:
            raise _lib.EkpError(_lib.ERR_ARG, "non-finite values in the input maps")
        if not bits & fatal_bits:
            return pp
        caps = _grow(pp, bits & fatal_bits)
        if caps is None:
            raise _lib.EkpCapacityError(_lib.ERR_CAPACITY, f"the batch exceeds the library's limits (overflow bits 0x{bits:x}: "
                                        f"peaks {_lib.LIMIT_PEAKS}, humans {_lib.LIMIT_HUMANS}, peaks per part {_lib.LIMIT_PART}, "
                                        f"candidates per limb {_lib.LIMIT_CAND})")


_ALL_OVF = _lib.OVF_PEAKS | _lib.OVF_PART | _lib.OVF_CANDIDATES | _lib.OVF_HUMANS


def postprocess_batch(heat, paf, *, layout: str = "nchw", frontend: str = "reference", thr: float = 0.15,
                      materialize: bool = False, max_peaks: int = 2048, max_humans: int = 128, max_part: int = 0,
                      max_cand: int = 0, device: Optional[int] = None) -> List[List[Human]]:
    """heat [n,19,h,w] / paf [n,38,h,w] (or NHWC) -> per-image list[Human].  CUDA tensors stay on their
    device; host arrays are copied to ``device`` (default EKP_DEVICE or 0).  The default front-end is the
    reference's own, so the people equal ``paf_to_pose_cpp``'s; ``frontend='dense'`` selects the north_star
    formulation.  A capacity overflow grows the capacity that overflowed (within the library's limits) and retries."""
    if device is None:
        device = heat.device.index if (_is_tensor(heat) and heat.is_cuda) else _default_device()
    shp = heat.shape
    n, h, w = (shp[0], shp[2], shp[3]) if layout == "nchw" else (shp[0], shp[1], shp[2])
    caps = dict(max_peaks=max_peaks, max_humans=max_humans, max_part=max_part, max_cand=max_cand)
    pp = _run_growing(device, heat, paf, int(n), int(h), int(w), caps, _ALL_OVF, layout=layout, frontend=frontend, thr=thr,
                      materialize=materialize)
    return pp.humans()


def paf_to_pose_cpp(heatmaps, pafs, config=None, *, frontend: str = "reference", device: Optional[int] = None) -> List[Human]:
    """Drop-in for paf_to_pose.py:346-380: one image, numpy HWC ``heatmaps[h,w,19]``,
    ``pafs[h,w,38]`` (the arrays estimator.get_outputs returns) -> ``list[Human]``.

    The default front-end is the reference's own (stride-8 NMS + bicubic refinement), so the
    people equal the reference's; ``frontend='dense'`` selects the north_star formulation.
    Transposed views of NCHW arrays (what get_outputs actually returns, estimator.py:85-86) are
    passed through without a host-side copy.
    """
    config = config or default_cfg
    if config.MODEL.NUM_KEYPOINTS != 18 or config.MODEL.DOWNSAMPLE != 8:
        raise ValueError("the CUDA path is built for NUM_KEYPOINTS=18, DOWNSAMPLE=8 (lib/config/default.py:16-17)")
    heatmaps = np.asarray(heatmaps)
    pafs = np.asarray(pafs)
    if heatmaps.ndim != 3 or pafs.ndim != 3:
        raise ValueError("heatmaps / pafs must be [h, w, C]")
    layout = "nhwc"
    hv, pv = heatmaps.transpose(2, 0, 1), pafs.transpose(2, 0, 1)
    if hv.flags.c_contiguous and pv.flags.c_contiguous and heatmaps.dtype == np.float32 and pafs.dtype == np.float32:
        heat4, paf4, layout = hv[None], pv[None], "nchw"   # a view of the network's CHW output: no copy
    else:
        heat4, paf4 = heatmaps[None], pafs[None]
    return postprocess_batch(heat4, paf4, layout=layout, frontend=frontend, thr=config.TEST.THRESH_HEATMAP, device=device)[0]


def compute_resized_coords(coords, resizeFactor):
    """paf_to_pose.py:39-57: index of a cell after resizing its array by resizeFactor, (c + 0.5) * f - 0.5."""
    return (np.array(coords, dtype=float) + 0.5) * resizeFactor - 0.5


def _peak_table(heat_hwc: np.ndarray, thr: float, frontend: str, device: Optional[int]):
    """Stages 1-3 of one map on the GPU: (line, part_off) of the part-sorted peak table in (part, y, x) order.  Only the
    peak table matters here: more peaks of one part than max_part (or whatever stages 4-5 ran into on an arbitrary
    map) does not cut it, more than max_peaks does -- that capacity grows."""
    h, w, _ = heat_hwc.shape
    device = _default_device() if device is None else device
    pp = _run_growing(device, heat_hwc[None], np.zeros((1, h, w, _lib.PAF_CH), np.float32), 1, h, w,
                      dict(max_peaks=2048, max_humans=128), _lib.OVF_PEAKS, layout="nhwc", frontend=frontend, thr=thr)
    res = pp.results(with_peaks=True, raise_on_overflow=False)
    return res["peaks"][0], res["part_off"][0]


def find_peaks(param, img, device: Optional[int] = None):
    """Drop-in for paf_to_pose.py:26-36: the local maxima (4-neighbour cross, in-bounds neighbours only) of a 2-D
    map that exceed ``param``, as an int array of [x, y] rows in row-major order.  Runs on the GPU (the map
    travels as part 0 of an otherwise empty heat tensor)."""
    img = np.asarray(img, np.float32)
    if img.ndim != 2:
        raise ValueError("img must be 2-D")
    h, w = img.shape
    if h < 5 or w < 5:
        raise ValueError("the CUDA path needs maps of at least 5 x 5")
    heat = np.full((h, w, _lib.HEAT_CH), -np.inf, np.float32)
    heat[:, :, 0] = img
    line, po = _peak_table(heat, float(param), "reference_coarse", device)
    rows = line[po[0]:po[1]]
    return np.stack([(rows["x"] - 3) // 8, (rows["y"] - 3) // 8], axis=1).astype(np.int64).reshape(-1, 2)


def NMS(heatmaps, upsampFactor=1., bool_refine_center=True, bool_gaussian_filt=False, config=None, device: Optional[int] = None):
    """Drop-in for paf_to_pose.py:60-133: list of 18 float64 arrays ``[n_k, 4]`` = (x, y, score, id).
    bool_refine_center=False returns the stride-8 maxima at compute_resized_coords(peak, 8) with the heat value
    as score (:119-122); bool_gaussian_filt=True smooths every upsampled patch with scipy's gaussian_filter(sigma=3)
    arithmetic before the arg-max (:111-112; it has no effect without refinement, as in the reference)."""
    config = config or default_cfg
    if int(upsampFactor) != 8 or float(upsampFactor) != 8.0:
        raise NotImplementedError("built: upsampFactor=8 (lib/config/default.py:17 MODEL.DOWNSAMPLE, the only value a caller passes)")
    heatmaps = np.ascontiguousarray(heatmaps, np.float32)
    h, w, _ = heatmaps.shape
    if not bool_refine_center:
        line, po = _peak_table(heatmaps, config.TEST.THRESH_HEATMAP, "reference_coarse", device)
        out = []
        for k in range(config.MODEL.NUM_KEYPOINTS):
            rows = line[po[k]:po[k + 1]]
            arr = np.zeros((len(rows), 4))
            arr[:, 0] = compute_resized_coords((rows["x"] - 3) // 8, 8)
            arr[:, 1] = compute_resized_coords((rows["y"] - 3) // 8, 8)
            arr[:, 2], arr[:, 3] = rows["score"], rows["id"]
            out.append(arr)
        return out
    line, po = _peak_table(heatmaps, config.TEST.THRESH_HEATMAP, "reference_gauss" if bool_gaussian_filt else "reference", device)
    out = []
    for k in range(config.MODEL.NUM_KEYPOINTS):
        rows = line[po[k]:po[k + 1]]
        arr = np.zeros((len(rows), 4))
        arr[:, 0], arr[:, 1], arr[:, 2], arr[:, 3] = rows["x"], rows["y"], rows["score"], rows["id"]
        out.append(arr)
    return out
