"""Keypoints smoothed across video frames on the device (``ekp_smooth_humans``).

``Smoother`` keeps a One Euro filter (Casiez, Roussel, Vogel, CHI 2012) per track id, part and axis for ``n_seq``
sequences in a CUDA byte tensor it owns, and filters the keypoints of the ``result_tensors()`` tables under the ids a
``Tracker`` gave their rows.  One kernel per ``update``, asynchronous, no host wait.  The full specification is in
include/ekpose_b200.h ("smoothing").
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

from . import _lib
from .paf_to_pose import PostProcessor, _check_out, _torch_stream

try:  # as in paf_to_pose: the package (and its host surface) imports without torch; a Smoother needs it
    import torch
except Exception:  # pragma: no cover
    torch = None


class Smoother:
    """One Euro filters of ``n_seq`` sequences on ``device``, one per track id, part and axis.  ``update`` takes the
    tables of n = n_seq x F images and the track ids of their rows, image i being frame i % F of sequence i // F, as
    ``Tracker.update`` does; give it the ids of a ``Tracker`` with the same ``n_seq``, ``max_tracks`` and ``max_age``,
    and its filters live exactly as long as that tracker's tracks.

    The defaults ``min_cutoff=1.0``, ``beta=0.007``, ``d_cutoff=1.0`` (Hz) are the paper's demonstration values, not
    values tuned for pose.  ``beta`` scales with the coordinate unit: the coordinates here are map pixels, and a larger
    map wants a smaller ``beta`` for the same response.  Lower ``min_cutoff`` smooths more at rest; higher ``beta`` lags
    less in fast motion.  ``fps`` is the frame rate of the video: a part unseen for g frames is filtered with a time
    step of g / fps."""

    def __init__(self, device=0, n_seq: int = 1, max_tracks: int = 256, max_age: int = 30, fps: float = 30.0,
                 min_cutoff: float = 1.0, beta: float = 0.007, d_cutoff: float = 1.0):
        if torch is None:
            raise ImportError("Smoother needs torch (its state and outputs are CUDA tensors)")
        dev = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        if dev.type != "cuda":
            raise ValueError(f"the smoother runs on a CUDA device, got {dev} (there is no CPU path)")
        self.device = dev.index if dev.index is not None else torch.cuda.current_device()
        self.n_seq, self.max_tracks, self.max_age = int(n_seq), int(max_tracks), int(max_age)
        self.fps, self.min_cutoff, self.beta, self.d_cutoff = float(fps), float(min_cutoff), float(beta), float(d_cutoff)
        nbytes = int(_lib.lib.ekp_smooth_state_bytes(self.n_seq, self.max_tracks))
        if not nbytes:
            raise ValueError(f"n_seq {n_seq} >= 1 and max_tracks {max_tracks} in [1, {_lib.LIMIT_TRACKS}] required")
        # the context supplies the device, the error reporting and the launch count; it holds no smoothing state
        self._pp = PostProcessor(device=self.device, max_batch=1, max_h=5, max_w=5, max_peaks=16, max_humans=4)
        self.state = torch.empty(nbytes, dtype=torch.uint8, device=torch.device("cuda", self.device))
        self.reset()
        # the clear is queued on the current stream; waiting for it here lets the first update run on any stream
        torch.cuda.current_stream(self.device).synchronize()

    def reset(self, stream=None) -> None:
        """Forgets every filter and frame count.  Asynchronous on ``stream`` (default: the current stream), so an update
        on another stream must be ordered after it by the caller, as for any work on two streams."""
        _lib.check(_lib.lib.ekp_smooth_reset(self._pp._ctx, self.state.data_ptr(), self.n_seq, self.max_tracks,
                                             self._pp._stream(stream)))

    def update(self, tensors: dict, ids: torch.Tensor, stream=None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The smoothed keypoints of the people of ``tensors`` (a ``result_tensors()`` dict; ``num_humans`` and
        ``parts`` are read) under their track ``ids`` (int32 [n, max_humans], as ``Tracker.update`` returns them):
        float32 [n, max_humans, 18, 2] (x, y) on this smoother's device, map pixels.  Rows with a negative id keep their
        raw coordinates; absent parts and rows from ``num_humans[i]`` on are 0 (presence is ``parts[..., 3] >= 0``).
        One kernel on ``stream`` (default: the current stream), after whatever wrote the tables and ids on that stream;
        nothing waits for the device.  ``out=`` takes an earlier result to write into instead (ValueError if its shape,
        dtype, device or contiguity does not fit)."""
        dev = torch.device("cuda", self.device)
        num, parts = tensors["num_humans"], tensors["parts"]
        if not (isinstance(parts, torch.Tensor) and parts.dim() == 4 and tuple(parts.shape[2:]) == (_lib.NUM_PART, 4)):
            raise ValueError("tensors['parts'] must be an int32 tensor [n, max_humans, 18, 4]")
        n, mh = int(parts.shape[0]), int(parts.shape[1])
        _check_out(parts, "tensors['parts']", (n, mh, _lib.NUM_PART, 4), torch.int32, dev)
        _check_out(num, "tensors['num_humans']", (n,), torch.int32, dev)
        _check_out(ids, "ids", (n, mh), torch.int32, dev)
        if out is None:
            st = _torch_stream(dev, stream)
            with torch.cuda.device(dev), torch.cuda.stream(st):
                out = torch.empty((n, mh, _lib.NUM_PART, 2), dtype=torch.float32, device=dev)
            stream = st
        else:
            _check_out(out, "out", (n, mh, _lib.NUM_PART, 2), torch.float32, dev)
        _lib.check(_lib.lib.ekp_smooth_humans(self._pp._ctx, num.data_ptr(), parts.data_ptr(), ids.data_ptr(), n, mh,
                                              self.state.data_ptr(), self.n_seq, self.max_tracks, self.max_age,
                                              C.c_double(self.fps), C.c_double(self.min_cutoff), C.c_double(self.beta),
                                              C.c_double(self.d_cutoff), out.data_ptr(), self._pp._stream(stream)))
        return out

    def kernel_launches(self) -> int:
        """Kernels the smoother has launched (one per ``update``)."""
        return self._pp.kernel_launches()

    def close(self) -> None:
        self._pp.close()
