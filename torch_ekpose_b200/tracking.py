"""Stable person ids across video frames on the device (``ekp_track_humans``).

``Tracker`` keeps the tracks of ``n_seq`` sequences in a CUDA byte tensor it owns and gives every person row of the
``result_tensors()`` tables the id of the same person in earlier frames: COCO OKS similarity to each track's last pose,
greedy one-to-one matching, new ids for the unmatched, tracks dropped after ``max_age`` frames unseen.  One kernel per
``update``, asynchronous, no host wait.  The full specification is in include/ekpose_b200.h ("tracking").
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

from . import _lib
from .paf_to_pose import PostProcessor, _check_out, _torch_stream

try:  # as in paf_to_pose: the package (and its host surface) imports without torch; a Tracker needs it
    import torch
except Exception:  # pragma: no cover
    torch = None


class Tracker:
    """Tracks of ``n_seq`` sequences on ``device``.  ``update`` takes the tables of n = n_seq x F images, image i being
    frame i % F of sequence i // F (``n_seq=1``: consecutive frames of one video; F = 1: one frame of each of
    ``n_seq`` cameras), and may be called with a different F each time: the tracks carry over."""

    def __init__(self, device=0, n_seq: int = 1, max_tracks: int = 256, min_oks: float = 0.5, max_age: int = 30):
        if torch is None:
            raise ImportError("Tracker needs torch (its state and outputs are CUDA tensors)")
        dev = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        if dev.type != "cuda":
            raise ValueError(f"the tracker runs on a CUDA device, got {dev} (there is no CPU path)")
        self.device = dev.index if dev.index is not None else torch.cuda.current_device()
        self.n_seq, self.max_tracks, self.min_oks, self.max_age = int(n_seq), int(max_tracks), float(min_oks), int(max_age)
        nbytes = int(_lib.lib.ekp_track_state_bytes(self.n_seq, self.max_tracks))
        if not nbytes:
            raise ValueError(f"n_seq {n_seq} >= 1 and max_tracks {max_tracks} in [1, {_lib.LIMIT_TRACKS}] required")
        # the context supplies the device, the error reporting and the launch count; it holds no tracking state
        self._pp = PostProcessor(device=self.device, max_batch=1, max_h=5, max_w=5, max_peaks=16, max_humans=4)
        self.state = torch.empty(nbytes, dtype=torch.uint8, device=torch.device("cuda", self.device))
        self.reset()
        # the clear is queued on the current stream; waiting for it here lets the first update run on any stream
        torch.cuda.current_stream(self.device).synchronize()

    def reset(self, stream=None) -> None:
        """Forgets every track: ids start again from 0.  Asynchronous on ``stream`` (default: the current stream), so
        an update on another stream must be ordered after it by the caller, as for any work on two streams."""
        _lib.check(_lib.lib.ekp_track_reset(self._pp._ctx, self.state.data_ptr(), self.n_seq, self.max_tracks,
                                            self._pp._stream(stream)))

    def update(self, tensors: dict, stream=None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The track ids of the people of ``tensors`` (a ``result_tensors()`` dict; ``num_humans`` and ``parts`` are
        read): int32 [n, max_humans] on this tracker's device, -1 from row ``num_humans[i]`` on.  One kernel on
        ``stream`` (default: the current stream), after whatever wrote the tables on that stream; nothing waits for the
        device.  ``out=`` takes an earlier result to write into instead (ValueError if its shape, dtype, device or
        contiguity does not fit)."""
        dev = torch.device("cuda", self.device)
        num, parts = tensors["num_humans"], tensors["parts"]
        if not (isinstance(parts, torch.Tensor) and parts.dim() == 4 and tuple(parts.shape[2:]) == (_lib.NUM_PART, 4)):
            raise ValueError("tensors['parts'] must be an int32 tensor [n, max_humans, 18, 4]")
        n, mh = int(parts.shape[0]), int(parts.shape[1])
        _check_out(parts, "tensors['parts']", (n, mh, _lib.NUM_PART, 4), torch.int32, dev)
        _check_out(num, "tensors['num_humans']", (n,), torch.int32, dev)
        if out is None:
            st = _torch_stream(dev, stream)
            with torch.cuda.device(dev), torch.cuda.stream(st):
                out = torch.empty((n, mh), dtype=torch.int32, device=dev)
            stream = st
        else:
            _check_out(out, "out", (n, mh), torch.int32, dev)
        _lib.check(_lib.lib.ekp_track_humans(self._pp._ctx, num.data_ptr(), parts.data_ptr(), n, mh, self.state.data_ptr(),
                                             self.n_seq, self.max_tracks, C.c_float(self.min_oks), self.max_age,
                                             out.data_ptr(), self._pp._stream(stream)))
        return out

    def kernel_launches(self) -> int:
        """Kernels the tracker has launched (one per ``update``)."""
        return self._pp.kernel_launches()

    def close(self) -> None:
        self._pp.close()
