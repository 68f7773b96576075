"""Batched, on-device hand-off from the network to the post-processing (SURVEY.md 8f rows f1 and f4).

The reference's ``get_outputs`` (/root/reference/lib/evaluate/estimator.py:71-87) runs ONE image
(batch 1, :80): host-side ``padding`` (cv2 resize of the long side to 368 + zero padding to a
multiple of 8, :52-68) and normalisation (lib/datasets/preprocessing.py:16-43), a forward pass, then
both outputs are copied to the host and handed to the post-processing as NumPy HWC views (:85-86).

``get_outputs_batched`` keeps that function's geometry and arithmetic but runs it on the GPU for a
whole batch of equally sized frames: the raw uint8 frames are uploaded once, ``padding`` +
normalisation are ONE CUDA kernel (``ekp_preprocess``, bit-identical to cv2's 8-bit fixed-point
resize and the reference's float32 normalisation), the model runs one forward pass, and its outputs
stay on the device in the layout it emits (NCHW): no device-to-host copy, no transpose.
``infer_humans`` feeds them straight to the CUDA post-processing on the same device.  There is no
host implementation of any of this in the package; the model itself is the caller's (cuDNN through
PyTorch; out of scope).
"""
from __future__ import annotations

from typing import List, Sequence

import numpy as np

from .paf_to_pose import PostProcessor

_prep_ctx = {}
_pp_cache = {}
_last_pp = [None]


def _device_index(device) -> int:
    import torch
    dev = torch.device(device)
    if dev.type != "cuda":
        raise ValueError(f"the hand-off runs on a CUDA device, got {dev} (there is no CPU path)")
    return dev.index if dev.index is not None else torch.cuda.current_device()


def get_outputs_batched(images, model, preprocess: str, device):
    """Batched ``get_outputs``: returns (pafs [n,38,h,w], heatmaps [n,19,h,w], im_scale) with the two
    tensors left on ``device``.  ``images``: a sequence of equally sized uint8 BGR frames [H,W,3]
    (frames of one stream) or one CUDA uint8 tensor [n,H,W,3] already on ``device``."""
    import torch
    idx = _device_index(device)
    dev = torch.device("cuda", idx)
    if isinstance(images, torch.Tensor):
        frames = images
        if not frames.is_cuda or frames.device.index != idx:
            frames = frames.to(dev, non_blocking=True)
    else:
        if len({im.shape for im in images}) != 1:
            raise ValueError("get_outputs_batched needs equally sized images (batch them per resolution)")
        frames = torch.from_numpy(np.stack(images)).to(dev, non_blocking=True)
    pp = _prep_ctx.get(idx)
    if pp is None:
        pp = _prep_ctx[idx] = PostProcessor(device=idx, max_batch=1, max_h=5, max_w=5, max_peaks=16, max_humans=4)
    with torch.cuda.device(dev):
        batch_var, scale = pp.preprocess(frames, mode=preprocess)
        with torch.no_grad():
            predicted, _ = model(batch_var)
    return predicted[-2], predicted[-1], scale


def infer_humans(images: Sequence[np.ndarray], model, preprocess: str, device, frontend: str = "reference",
                 thr: float = 0.15) -> List[list]:
    """images -> per-image list[Human]: GPU preprocessing, one forward pass, post-processing on the same GPU
    (the network's outputs never leave the device, and 16-bit outputs of a model under torch.autocast are taken as
    they are).  ``frontend='reference'`` gives the reference's people."""
    pafs, heats, _ = get_outputs_batched(images, model, preprocess, device)
    n, _, h, w = heats.shape
    idx = heats.device.index
    key = (idx, n, h, w)
    pp = _pp_cache.get(key)
    if pp is None:
        pp = _pp_cache[key] = PostProcessor(device=idx, max_batch=n, max_h=h, max_w=w, max_peaks=2048, max_humans=128)
    _last_pp[0] = pp
    pp.run(heats, pafs, layout="nchw", frontend=frontend, thr=thr)   # bf16 / fp16 under autocast: widened on the device
    return pp.humans()


def last_postprocessor():
    """The context the last ``infer_humans`` call used (stage timing in the benchmark)."""
    return _last_pp[0]
