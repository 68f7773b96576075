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
``infer_humans`` feeds them straight to the CUDA post-processing on the same device, and
``infer_and_draw`` also paints the people onto the uploaded frames (``ekp_draw_humans``, byte for
byte the reference's ``draw_humans``), and ``infer_human_tensors`` returns the people as CUDA tensors
(``ekp_results_device``) without waiting for the device.  There is no host implementation of any of this in the
package; the model itself is the caller's (cuDNN through PyTorch; out of scope).
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


def _upload(images, idx: int):
    """The frames as a CUDA uint8 tensor [n,H,W,3] on cuda:``idx``: a CUDA tensor already there as it is, anything
    else copied there once."""
    import torch
    dev = torch.device("cuda", idx)
    if isinstance(images, torch.Tensor):
        frames = images
        if not frames.is_cuda or frames.device.index != idx:
            frames = frames.to(dev, non_blocking=True)
        return frames
    if len({im.shape for im in images}) != 1:
        raise ValueError("get_outputs_batched needs equally sized images (batch them per resolution)")
    return torch.from_numpy(np.stack(images)).to(dev, non_blocking=True)


def _forward(frames, model, preprocess: str, idx: int):
    import torch
    pp = _prep_ctx.get(idx)
    if pp is None:
        pp = _prep_ctx[idx] = PostProcessor(device=idx, max_batch=1, max_h=5, max_w=5, max_peaks=16, max_humans=4)
    with torch.cuda.device(idx):
        batch_var, scale = pp.preprocess(frames, mode=preprocess)
        with torch.no_grad():
            predicted, _ = model(batch_var)
    return predicted[-2], predicted[-1], scale


def get_outputs_batched(images, model, preprocess: str, device):
    """Batched ``get_outputs``: returns (pafs [n,38,h,w], heatmaps [n,19,h,w], im_scale) with the two
    tensors left on ``device``.  ``images``: a sequence of equally sized uint8 BGR frames [H,W,3]
    (frames of one stream) or one CUDA uint8 tensor [n,H,W,3] already on ``device``."""
    idx = _device_index(device)
    return _forward(_upload(images, idx), model, preprocess, idx)


def _postprocess(heats, pafs, frontend: str, thr: float) -> PostProcessor:
    n, _, h, w = heats.shape
    idx = heats.device.index
    key = (idx, n, h, w)
    pp = _pp_cache.get(key)
    if pp is None:
        pp = _pp_cache[key] = PostProcessor(device=idx, max_batch=n, max_h=h, max_w=w, max_peaks=2048, max_humans=128)
    _last_pp[0] = pp
    pp.run(heats, pafs, layout="nchw", frontend=frontend, thr=thr)   # bf16 / fp16 under autocast: widened on the device
    return pp


def infer_humans(images: Sequence[np.ndarray], model, preprocess: str, device, frontend: str = "reference",
                 thr: float = 0.15) -> List[list]:
    """images -> per-image list[Human]: GPU preprocessing, one forward pass, post-processing on the same GPU
    (the network's outputs never leave the device, and 16-bit outputs of a model under torch.autocast are taken as
    they are).  ``frontend='reference'`` gives the reference's people."""
    pafs, heats, _ = get_outputs_batched(images, model, preprocess, device)
    return _postprocess(heats, pafs, frontend, thr).humans()


def infer_human_tensors(images, model, preprocess: str, device, frontend: str = "reference", thr: float = 0.15,
                        subset: bool = False):
    """``infer_humans`` with the people left on the GPU: returns (tensors, im_scale), ``tensors`` being the dict of
    CUDA tensors ``PostProcessor.result_tensors(subset=subset)`` returns (per image num_humans, overflow, n_peaks,
    the part table, part and human scores) and ``im_scale`` that of ``get_outputs_batched``.  Nothing waits for the
    device and nothing raises on a capacity overflow: the caller checks ``tensors['overflow']``."""
    pafs, heats, im_scale = get_outputs_batched(images, model, preprocess, device)
    return _postprocess(heats, pafs, frontend, thr).result_tensors(subset=subset), im_scale


def infer_and_draw(images, model, preprocess: str, device, frontend: str = "reference", thr: float = 0.15):
    """``infer_humans`` followed by the reference's ``draw_humans`` on every frame, all on the GPU: returns the drawn
    frames, a CUDA uint8 tensor [n,H,W,3] on ``device``.  Host frames are drawn on the copy uploaded for the
    preprocessing; a CUDA tensor on ``device`` (contiguous) is drawn in place.  The people stay available through
    ``last_postprocessor()``; the call does not wait for the device."""
    idx = _device_index(device)
    frames = _upload(images, idx)
    pafs, heats, _ = _forward(frames, model, preprocess, idx)
    return _postprocess(heats, pafs, frontend, thr).draw_humans(frames)


def last_postprocessor():
    """The context the last ``infer_humans`` / ``infer_and_draw`` / ``infer_human_tensors`` call used (stage timing in the benchmark)."""
    return _last_pp[0]
