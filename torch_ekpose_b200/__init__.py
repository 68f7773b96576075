"""torch_ekpose_b200 -- B200-native PAF post-processing for torch_ekpose.

One hot path, nothing else: the part-affinity-field post-processing of
ek1den2/torch_ekpose (lib/pafprocess + the Python-side preprocessing in
lib/utils/paf_to_pose.py) as hand-written sm_100a CUDA kernels behind the reference's own
operator surface.  See DESIGN.md and INTEGRATION.md.

    from torch_ekpose_b200 import pafprocess          # drop-in for lib.pafprocess.pafprocess
    from torch_ekpose_b200 import paf_to_pose_cpp      # drop-in for lib.utils.paf_to_pose.paf_to_pose_cpp
    from torch_ekpose_b200 import PostProcessor, postprocess_batch   # batched device API
    from torch_ekpose_b200 import Tracker                            # stable person ids across video frames
    from torch_ekpose_b200 import Smoother                           # keypoints smoothed per track id (One Euro)
    from torch_ekpose_b200 import coco_eval                          # COCO keypoint AP on the device (COCOeval)

Importing the package loads libekpose_b200.so and fails loudly when it has not been built; there
is no CPU fallback.
"""
from . import _lib, coco_eval, pafprocess  # noqa: F401
from .common import BodyPart, CocoPairs, CocoPart, Human  # noqa: F401
from .config import cfg  # noqa: F401
from .paf_to_pose import NMS, PinnedBatch, PostProcessor, compute_resized_coords, find_peaks, paf_to_pose_cpp, postprocess_batch  # noqa: F401
from .smoothing import Smoother  # noqa: F401
from .tracking import Tracker  # noqa: F401

__all__ = ["pafprocess", "paf_to_pose_cpp", "NMS", "find_peaks", "compute_resized_coords", "PostProcessor", "PinnedBatch", "postprocess_batch", "Tracker", "Smoother", "Human", "BodyPart",
           "CocoPart", "CocoPairs", "cfg"]
