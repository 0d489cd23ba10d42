"""hpdecode -- B200-native (sm_100a) HigherHRNet bottom-up keypoint decoding.

Drop-in for the decode path of thawro/pytorch-human-pose (src/keypoints grouping / results /
model flip logic).  All compute runs in libhpdecode.so (hand-written CUDA, C ABI in
include/hpdecode.h); importing this package registers the ``torch.ops.hpd.*`` custom ops.
There is no CPU or eager-PyTorch fallback: ops raise if the library or a CUDA device is missing.
"""
from . import _lib, ops  # noqa: F401  (registers torch.ops.hpd.*)
from . import geometry  # noqa: F401
from .decoder import BottomUpDecoder, DecodePipeline, DecodeResult, Records  # noqa: F401
from .grouping import MPPEHeatmapParser  # noqa: F401
from .results import BaseKeypointsResult, InferenceKeypointsResult, KeypointsResult  # noqa: F401
from .model import InferenceKeypointsModel  # noqa: F401
from .stream import FrameStream  # noqa: F401
from .track import OneEuro, PoseTracker  # noqa: F401
from .render import PoseRenderer, PoseStyle  # noqa: F401
from .coco import batch_to_coco, eval_coco, evaluate_dataset_batched, result_to_coco  # noqa: F401
from .cocoeval import KeypointEvaluator, KeypointGroundTruth  # noqa: F401

__all__ = ["BottomUpDecoder", "DecodePipeline", "DecodeResult", "Records", "MPPEHeatmapParser", "BaseKeypointsResult",
           "InferenceKeypointsResult", "KeypointsResult", "InferenceKeypointsModel", "FrameStream", "PoseTracker",
           "OneEuro", "PoseRenderer", "PoseStyle", "batch_to_coco",
           "evaluate_dataset_batched", "result_to_coco", "geometry", "ops", "eval_coco", "KeypointEvaluator",
           "KeypointGroundTruth"]
