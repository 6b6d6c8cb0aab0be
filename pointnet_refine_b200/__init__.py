"""pointnet_refine_b200 -- B200-native (sm_100a) forward hot path of LineRefineNet.

Importing the package loads the in-tree CUDA library (pointnet_refine_b200/liblrn_b200.so) through
its C ABI (include/lrn_b200.h) and raises if it has not been built: there is no CPU or PyTorch
fallback for the hot path.
"""
from . import _lib, ops  # noqa: F401  (loads liblrn_b200.so; raises if missing)
from .model import (DetrTransformerDecoderLayer, LineRefineNet, MultiScalePointNetEncoder,  # noqa: F401
                    PositionalEncoding)

from .graph import GraphedLineRefineNet, GraphedTrainStep  # noqa: F401,E402
from .ddp import FlatDataParallel  # noqa: F401,E402  (flat-gradient data parallelism for train_dist.py-style loops)
from . import scene  # noqa: F401,E402  (whole-scene front end: build_segments, refine_scene)
from . import data  # noqa: F401,E402  (SceneTrainingSet: shuffled training batches from device-resident scenes)

__all__ = ["FlatDataParallel", "GraphedLineRefineNet", "GraphedTrainStep", "LineRefineNet", "MultiScalePointNetEncoder", "PositionalEncoding", "DetrTransformerDecoderLayer", "ops", "scene", "data"]
