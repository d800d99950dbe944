"""echo-b200: a B200-native path-tracing core behind Echo's evaluator/aggregator interface (see DESIGN.md).

The package holds only what the hot path needs: csrc/ (hand-written CUDA for sm_100a + the C ABI, and the host-side
scene preparation in C++), the ctypes binding, and the host-side mirror of the reference interface for this path.
"""
from . import structs  # noqa: F401
from .host import InstanceDescription, PackDescription, PreparedArrays, SceneDescription, TextureDescription, prepare  # noqa: F401
from .scene import (AlbedoEvaluator, EvaluationOperation, EvaluationProfile, NormalDepthEvaluator, PathTracedEvaluator,  # noqa: F401
                    PreparedScene, RenderTexture, StandardNaiveEvaluator, build_light_tree_device, build_packs_device, build_qbvh_device, hilbert_curve_pattern, ordered_pattern,
                    shard_epochs, shard_tiles)
from ._native import EchoNativeError  # noqa: F401

__version__ = "0.1.0"
