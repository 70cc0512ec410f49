"""Batched render-and-compare loop driving the renderer (reference: estimation/simple_setup.py)."""
from .hypotheses import HypothesisOptimizer, gather_losses, global_best, shard_range  # noqa: F401
from .losses import (depth_to_pointcloud, depth_to_pointclouds, extract_instances, point_loss,  # noqa: F401
                     subsample_points)
from .streaming import StreamedDecodeRenderCompare, StreamedRenderCompare  # noqa: F401
from .decoder import (FusedTailDecoder, SDFDecoder, SurfaceDecoder, decoder_tail,  # noqa: F401
                      trunk_stage)
from .fused import decode_render_compare  # noqa: F401
from .view_dataset import BatchedSDFViewGenerator  # noqa: F401
from . import runtime_analysis  # noqa: F401
from .pipeline import NoDepthError, SDFPipeline  # noqa: F401
from . import views  # noqa: F401
