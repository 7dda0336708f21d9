"""B200-native flow-based temporal-consistency path (warp + occlusion mask + masked temporal error).

The directory name is not a Python identifier; import it with
``importlib.import_module("gan-based-video-style-transfer_b200")`` or through the ``tcl_b200`` shim at
the repository root.  ``dropin/`` holds modules named like the reference's (``flowtools``, ``fs_lib``,
``sintel_eval``) for ``sys.path``-style drop-in use.
"""
from . import _cabi  # noqa: F401
from .ops import (FusedResult, free_workspaces, generateMask, fbcCheckTorch, fbcCheckTorch_mob, fbcheck_with_near_count, fs_warp,  # noqa: F401
                  fused_forward, gradient, temporal_error, temporal_error_clip, temporal_error_host, temporal_error_per_pair, temporal_loss,
                  temporal_rmse_per_sample, upsample_flow, warp, warp_blend, warping_error_per_pair, window_evaluations, temporal_error_window)
from .sintel_eval import (aggregate_means, computeTCL, computeTCL_from_flows, save_dict_as_json)  # noqa: F401
from .sharding import (ShardPlan, plan_shards, evaluate_sharded, evaluate_sharded_host, evaluate_banded, band_rows, allreduce_sums)  # noqa: F401
from .chains import reconet_output_temporal_loss, ruder_network_input, long_term_blend_step  # noqa: F401
from . import synth  # noqa: F401
from . import ingest  # noqa: F401
from . import cv2compat  # noqa: F401
from . import library  # noqa: F401  (registers the torch.ops.tcl_b200 operators)
from .ingest import hwc_split, split_fc2_block, flow_hw2_to_planar, load_flo_planar, sintel_occlusion_mask  # noqa: F401

__all__ = ["gradient", "warp", "fbcCheckTorch", "fbcCheckTorch_mob", "fs_warp", "fused_forward",
           "temporal_error", "temporal_error_per_pair", "warping_error_per_pair", "temporal_error_clip", "temporal_error_host", "generateMask", "temporal_loss", "temporal_rmse_per_sample",
           "warp_blend", "computeTCL", "computeTCL_from_flows", "save_dict_as_json", "aggregate_means",
           "plan_shards", "evaluate_sharded", "evaluate_sharded_host", "allreduce_sums", "synth",
           "reconet_output_temporal_loss", "ruder_network_input", "long_term_blend_step", "window_evaluations", "temporal_error_window"]
