"""B200-native fused D3PM / VQ-Diffusion reverse-diffusion token update.

Drop-in for the sampling-time methods of the reference's
`src/models/motionencoder/diffusion_transformer.py::DiffusionTransformer`
(p_sample / p_pred / cf_predict_start / predict_start / q_posterior /
log_sample_categorical / sample) on top of the C-ABI library `csrc/libd3pm_b200.so`
(hand-written sm_100a CUDA, declared in `include/d3pm_b200.h`).  Import as `d3pm_b200`.
"""
from d3pm_b200._lib import D3PMError, library_path, load_library  # noqa: F401
from d3pm_b200 import attention, decode, head, ops, train  # noqa: F401
from d3pm_b200.diffusion_transformer import FusedDiffusionTransformer, alpha_schedule  # noqa: F401
from d3pm_b200.distributed import gather_tokens, shard_range  # noqa: F401

__all__ = ["FusedDiffusionTransformer", "alpha_schedule", "ops", "D3PMError", "load_library", "library_path",
           "gather_tokens", "shard_range"]
