"""Model families with fused sm_100a kernels (and eager PyTorch oracles)."""
from .base import ShardModel
from .custom import CustomFamily
from .glm import (
    FAMILY_PARAMS,
    Fp8GlmShards,
    GlmShards,
    dequantize_block_fp8,
    quantize_block_fp8,
    synth_glm_shard,
    synth_logistic_shard,
    synth_logistic_shard_fp8,
)
from .linreg import LinregShards, make_demo_data
from .ode import LOTKA_VOLTERRA, OdeShards, OdeSystem, synth_lv_shard, synth_ode_shard

__all__ = [
    "ShardModel",
    "CustomFamily",
    "LinregShards",
    "make_demo_data",
    "GlmShards",
    "Fp8GlmShards",
    "FAMILY_PARAMS",
    "quantize_block_fp8",
    "dequantize_block_fp8",
    "synth_logistic_shard",
    "synth_logistic_shard_fp8",
    "synth_glm_shard",
    "OdeShards",
    "OdeSystem",
    "LOTKA_VOLTERRA",
    "synth_ode_shard",
    "synth_lv_shard",
]
