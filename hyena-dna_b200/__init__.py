"""hyena_b200 -- Blackwell-native (sm_100a) Hyena long-convolution operator.

Drop-in for the HyenaOperator / HyenaFilter / fftconv surface of HazyResearch/hyena-dna
(src/models/sequence/hyena.py, src/ops/fftconv.py, csrc/fftconv).  Import as ``hyena_dna_b200``.
"""
from ._lib import HyenaB200Error, LIB_PATH, build, launch_count  # noqa: F401
from .hyena import (ExponentialModulation, HyenaFilter, HyenaInferenceCache, HyenaOperator, OptimModule,  # noqa: F401
                    PositionalEmbedding, Sin)
from .fftconv import FFTConvFunc, fftconv_bwd, fftconv_func, fftconv_fwd, fftconv_ref  # noqa: F401
from . import block, distributed, ops, registry, stack  # noqa: F401
from .block import Backbone, Block  # noqa: F401
from .stack import CheckpointedHyenaStack, enable_filter_cache, memory_plan  # noqa: F401
from .host import HostStep  # noqa: F401

__all__ = ["HyenaOperator", "HyenaInferenceCache", "HyenaFilter", "PositionalEmbedding", "ExponentialModulation", "Sin", "OptimModule",
           "fftconv_func", "fftconv_ref", "FFTConvFunc", "fftconv_fwd", "fftconv_bwd", "registry", "distributed", "ops",
           "HostStep", "Block", "Backbone", "block", "CheckpointedHyenaStack", "enable_filter_cache", "memory_plan", "stack", "build", "launch_count", "HyenaB200Error", "LIB_PATH"]
