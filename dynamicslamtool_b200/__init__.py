"""mor-b200: B200-native (sm_100a) implementation of MOR's per-frame filtering hot path.

The product is `libmor_b200.so` (CUDA kernels + C ABI, include/mor_b200.h) and the C++ class
`MovingObjectRemoval` (include/MOR/MovingObjectRemoval.h). This Python package is only the ctypes
binding used by the tests and bench.py, plus the build recipe.
"""
from .binding import (MixedBatch, MorBinding, MorConfig, MorError, MorLimits, MovingObjectRemoval, SequenceBatch, Synth, load_product,  # noqa: F401
                      parse_config, PRODUCT_LIB, SYNTH_LIB, REPO_ROOT, TAPS, COUNT_NAMES)
