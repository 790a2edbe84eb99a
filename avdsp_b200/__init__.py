"""avdsp_b200 -- B200-native batched executor for AVDSP encoded DSP programs.

Only what the hot path needs: the CUDA kernels + C ABI (csrc/, libavdsp_b200.so), the host-side
mirror of the reference runtime interface (executor.py, compat.py), program-file readers, synthetic
PCM, and stream sharding.  Importing the package does not load the CUDA library; the first use does,
and fails loudly when it is missing.
"""
from .executor import (AvdspError, Executor, describe, coef_words, fir_tap_words, measure_int_peak, measure_f32_peak, INTERLEAVED, PLANAR, HOST, DEVICE,  # noqa: F401
                       KERNEL_AUTO, KERNEL_GENERIC, KERNEL_CHAIN, KERNEL_CHAIN_V1, KERNEL_MIX, KERNEL_FIR, KERNEL_FIR_TC,
                       KERNEL_CHAIN_V2, KERNEL_CHAIN_V3, KERNEL_DAG)
from .program import load, load_bin, load_hex, header  # noqa: F401
from .sharding import shard_range  # noqa: F401
from . import params  # noqa: F401
