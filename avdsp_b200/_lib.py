"""ctypes binding of libavdsp_b200.so (the C ABI declared in include/avdsp_b200.h).

There is no fallback: if the CUDA extension has not been built this raises, and every compute call
fails when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libavdsp_b200.so")

# every symbol include/avdsp_b200.h declares (tests check the library exports all of them)
SYMBOLS = [
    "dspRuntimeInit", "dspRuntimeReset", "dspFindCore", "dspFindCoreBegin",
    "dspRuntime_2", "dspRuntime_3", "dspRuntime_4", "dspRuntime_5", "dspRuntime_6",
    "dspQNM", "dspQM64", "dspQM32", "dspOpcodeText",
    "avdsp_b200_create", "avdsp_b200_destroy", "avdsp_b200_reset", "avdsp_b200_io_map",
    "avdsp_b200_process", "avdsp_b200_process_async", "avdsp_b200_process_range", "avdsp_b200_process_pcm",
    "avdsp_b200_set_order", "avdsp_b200_set_kernel", "avdsp_b200_last_kernel", "avdsp_b200_last_chain_variant", "avdsp_b200_describe", "avdsp_b200_launch_count",
    "avdsp_b200_reload_params", "avdsp_b200_state_words", "avdsp_b200_data_size", "avdsp_b200_aux_offset",
    "avdsp_b200_mem_offset", "avdsp_b200_num_mem", "avdsp_b200_mem_word", "avdsp_b200_get_state",
    "avdsp_b200_set_state", "avdsp_b200_num_streams", "avdsp_b200_num_cores", "avdsp_b200_trace",
    "avdsp_b200_last_error", "avdsp_b200_measure_int_peak", "avdsp_b200_measure_f32_peak",
    "avdsp_b200_create_multi", "avdsp_b200_num_devices", "avdsp_b200_shard_info", "avdsp_b200_host_alloc", "avdsp_b200_host_free",
    "avdsp_b200_copy_only", "avdsp_b200_param_index", "avdsp_b200_set_param", "avdsp_b200_num_variants",
    "avdsp_b200_coef_words", "avdsp_b200_set_coefs", "avdsp_b200_fir_tap_words", "avdsp_b200_set_fir_taps",
]

_lib = None


def build(verbose: bool = False) -> str:
    """Compile the CUDA extension in-tree (nvcc, sm_100a).  Returns the library path."""
    import subprocess
    r = subprocess.run(["make", "-C", os.path.join(HERE, "csrc"), "-j4"], capture_output=True, text=True)
    if verbose or r.returncode:
        print(r.stdout[-4000:], r.stderr[-4000:])
    if r.returncode:
        raise RuntimeError("building libavdsp_b200.so failed")
    return LIB_PATH


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build the CUDA extension first "
            "(python -c 'import __graft_entry__ as g; g.build()').  avdsp_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, ci, pi = C.c_void_p, C.c_int, C.POINTER(C.c_int)
    L.avdsp_b200_create.argtypes = [C.POINTER(vp), vp, ci, ci, ci, ci, vp, ci, ci]
    L.avdsp_b200_create.restype = ci
    L.avdsp_b200_create_multi.argtypes = [C.POINTER(vp), vp, ci, ci, ci, ci, vp, ci, C.c_uint]
    L.avdsp_b200_create_multi.restype = ci
    L.avdsp_b200_num_devices.argtypes = [vp]
    L.avdsp_b200_shard_info.argtypes = [vp, ci, pi, pi, pi, pi]
    L.avdsp_b200_host_alloc.argtypes = [vp, C.c_size_t]
    L.avdsp_b200_host_alloc.restype = vp
    L.avdsp_b200_host_free.argtypes = [vp, vp]
    L.avdsp_b200_host_free.restype = None
    L.avdsp_b200_copy_only.argtypes = [vp, vp, vp, ci, ci]
    L.avdsp_b200_param_index.argtypes = [vp, ci, ci]
    L.avdsp_b200_set_param.argtypes = [vp, ci, ci, ci, vp, ci]
    L.avdsp_b200_num_variants.argtypes = [vp]
    L.avdsp_b200_coef_words.argtypes = [vp, ci, ci, vp, ci]
    L.avdsp_b200_set_coefs.argtypes = [vp, ci, ci, vp, ci, vp]
    L.avdsp_b200_fir_tap_words.argtypes = [vp, ci, ci, vp, ci]
    L.avdsp_b200_set_fir_taps.argtypes = [vp, ci, ci, vp, ci, vp]
    L.avdsp_b200_destroy.argtypes = [vp]
    L.avdsp_b200_destroy.restype = None
    L.avdsp_b200_reset.argtypes = [vp, ci, vp, ci]
    L.avdsp_b200_io_map.argtypes = [vp, pi, pi, pi, pi]
    L.avdsp_b200_process.argtypes = [vp, vp, vp, ci, ci, ci]
    L.avdsp_b200_process_async.argtypes = [vp, vp, vp, ci, ci, vp]
    L.avdsp_b200_process_pcm.argtypes = [vp, vp, ci, vp, ci, ci]
    L.avdsp_b200_process_range.argtypes = [vp, vp, vp, ci, ci, ci, ci, vp]
    L.avdsp_b200_set_order.argtypes = [vp, ci]
    L.avdsp_b200_set_kernel.argtypes = [vp, ci]
    L.avdsp_b200_last_kernel.argtypes = [vp]
    L.avdsp_b200_last_chain_variant.argtypes = [vp]
    L.avdsp_b200_describe.argtypes = [vp, ci, ci, ci, ci, ci, ci, C.c_char_p, ci]
    L.avdsp_b200_launch_count.argtypes = [vp]
    L.avdsp_b200_launch_count.restype = C.c_longlong
    L.avdsp_b200_reload_params.argtypes = [vp, vp, ci]
    for f in ("state_words", "data_size", "aux_offset", "mem_offset", "num_mem", "num_streams", "num_cores"):
        getattr(L, "avdsp_b200_" + f).argtypes = [vp]
    L.avdsp_b200_mem_word.argtypes = [vp, ci]
    L.avdsp_b200_get_state.argtypes = [vp, ci, vp]
    L.avdsp_b200_set_state.argtypes = [vp, ci, vp]
    L.avdsp_b200_trace.argtypes = [vp]
    L.avdsp_b200_trace.restype = C.c_char_p
    L.avdsp_b200_last_error.argtypes = []
    L.avdsp_b200_last_error.restype = C.c_char_p
    L.avdsp_b200_measure_int_peak.argtypes = [ci, ci]
    L.avdsp_b200_measure_int_peak.restype = C.c_double
    L.avdsp_b200_measure_f32_peak.argtypes = [ci, ci, ci]
    L.avdsp_b200_measure_f32_peak.restype = C.c_double
    # reference entry points
    L.dspRuntimeInit.argtypes = [vp, ci, ci, ci, ci]
    L.dspRuntimeReset.argtypes = [ci, ci, ci]
    L.dspFindCore.argtypes = [vp, ci]
    L.dspFindCore.restype = vp
    L.dspFindCoreBegin.argtypes = [vp]
    L.dspFindCoreBegin.restype = vp
    for f in (2, 3, 4, 5, 6):
        fn = getattr(L, f"dspRuntime_{f}")
        fn.argtypes = [vp, vp, vp]
        fn.restype = ci
    L.dspQNM.argtypes = [C.c_double, ci, ci]
    L.dspQNM.restype = C.c_longlong
    L.dspQM64.argtypes = [C.c_double, ci]
    L.dspQM64.restype = C.c_longlong
    L.dspQM32.argtypes = [C.c_double, ci]
    L.dspQM32.restype = ci
    _lib = L
    return L


def last_error() -> str:
    return lib().avdsp_b200_last_error().decode()
