"""Host-side mirror of the reference's runtime interface for the batched path.

`Executor` plays the role of dspRuntimeInit + dspRuntimeReset + the per-period loop of dsp_transfer
(/root/reference/module_avdsp/linux/avdsp_plugin.c:71-163) for `n_streams` independent instances of one
program; all work happens in libavdsp_b200.so (hand-written CUDA, sm_100a).  Return codes of the
reference (-1..-6) surface as `AvdspError.code`.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib

INTERLEAVED, PLANAR = 0, 1
HOST, DEVICE = 0, 1
KERNEL_AUTO, KERNEL_GENERIC, KERNEL_CHAIN, KERNEL_CHAIN_V1, KERNEL_MIX, KERNEL_FIR, KERNEL_FIR_TC = 0, 1, 2, 3, 4, 5, 6
KERNEL_CHAIN_V2, KERNEL_CHAIN_V3 = 7, 8        # force k_chain2 / k_chain3 (KERNEL_CHAIN and AUTO choose between them)
KERNEL_DAG = 9                                 # X/Y dataflow programs (kernel_dag.cu)
PCM_S32, PCM_S16, PCM_S24_3LE = 0, 1, 2
KERNEL_NAMES = {0: "none", 1: "generic", 2: "chain", 3: "chain_v1", 4: "mix", 5: "fir", 6: "fir_tc", 9: "dag"}


class AvdspError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"avdsp_b200 error {code}: {msg}")
        self.code = code


def _check(rc: int) -> int:
    if rc < 0:
        raise AvdspError(rc, _lib.last_error())
    return rc


class Executor:
    """n_streams independent instances of one encoded DSP program on one GPU."""

    def __init__(self, words, fs: int, fmt: int = 2, n_streams: int = 1, seeds=None, dither: int = 31, device: int = 0, devices=None):
        """devices: list of CUDA ordinals -> one multi-device instance (avdsp_b200_create_multi): the streams are cut into
        contiguous ranges, one per GPU; such an instance takes host (numpy) buffers only."""
        L = _lib.lib()
        self._L = L
        self.words = np.ascontiguousarray(words, dtype=np.int32)
        self.fs, self.fmt, self.n_streams, self.device = fs, fmt, n_streams, device
        self._h = C.c_void_p()
        sp = None
        if seeds is not None:
            self._seeds = np.ascontiguousarray(seeds, dtype=np.int32)
            assert self._seeds.shape == (n_streams,)
            sp = self._seeds.ctypes.data
        if devices is None:
            self.total_length = _check(L.avdsp_b200_create(C.byref(self._h), self.words.ctypes.data, len(self.words), fs, fmt,
                                                           n_streams, sp, dither, device))
        else:
            mask = 0
            for d in devices:
                mask |= 1 << int(d)
            self.total_length = _check(L.avdsp_b200_create_multi(C.byref(self._h), self.words.ctypes.data, len(self.words), fs, fmt,
                                                                 n_streams, sp, dither, mask))
        self.n_devices = L.avdsp_b200_num_devices(self._h)
        n_in, n_out = C.c_int(), C.c_int()
        a, b = (C.c_int * 32)(), (C.c_int * 32)()
        L.avdsp_b200_io_map(self._h, C.byref(n_in), a, C.byref(n_out), b)
        self.in_idx, self.out_idx = list(a[: n_in.value]), list(b[: n_out.value])
        self.n_in, self.n_out = n_in.value, n_out.value
        self.state_words = L.avdsp_b200_state_words(self._h)
        self.data_size = L.avdsp_b200_data_size(self._h)
        self.aux_offset = L.avdsp_b200_aux_offset(self._h)
        self.mem_offset = L.avdsp_b200_mem_offset(self._h)
        self.num_mem = L.avdsp_b200_num_mem(self._h)
        self.mem_words = [L.avdsp_b200_mem_word(self._h, k) for k in range(self.num_mem)]
        self.num_cores = L.avdsp_b200_num_cores(self._h)

    def shards(self):
        """[(device, first_stream, n_streams, numa_node)] per GPU of the instance"""
        out = []
        for k in range(self.n_devices):
            v = [C.c_int() for _ in range(4)]
            _check(self._L.avdsp_b200_shard_info(self._h, k, *[C.byref(q) for q in v]))
            out.append(tuple(q.value for q in v))
        return out

    def alloc_pcm(self, n_frames: int, channels: int) -> np.ndarray:
        """Page-locked int32 [n_streams, n_frames, channels] buffer placed for this instance (avdsp_b200_host_alloc: each GPU's
        slice on the host NUMA node next to it).  Freed with the Executor."""
        per = n_frames * channels * 4
        p = self._L.avdsp_b200_host_alloc(self._h, per)
        if not p:
            raise AvdspError(-9, _lib.last_error())
        buf = (C.c_int32 * (self.n_streams * n_frames * channels)).from_address(p)
        return np.ctypeslib.as_array(buf).reshape(self.n_streams, n_frames, channels)

    def copy_only(self, x_host: np.ndarray, y_host: np.ndarray, layout: int = INTERLEAVED):
        """The DMA schedule of the host path without the kernel (avdsp_b200_copy_only): the copy roofline of process()."""
        n_frames = x_host.shape[1] if layout == INTERLEAVED else x_host.shape[2]
        _check(self._L.avdsp_b200_copy_only(self._h, x_host.ctypes.data, y_host.ctypes.data, n_frames, layout))

    def close(self):
        if getattr(self, "_h", None):
            self._L.avdsp_b200_destroy(self._h)
            self._h = None

    __del__ = close

    # -- control -----------------------------------------------------------------------------------
    def reset(self, fs=None, seeds=None, dither: int = 31):
        sp = None
        if seeds is not None:
            self._seeds = np.ascontiguousarray(seeds, dtype=np.int32)
            sp = self._seeds.ctypes.data
        _check(self._L.avdsp_b200_reset(self._h, self.fs if fs is None else fs, sp, dither))
        if fs is not None:
            self.fs = fs

    def set_order(self, period: int = 0):
        _check(self._L.avdsp_b200_set_order(self._h, period))

    def set_kernel(self, which: int):
        _check(self._L.avdsp_b200_set_kernel(self._h, which))

    def reload_params(self, words):
        w = np.ascontiguousarray(words, dtype=np.int32)
        _check(self._L.avdsp_b200_reload_params(self._h, w.ctypes.data, len(w)))
        self.words = w

    def param_index(self, offset: int, param_num: int = 0) -> int:
        """dump-file entry (offset, PARAM_NUM number) -> word index in the program (avdsp_b200_param_index)"""
        return _check(self._L.avdsp_b200_param_index(self._h, offset, param_num))

    def set_param(self, first_stream: int, n_streams: int, word_index: int, values):
        """streams [first_stream, first_stream + n_streams) run with program words [word_index, ...) replaced by `values`"""
        v = np.ascontiguousarray(values, dtype=np.int32).reshape(-1)
        _check(self._L.avdsp_b200_set_param(self._h, first_stream, n_streams, word_index, v.ctypes.data, len(v)))

    def set_coefs(self, first: int, values):
        """Per-stream biquad coefficients (avdsp_b200_set_coefs): row s of `values` ([n, nCoef], columns in the order of
        coef_words(words, fmt)) holds the coefficient words of stream first + s.  A numpy array is copied from the host; a
        contiguous int32 or float32 CUDA tensor on the instance's device is read on torch.cuda.current_stream() without a host
        sync (a tensor on another device is refused).  Float arrays are bit patterns, never value-cast."""
        self._set_rows(self._L.avdsp_b200_set_coefs, first, values, self.n_coef, "coefficient")

    def set_fir_taps(self, first: int, values):
        """Per-stream FIR taps (avdsp_b200_set_fir_taps): row s of `values` ([n, nTaps], columns in the order of
        fir_tap_words(words, fmt)) holds the tap words of stream first + s.  Host and device rows as for set_coefs."""
        self._set_rows(self._L.avdsp_b200_set_fir_taps, first, values, self.n_taps, "FIR tap")

    @property
    def n_coef(self) -> int:
        """columns of a set_coefs row"""
        return len(coef_words(self.words, self.fmt))

    @property
    def n_taps(self) -> int:
        """columns of a set_fir_taps row"""
        return len(fir_tap_words(self.words, self.fmt))

    def _set_rows(self, fn, first, values, ncol, what):
        if isinstance(values, np.ndarray):
            v = self._as_words(values)
            if v.ndim != 2 or v.shape[1] != ncol:
                raise ValueError(f"{what} rows must be [n, {ncol}], not {v.shape}")
            _check(fn(self._h, first, v.shape[0], v.ctypes.data, HOST, None))
            return
        import torch
        if not (values.is_cuda and values.dtype in (torch.int32, torch.float32) and values.is_contiguous() and values.dim() == 2):
            raise ValueError(f"device {what} rows must be a contiguous 2-D int32 or float32 CUDA tensor")
        if values.shape[1] != ncol:
            raise ValueError(f"{what} rows must be [n, {ncol}], not {tuple(values.shape)}")
        if self.n_devices == 1 and values.device.index != self.device:
            raise ValueError(f"device {what} rows must be on cuda:{self.device}, not {values.device}")
        stream = torch.cuda.current_stream(values.device).cuda_stream
        _check(fn(self._h, first, int(values.shape[0]), values.data_ptr(), DEVICE, stream))

    @property
    def num_variants(self) -> int:
        return int(self._L.avdsp_b200_num_variants(self._h))

    @property
    def last_kernel(self) -> str:
        return KERNEL_NAMES[self._L.avdsp_b200_last_kernel(self._h)]

    @property
    def last_chain_variant(self) -> int:
        """2 / 3: which chain kernel (kernel_chain2.cu / kernel_chain3.cu) the last call ran, 0 if it was no chain kernel."""
        return int(self._L.avdsp_b200_last_chain_variant(self._h))

    @property
    def launch_count(self) -> int:
        return int(self._L.avdsp_b200_launch_count(self._h))

    @property
    def trace(self) -> str:
        return self._L.avdsp_b200_trace(self._h).decode()

    # -- state --------------------------------------------------------------------------------------
    def get_state(self, stream: int) -> np.ndarray:
        w = np.zeros(self.state_words, dtype=np.int32)
        _check(self._L.avdsp_b200_get_state(self._h, stream, w.ctypes.data))
        return w

    def set_state(self, stream: int, words):
        w = np.ascontiguousarray(words, dtype=np.int32)
        assert w.shape == (self.state_words,)
        _check(self._L.avdsp_b200_set_state(self._h, stream, w.ctypes.data))

    # -- processing ---------------------------------------------------------------------------------
    def _shapes(self, n_frames, layout):
        if layout == INTERLEAVED:
            return (self.n_streams, n_frames, self.n_in), (self.n_streams, n_frames, self.n_out)
        return (self.n_streams, self.n_in, n_frames), (self.n_streams, self.n_out, n_frames)

    def process(self, x, layout: int = INTERLEAVED, out=None):
        """x: int32 PCM (float32 bit patterns for formats 5/6), [S, T, nIn] interleaved or [S, nIn, T]
        planar.  numpy array -> host path (copies inside the call); torch CUDA tensor -> device path.
        Returns the outputs in the same layout and memory space."""
        if isinstance(x, np.ndarray):
            x = self._as_words(x)
            n_frames = x.shape[1] if layout == INTERLEAVED else x.shape[2]
            si, so = self._shapes(n_frames, layout)
            if x.shape != si:
                raise ValueError(f"input shape {x.shape}, expected {si}")
            if out is None:
                y = np.empty(so, dtype=np.int32)
            else:       # the C call writes prod(so) words through this pointer: it has to be exactly that buffer
                if not (isinstance(out, np.ndarray) and out.shape == so and out.dtype.itemsize == 4 and out.dtype.kind in "iuf"
                        and out.flags.c_contiguous and out.flags.writeable):
                    raise ValueError(f"out must be a writable C-contiguous 32-bit array of shape {so}")
                y = out
            _check(self._L.avdsp_b200_process(self._h, x.ctypes.data, y.ctypes.data, n_frames, layout, HOST))
            return y
        import torch
        if not (x.is_cuda and x.dtype in (torch.int32, torch.float32) and x.is_contiguous()):
            raise ValueError("device input must be a contiguous int32 (float32 for DSP_FORMAT 5/6) CUDA tensor")
        n_frames = x.shape[1] if layout == INTERLEAVED else x.shape[2]
        si, so = self._shapes(n_frames, layout)
        if tuple(x.shape) != si:
            raise ValueError(f"input shape {tuple(x.shape)}, expected {si}")
        if out is None:
            y = torch.empty(so, dtype=x.dtype, device=x.device)
        else:
            if not (out.is_cuda and out.device == x.device and tuple(out.shape) == so and out.is_contiguous()
                    and out.dtype in (torch.int32, torch.float32)):
                raise ValueError(f"out must be a contiguous 32-bit CUDA tensor of shape {so} on {x.device}")
            y = out
        stream = torch.cuda.current_stream(x.device).cuda_stream
        _check(self._L.avdsp_b200_process_async(self._h, x.data_ptr(), y.data_ptr(), n_frames, layout, stream))
        return y

    def process_range(self, x, first: int, out=None, layout: int = INTERLEAVED, stream=None):
        """Streams [first, first + x.shape[0]) only, device tensors, enqueued on `stream` (a torch.cuda.Stream; default: the
        current one).  Calls on one Executor are ordered by the library whatever stream they are given."""
        import torch
        n = int(x.shape[0])
        n_frames = x.shape[1] if layout == INTERLEAVED else x.shape[2]
        if not (x.is_cuda and x.dtype in (torch.int32, torch.float32) and x.is_contiguous()):
            raise ValueError("device input must be a contiguous 32-bit CUDA tensor")
        so = (n, n_frames, self.n_out) if layout == INTERLEAVED else (n, self.n_out, n_frames)
        y = torch.empty(so, dtype=x.dtype, device=x.device) if out is None else out
        if tuple(y.shape) != so or not y.is_contiguous():
            raise ValueError(f"out must be contiguous with shape {so}")
        st = (stream or torch.cuda.current_stream(x.device)).cuda_stream
        _check(self._L.avdsp_b200_process_range(self._h, x.data_ptr(), y.data_ptr(), n_frames, layout, first, n, st))
        return y

    @staticmethod
    def _as_words(x: np.ndarray) -> np.ndarray:
        """32-bit samples as they are: int32 s.31, or float32 BIT PATTERNS for DSP_FORMAT 5/6 (never value-cast)."""
        if x.dtype == np.float32 or x.dtype == np.uint32:
            return np.ascontiguousarray(x).view(np.int32)
        if x.dtype != np.int32:
            raise ValueError(f"PCM must be int32 (or float32 for DSP_FORMAT 5/6), not {x.dtype}")
        return np.ascontiguousarray(x)

    def process_pcm(self, raw: np.ndarray, pcm_format: int, n_frames: int) -> np.ndarray:
        """ALSA sample formats (linux/avdsp_plugin.c:109-121): raw = interleaved S16_LE (int16 array) or S24_3LE
        (uint8 array, 3 bytes per sample) or S32 frames of all streams; returns int32 [S, T, nOut]."""
        raw = np.ascontiguousarray(raw)
        y = np.empty((self.n_streams, n_frames, self.n_out), dtype=np.int32)
        _check(self._L.avdsp_b200_process_pcm(self._h, raw.ctypes.data, pcm_format, y.ctypes.data, n_frames, HOST))
        return y

    def process_pinned(self, x_host, y_host, layout: int = INTERLEAVED):
        """Host path on caller-owned (ideally pinned) buffers given as torch CPU tensors or numpy arrays."""
        n_frames = x_host.shape[1] if layout == INTERLEAVED else x_host.shape[2]
        xp = x_host.data_ptr() if hasattr(x_host, "data_ptr") else x_host.ctypes.data
        yp = y_host.data_ptr() if hasattr(y_host, "data_ptr") else y_host.ctypes.data
        _check(self._L.avdsp_b200_process(self._h, xp, yp, n_frames, layout, HOST))
        return y_host


def describe(words, fs: int, fmt: int = 2, n_streams: int = 1, dither: int = 31, num_sms: int = 148) -> str:
    """Lowering trace + kernel geometries for `n_streams` streams on a GPU with `num_sms` SMs.  Host-only (no CUDA device needed)."""
    w = np.ascontiguousarray(words, dtype=np.int32)
    buf = C.create_string_buffer(1 << 16)
    _check(_lib.lib().avdsp_b200_describe(w.ctypes.data, len(w), fs, fmt, dither, n_streams, num_sms, buf, len(buf)))
    return buf.value.decode()


def _table_words(fn, words, fmt: int) -> np.ndarray:
    w = np.ascontiguousarray(words, dtype=np.int32)
    out = np.zeros(_check(fn(w.ctypes.data, len(w), fmt, None, 0)), dtype=np.int32)
    if out.size:
        _check(fn(w.ctypes.data, len(w), fmt, out.ctypes.data, out.size))
    return out


def coef_words(words, fmt: int = 2) -> np.ndarray:
    """Word indices of the program's biquad coefficients (every section, every fs column, bypassed blocks too), ascending: the
    column order of Executor.set_coefs.  Host-only (no CUDA device needed)."""
    return _table_words(_lib.lib().avdsp_b200_coef_words, words, fmt)


def fir_tap_words(words, fmt: int = 2) -> np.ndarray:
    """Word indices of the program's FIR taps (every convolution entry of every DSP_FIR, every fs column), ascending, each
    word once: the column order of Executor.set_fir_taps.  Host-only (no CUDA device needed)."""
    return _table_words(_lib.lib().avdsp_b200_fir_tap_words, words, fmt)


def measure_int_peak(device: int = 0, iters: int = 4096) -> float:
    """mad.wide.s32 per second the whole device sustains (denominator of the INT-pipe roofline)."""
    return float(_lib.lib().avdsp_b200_measure_int_peak(device, iters))


def measure_f32_peak(device: int = 0, iters: int = 4096, packed: bool = False) -> float:
    """Non-fused float MACs (mul.rz.ftz + add.rn) per second the whole device sustains (FP32-pipe roofline)."""
    return float(_lib.lib().avdsp_b200_measure_f32_peak(device, iters, 1 if packed else 0))
