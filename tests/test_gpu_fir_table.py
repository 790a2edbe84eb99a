"""Per-stream FIR tables (avdsp_b200_set_fir_taps): every stream its own room-correction filter in one launch.  Every case is
checked against one oracle instance per stream running that stream's own program (the loaded words with its row patched in):
outputs and data area (delay lines) bit-exact."""
import os

import numpy as np
import pytest

from conftest import load_program
from avdsp_b200 import (Executor, AvdspError, synth, coef_words, fir_tap_words, KERNEL_AUTO, KERNEL_FIR, KERNEL_FIR_TC,
                        KERNEL_GENERIC)
from oracle import wire
from test_fir_table import fir_program, taps

pytestmark = pytest.mark.gpu

ERR_UNSUPPORTED, ERR_ARG = -8, -9


def impulse_rows(base, tw, n, fmt, seed):
    """n distinct impulse responses: every tap of the program moved by up to 4096 LSBs (Q4.28) or by a relative 1e-3 (float)"""
    rng = np.random.default_rng(seed)
    v = base[tw].astype(np.int32)
    if fmt == 2:
        return (v[None, :].astype(np.int64) + rng.integers(-4096, 4097, (n, len(tw)))).astype(np.int32)
    f = v.view(np.float32).astype(np.float64)[None, :] * (1.0 + rng.uniform(-1e-3, 1e-3, (n, len(tw))))
    return np.ascontiguousarray(f.astype(np.float32).view(np.int32))


def own_program(base, tw, row):
    p = base.copy()
    p[tw] = row
    return p


def check_streams(oracle_lib, y, ex, progs_of, x, fmt, fs, streams, switch=0, base=None, dither=31):
    """stream s ran `base` for frames [0, switch), then progs_of(s)"""
    for s in streams:
        o = oracle_lib.Oracle(base if switch else progs_of(s), fmt, fs, seed=s, dither=dither)
        parts = []
        if switch:
            parts.append(o.process(x[s, :switch]))
            p = progs_of(s)
            o.code[: len(p)] = p[: len(o.code)]
        parts.append(o.process(x[s, switch:]))
        assert np.array_equal(y[s], np.concatenate(parts)), s
        assert np.array_equal(ex.get_state(s)[: ex.data_size], o.data), s


def make(base, fs, fmt, S, dither=31):
    return Executor(base, fs, fmt, S, seeds=np.arange(S, dtype=np.int32), dither=dither)


@pytest.mark.parametrize("fmt,kernel", [(f, k) for f in (2, 3) for k in (KERNEL_AUTO, KERNEL_FIR, KERNEL_GENERIC)] + [(2, KERNEL_FIR_TC)])
def test_64_streams_64_impulse_responses(oracle_lib, kernel, fmt):
    """C4 (two 4096-tap paths), 64 rooms with 64 different impulse responses, switched in between two calls"""
    fs, S, T, cut = 48000, 64, 700, 300
    base = load_program(f"c4_fir4096_f{fmt}_48k")
    tw = fir_tap_words(base, fmt)
    rows = impulse_rows(base, tw, S, fmt, seed=3 + fmt)
    assert len(np.unique(rows, axis=0)) == S
    ex = make(base, fs, fmt, S)
    ex.set_kernel(kernel)
    x = synth.pcm("noise", S, T, ex.n_in, fs)
    ya = ex.process(x[:, :cut])
    ex.set_fir_taps(0, rows)
    l1 = ex.launch_count
    yb = ex.process(x[:, cut:])
    assert ex.num_variants == 1
    if kernel == KERNEL_FIR_TC:         # the per-stream tensor-core form: Toeplitz planes built once, pack + GEMM + delay lines
        assert ex.last_kernel == "fir_tc" and ex.launch_count - l1 == 1 + 3
    else:
        assert ex.last_kernel == ("generic" if kernel == KERNEL_GENERIC else "fir")
        assert ex.launch_count - l1 == (1 if kernel == KERNEL_GENERIC else 2 + (fmt == 3))   # k_fir + k_fir_state (+ the exact pass)
    y = np.concatenate([ya, yb], axis=1)
    check_streams(oracle_lib, y, ex, lambda s: own_program(base, tw, rows[s]), x, fmt, fs, range(S), switch=cut, base=base)


def test_1024_streams_c4_frames_auto_alternates(oracle_lib):
    """1024 distinct streams over the C4 frame count, in short and long calls: AUTO alternates between k_fir (< 8192 frames)
    and the per-stream tensor-core form, and a row change between calls rebuilds the Toeplitz planes; spot streams across the
    batch and the call"""
    fs, S = 48000, 1024
    base = load_program("c4_fir4096_f2_48k")
    tw = fir_tap_words(base, 2)
    rows = impulse_rows(base, tw, S, 2, seed=11)
    ex = make(base, fs, 2, S)
    ex.set_fir_taps(0, rows)
    import torch
    cuts = [(37, "fir"), (37 + 8192, "fir_tc"), (1237 + 8192, "fir"), (65536, "fir_tc")]
    x = synth.pcm("noise", S, 65536, ex.n_in, fs)
    xd = torch.from_numpy(x).cuda()                             # device buffers: each call reaches the kernels whole
    parts, a = [], 0
    for b, kern in cuts:
        parts.append(ex.process(xd[:, a:b].contiguous()))
        assert ex.last_kernel == kern, b
        a = b
    y = torch.cat(parts, dim=1).cpu().numpy()
    check_streams(oracle_lib, y, ex, lambda s: own_program(base, tw, rows[s]), x, 2, fs, (0, 1, 300, 511, 512, 1023))


@pytest.mark.parametrize("kernel", [KERNEL_AUTO, KERNEL_FIR])
def test_float_rows_with_a_tiny_tap_stay_exact(oracle_lib, kernel):
    """a tap below 2^-60 on a few streams: those streams leave the FIR kernel for the interpreter inside the same call"""
    fs, S, T = 48000, 48, 500
    base = load_program("c4_fir4096_f3_48k")
    tw = fir_tap_words(base, 3)
    rows = impulse_rows(base, tw, S, 3, seed=5)
    tiny = {3: 10, 17: 4096 + 7, 47: 4095}                      # stream -> column (both paths)
    for s, c in tiny.items():
        rows[s, c] = np.float32(2.0 ** -70).view(np.int32)
    rows[20, 5] = np.float32(-(2.0 ** -100)).view(np.int32)
    ex = make(base, fs, 3, S)
    ex.set_kernel(kernel)
    ex.set_fir_taps(0, rows)
    x = synth.pcm("full", S, T, ex.n_in, fs)
    y = ex.process(x)
    assert ex.last_kernel == "fir"
    check_streams(oracle_lib, y, ex, lambda s: own_program(base, tw, rows[s]), x, 3, fs, range(S))


def test_set_param_reload_and_reset(oracle_lib):
    fs, S, T = 48000, 16, 300
    imps = [[taps(300, 2, 1), taps(50, 2, 2), taps(64, 2, 3)], [taps(257, 2, 4), None, None]]     # 48k, 88.2k, 96k
    base = fir_program(2, imps, fmin=48000, fmax=96000)
    tw = fir_tap_words(base, 2)
    rows = impulse_rows(base, tw, S, 2, seed=9)
    ex = make(base, fs, 2, S)
    ex.set_fir_taps(0, rows)
    # set_param on tap words writes rows, no variant
    w0, vals = int(tw[5]), np.array([1 << 26, -(1 << 25), 77], np.int32)
    ex.set_param(2, 5, w0, vals)
    assert ex.num_variants == 1
    rows[2:7, 5:8] = vals
    x = synth.pcm("noise", S, T, ex.n_in, fs)
    y = ex.process(x)
    assert ex.last_kernel == "fir"
    check_streams(oracle_lib, y, ex, lambda s: own_program(base, tw, rows[s]), x, 2, fs, range(S))
    # reset keeps the table, also at another rate (the 96k columns of the rows)
    for rate in (96000, 48000):
        ex.reset(rate, seeds=np.arange(S, dtype=np.int32), dither=31)
        x = synth.pcm("noise", S, T, ex.n_in, rate)
        y = ex.process(x)
        check_streams(oracle_lib, y, ex, lambda s: own_program(base, tw, rows[s]), x, 2, rate, range(S))
    # reload_params drops it
    ex.reload_params(base)
    ex.reset(fs, seeds=np.arange(S, dtype=np.int32), dither=31)
    y = ex.process(x)
    check_streams(oracle_lib, y, ex, lambda s: base, x, 2, fs, range(S))


def test_table_starts_from_variants_and_combines_with_them(oracle_lib):
    fs, S, T = 48000, 12, 400
    imps = [[taps(200, 3, 4)], [taps(150, 3, 5)]]
    base = fir_program(3, imps)
    tw = fir_tap_words(base, 3)
    ex = make(base, fs, 3, S)
    v = taps(3, 3, 6)
    vw = np.array(v, np.float32).view(np.int32)
    ex.set_param(0, 4, int(tw[10]), vw)                          # streams 0..3 on a variant before the table exists
    assert ex.num_variants == 2
    rows = impulse_rows(base, tw, 6, 3, seed=8)
    ex.set_fir_taps(6, rows)                                     # streams 6..11: rows; 0..5 keep what they ran with
    assert ex.num_variants == 2
    progs = [base.copy() for _ in range(S)]
    for s in range(4):
        progs[s][tw[10]: tw[10] + 3] = vw
    for s in range(6, S):
        progs[s] = own_program(base, tw, rows[s - 6])
    x = synth.pcm("noise", S, T, ex.n_in, fs)
    y = ex.process(x)
    check_streams(oracle_lib, y, ex, lambda s: progs[s], x, 3, fs, range(S))


def test_host_and_device_rows(oracle_lib):
    import torch
    fs, S, T = 48000, 40, 600
    base = load_program("c4s_fir_f2_multifs")
    tw = fir_tap_words(base, 2)
    rows = impulse_rows(base, tw, S, 2, seed=13)
    rows2 = impulse_rows(base, tw, S, 2, seed=14)
    ex = make(base, fs, 2, S)
    src = torch.from_numpy(rows).cuda()
    torch.cuda.synchronize()
    dev = torch.empty_like(src)
    torch.add(src, 0, out=dev)                                   # a kernel on the current stream writes the rows
    ex.set_fir_taps(0, dev)
    x = synth.pcm("noise", S, T, ex.n_in, fs)
    xd = torch.from_numpy(x).cuda()
    ya = ex.process(xd[:, :250].contiguous())
    src2 = torch.from_numpy(rows2).cuda()
    dev2 = torch.empty_like(src2)
    torch.add(src2, 0, out=dev2)
    ex.set_fir_taps(0, dev2)                                     # between two calls, no host sync
    yb = ex.process(xd[:, 250:].contiguous())
    torch.cuda.synchronize()
    y = torch.cat([ya, yb], dim=1).cpu().numpy()
    for s in range(S):
        o = oracle_lib.Oracle(own_program(base, tw, rows[s]), 2, fs, seed=s, dither=31)
        r = [o.process(x[s, :250])]
        o.code[: len(base)] = own_program(base, tw, rows2[s])
        r.append(o.process(x[s, 250:]))
        assert np.array_equal(y[s], np.concatenate(r)), s
        assert np.array_equal(ex.get_state(s)[: ex.data_size], o.data), s


def fir_and_biquad_tables(fmt, S, fs):
    """a program mixing FIR and biquads, with a FIR table and a coefficient table whose rows all differ"""
    base = fir_program(fmt, [[taps(40, fmt, 1)], [taps(33, fmt, 2)]], biquad=True)
    tw, cw = fir_tap_words(base, fmt), coef_words(base, fmt)
    rows = impulse_rows(base, tw, S, 2 if fmt == 2 else 3, seed=15)     # taps are float bit patterns in every float format
    rng = np.random.default_rng(16)
    cv = base[cw].astype(np.int32)
    crow = np.repeat(cv[None, :], S, 0)
    if fmt == 2:
        crow[:, :3] += rng.integers(-64, 65, (S, 3)).astype(np.int32)
    else:
        crow[:, :3] = (cv[:3].view(np.float32)[None, :] * (1 + rng.uniform(-1e-3, 1e-3, (S, 3)))).astype(np.float32).view(np.int32)
    ex = make(base, fs, fmt, S, dither=24)
    ex.set_fir_taps(0, rows)
    ex.set_coefs(0, np.ascontiguousarray(crow))

    def prog(s):
        p = own_program(base, tw, rows[s])
        p[cw] = crow[s]
        return p
    return ex, base, tw, cw, prog


@pytest.mark.parametrize("fmt", [2, 3, 4, 6])
def test_fir_and_biquad_tables_on_generic(oracle_lib, fmt):
    """a program mixing FIR and biquads runs on k_generic: both tables meet there"""
    fs, S, T = 48000, 24, 300
    ex, _, _, _, prog = fir_and_biquad_tables(fmt, S, fs)
    x = (synth.pcm_float if fmt >= 5 else synth.pcm)("noise", S, T, ex.n_in, fs)
    y = ex.process(x)
    assert ex.last_kernel == "generic"
    check_streams(oracle_lib, y, ex, prog, x, fmt, fs, range(S), dither=24)


@pytest.mark.parametrize("fmt", [2, 3])
def test_one_set_param_spans_both_tables_and_a_variant_word(oracle_lib, fmt):
    """one set_param over core 0's last tap, the words of the BIQUADS block before its first coefficient, and that coefficient:
    the tap goes into the FIR rows, the coefficient into the coefficient rows, and the informational type word makes one
    variant for the range"""
    fs, S, T, first, n = 48000, 24, 300, 5, 11
    ex, base, tw, cw, prog = fir_and_biquad_tables(fmt, S, fs)
    a, b = int(tw[tw < cw[0]][-1]), int(cw[0])
    hdr = a + 1 + int(np.flatnonzero((base[a + 1: b] >> 16) == wire.OP["BIQUADS"])[0])
    vals = base[a: b + 1].copy()
    vals[0] = np.float32(0.03125).view(np.int32) if fmt != 2 else 1 << 24                # the tap
    vals[hdr + 2 - a] = 0x00020000 | 1000                                                 # section type << 16 | freq
    vals[-1] = np.float32(0.09375).view(np.int32) if fmt != 2 else int(base[b]) + 99      # b0
    assert sum(w in tw for w in range(a, b + 1)) == 1 and sum(w in cw for w in range(a, b + 1)) == 1
    ex.set_param(first, n, a, vals)
    assert ex.num_variants == 2
    x = synth.pcm("noise", S, T, ex.n_in, fs)
    y = ex.process(x)

    def prog2(s):
        p = prog(s)
        if first <= s < first + n:
            p[a: b + 1] = vals
        return p
    check_streams(oracle_lib, y, ex, prog2, x, fmt, fs, range(S), dither=24)


def test_refusals_change_nothing(oracle_lib):
    from avdsp_b200 import _lib
    import torch
    fs, S, T = 48000, 8, 300
    exm = Executor(load_program("c2_testrpi_xover_f2_192k"), 192000, 2, 2)
    with pytest.raises(AvdspError) as e:
        exm.set_fir_taps(0, np.zeros((2, 0), np.int32))
    assert e.value.code == ERR_UNSUPPORTED
    base = fir_program(2, [[taps(100, 2, 1)], [taps(60, 2, 2)]])
    tw = fir_tap_words(base, 2)
    rows = impulse_rows(base, tw, S, 2, seed=17)
    ex = make(base, fs, 2, S)
    ex.set_fir_taps(0, rows)
    for first, r in ((-1, rows), (1, rows), (S, rows[:1])):
        with pytest.raises(AvdspError) as e:
            ex.set_fir_taps(first, r)
        assert e.value.code == ERR_ARG
    L = _lib.lib()
    assert L.avdsp_b200_set_fir_taps(ex._h, 0, 1, None, 0, None) == ERR_ARG
    assert L.avdsp_b200_set_fir_taps(ex._h, 0, 1, rows.ctypes.data, 7, None) == ERR_ARG
    for bad in (rows[:, :-1], np.concatenate([rows, rows[:, :1]], axis=1)):
        with pytest.raises(ValueError):
            ex.set_fir_taps(0, np.ascontiguousarray(bad))
    with pytest.raises(ValueError):
        ex.set_fir_taps(0, torch.from_numpy(np.ascontiguousarray(rows[:, :-1])).cuda())
    # a set_param that changes a tap block's length is refused before it changes anything (not even the tap it carries)
    t = int(tw[0]) - 1
    with pytest.raises(AvdspError) as e:
        ex.set_param(0, 2, t, np.array([99, 12345], np.int32))
    assert e.value.code == ERR_UNSUPPORTED
    assert ex.num_variants == 1
    x = synth.pcm("noise", S, T, ex.n_in, fs)
    ex.set_fir_taps(S - 1, rows[S - 1:])                         # the table still takes rows
    y = ex.process(x)
    check_streams(oracle_lib, y, ex, lambda s: own_program(base, tw, rows[s]), x, 2, fs, range(S))


def test_multi_device_host_rows(oracle_lib):
    import torch
    fs, S, T = 48000, 40, 300
    base = fir_program(2, [[taps(120, 2, 3)], [taps(70, 2, 4)]])
    tw = fir_tap_words(base, 2)
    rows = impulse_rows(base, tw, S, 2, seed=19)
    ndev = torch.cuda.device_count()
    old = os.environ.get("AVDSP_B200_MULTI_REPLICATE")
    if ndev < 2:
        os.environ["AVDSP_B200_MULTI_REPLICATE"] = "2"           # two shards on the one GPU there is
    try:
        ex = Executor(base, fs, 2, S, seeds=np.arange(S, dtype=np.int32), dither=31, devices=list(range(min(ndev, 4))))
    finally:
        if old is None:
            os.environ.pop("AVDSP_B200_MULTI_REPLICATE", None)
        else:
            os.environ["AVDSP_B200_MULTI_REPLICATE"] = old
    assert ex.n_devices >= 2
    with pytest.raises(AvdspError) as e:
        ex.set_fir_taps(0, torch.from_numpy(rows).cuda())
    assert e.value.code == ERR_UNSUPPORTED
    ex.set_fir_taps(3, rows[3:])
    x = synth.pcm("noise", S, T, ex.n_in, fs)
    y = ex.process(x)
    check_streams(oracle_lib, y, ex, lambda s: own_program(base, tw, rows[s]) if s >= 3 else base, x, 2, fs, range(S))


def test_per_stream_tensor_core_rows_change_between_calls(oracle_lib):
    """the per-stream tensor-core form rebuilds its Toeplitz planes after set_fir_taps and set_param on a tap word, and a ragged
    call length (not a multiple of 8192) runs through its padded last block group"""
    fs, S, T1, T2 = 48000, 96, 8192 + 300, 9000
    base = fir_program(2, [[taps(700, 2, 21)], [taps(300, 2, 22)]])
    tw = fir_tap_words(base, 2)
    rows = impulse_rows(base, tw, S, 2, seed=23)
    rows2 = impulse_rows(base, tw, S, 2, seed=24)
    ex = make(base, fs, 2, S)
    ex.set_fir_taps(0, rows)
    x = synth.pcm("noise", S, T1 + T2, ex.n_in, fs)
    ya = ex.process(x[:, :T1])
    assert ex.last_kernel == "fir_tc"
    ex.set_fir_taps(0, rows2)
    ex.set_param(5, 3, int(tw[7]), np.array([1 << 27], np.int32))
    rows2[5:8, 7] = 1 << 27
    yb = ex.process(x[:, T1:])
    assert ex.last_kernel == "fir_tc"
    y = np.concatenate([ya, yb], axis=1)
    for s in range(S):
        o = oracle_lib.Oracle(own_program(base, tw, rows[s]), 2, fs, seed=s, dither=31)
        r = [o.process(x[s, :T1])]
        o.code[: len(base)] = own_program(base, tw, rows2[s])
        r.append(o.process(x[s, T1:]))
        assert np.array_equal(y[s], np.concatenate(r)), s
        assert np.array_equal(ex.get_state(s)[: ex.data_size], o.data), s


def test_float_table_refuses_the_tf32_tensor_core_form():
    fs, S = 48000, 8
    base = fir_program(3, [[taps(300, 3, 1)], [taps(260, 3, 2)]])
    ex = make(base, fs, 3, S)
    ex.set_fir_taps(0, impulse_rows(base, fir_tap_words(base, 3), S, 3, seed=3))
    ex.set_kernel(KERNEL_FIR_TC)
    st0 = [ex.get_state(s).copy() for s in range(S)]
    with pytest.raises(AvdspError) as e:
        ex.process(synth.pcm("noise", S, 9000, ex.n_in, fs))
    assert e.value.code == ERR_UNSUPPORTED
    assert all(np.array_equal(ex.get_state(s), st0[s]) for s in range(S))
