"""Per-stream PARAM overrides (SURVEY.md 8f-3): avdsp_b200_set_param gives every stream (every room of a multi-room host) its
own crossover / EQ / delay / gain inside ONE instance; the dump-file symbol table of the reference's dspcreate
(encoder/dsp_encoder.c:476-503) names the words.  Checked against one oracle instance per stream running that stream's
own program."""
import math
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_program
from avdsp_b200 import Executor, AvdspError, synth, params, coef_words, KERNEL_GENERIC, KERNEL_AUTO
from oracle import wire

pytestmark = pytest.mark.gpu


def lowpass(fs, f, q=0.7071):
    w0 = 2 * math.pi * f / fs
    al, c = math.sin(w0) / 2 / q, math.cos(w0)
    a0 = 1 + al
    return ((1 - c) / 2 / a0, (1 - c) / a0, (1 - c) / 2 / a0, 2 * c / a0, -(1 - al) / a0)


def highpass(fs, f, q=0.7071):
    w0 = 2 * math.pi * f / fs
    al, c = math.sin(w0) / 2 / q, math.cos(w0)
    a0 = 1 + al
    return ((1 + c) / 2 / a0, -(1 + c) / a0, (1 + c) / 2 / a0, 2 * c / a0, -(1 - al) / a0)


def crossover_program(fx, us, gain, fs=48000, fmt=2):
    """2-way LR4 crossover at fx Hz, the tweeter delayed by `us` microseconds, woofer gain `gain`; always the same opcodes"""
    a = wire.Asm(fmt=fmt, fmin=fs, fmax=fs)
    a.core()
    a.tpdf_calc(24)
    a.param()
    lo = a.biquad_sections([[lowpass(fs, fx)], [lowpass(fs, fx)], [wire.rbj_peak(fs, fx / 2, 1.2, 1.3)]])
    hi = a.biquad_sections([[highpass(fs, fx)], [highpass(fs, fx)]])
    dl = a.delay_param(2000, us, fs)
    g = a.num(gain)
    a.load_gain(8, 0.9)
    a.biquads(lo)
    a.gain(addr=g)
    a.sat0db()
    a.store(0)
    a.load_gain(8, 0.9)
    a.biquads(hi)
    a.sat0db_tpdf()
    a.delay(dl)
    a.store(1)
    return a.end()


def apply_diff(ex, first, n, base, prog):
    """hand the words that differ from the loaded program over as contiguous runs"""
    d = np.nonzero(base != prog)[0]
    assert d.size
    runs = np.split(d, np.nonzero(np.diff(d) != 1)[0] + 1)
    for r in runs:
        ex.set_param(first, n, int(r[0]), prog[r[0]: r[-1] + 1])


@pytest.mark.parametrize("fmt", [2, 3])
@pytest.mark.parametrize("kernel", [KERNEL_AUTO, KERNEL_GENERIC])
def test_64_streams_64_crossovers(oracle_lib, kernel, fmt):
    fs, S, T = 48000, 64, 600
    progs = [crossover_program(200.0 * 1.06 ** s, 100 + 25 * s, 0.5 + 0.005 * s, fs, fmt) for s in range(S)]
    assert all(p.shape == progs[0].shape for p in progs)
    ops = [(i, op) for i, op, _ in wire.walk(progs[0].view(np.uint32))]
    assert all([(i, op) for i, op, _ in wire.walk(p.view(np.uint32))] == ops for p in progs)      # same structure
    seeds = np.arange(S, dtype=np.int32)
    ex = Executor(progs[0], fs, fmt, S, seeds=seeds, dither=24)
    ex.set_kernel(kernel)
    x = synth.pcm("full", S, T, ex.n_in, fs)
    ya = ex.process(x[:, :200])                      # everybody on stream 0's crossover first
    for s in range(1, S):
        apply_diff(ex, s, 1, progs[0], progs[s])
    assert ex.num_variants == S
    yb = ex.process(x[:, 200:])                      # state carries over, parameters differ from here on
    y = np.concatenate([ya, yb], axis=1)
    for s in range(S):
        o = oracle_lib.Oracle(progs[0], fmt, fs, seed=s, dither=24)
        ref_a = o.process(x[s, :200])
        # the oracle instance of stream s gets its own PARAM words at the same moment (the reference re-reads the program every frame)
        o.code[:] = np.where(np.arange(len(o.code)) < len(progs[s]), progs[s][: len(o.code)], o.code)
        ref_b = o.process(x[s, 200:])
        assert np.array_equal(y[s], np.concatenate([ref_a, ref_b])), s
        assert np.array_equal(ex.get_state(s)[: ex.data_size], o.data), s
    assert ex.last_kernel == ("generic" if kernel == KERNEL_GENERIC else "chain")


def test_rooms_share_variants_and_overrides_are_cumulative(oracle_lib):
    fs, S, T = 48000, 96, 300
    base = crossover_program(300.0, 200, 0.5, fs)
    room_b = crossover_program(1200.0, 200, 0.5, fs)            # other crossover
    room_c = crossover_program(1200.0, 700, 0.25, fs)           # ... and other delay + gain on top
    ex = Executor(base, fs, 2, S, dither=31)
    apply_diff(ex, 32, 64, base, room_b)                        # streams 32..95
    assert ex.num_variants == 2
    apply_diff(ex, 64, 32, room_b, room_c)                      # cumulative: 64..95 move on from room_b's words
    assert ex.num_variants == 3
    x = synth.pcm("noise", S, T, ex.n_in, fs)
    l0 = ex.launch_count
    y = ex.process(x)
    assert ex.launch_count - l0 == 3                            # one launch per run of neighbours sharing a parameter set
    for s, prog in ((0, base), (31, base), (32, room_b), (63, room_b), (64, room_c), (95, room_c)):
        assert np.array_equal(y[s], oracle_lib.Oracle(prog, 2, fs, seed=0, dither=31).process(x[s])), s
    # back to the loaded program: the variant is released
    apply_diff(ex, 64, 32, room_c, base)
    assert ex.num_variants == 2
    # reload_params = a new program for everybody, overrides start over
    ex.reload_params(room_c)
    assert ex.num_variants == 1
    # an override may not touch opcode words
    with pytest.raises(AvdspError):
        ex.set_param(0, 1, 12, [0])


def test_dump_file_symbols_on_c1(oracle_lib):
    """crossover2x2lfe with the symbol table dspcreate -dumpfile wrote for it: another delay and a bypassed EQ for one stream"""
    w = load_program("c1_crossover2x2lfe_f2_48k")
    table = params.load_dump(os.path.join(GOLDEN, "programs", "c1_crossover2x2lfe_f2_48k.dump"))
    fs, S, T = 48000, 5, 400
    ex = Executor(w, fs, 2, S, seeds=np.arange(S, dtype=np.int32), dither=24)
    d = table["DELAY_HIGH_LOW_1"]
    assert ex.param_index(d.offset, d.param_num) == params.word_index(w, d)
    wd = params.word_index(w, d)
    wq = params.word_index(w, table["BQ4_EQ_LFE_-1"])
    assert (int(w[wq]) >> 16) == wire.OP["BIQUADS"] and int(w[wq + 1]) == 1
    mine = w.copy()
    mine[wd] = (int(w[wd]) & ~0xFFFF) | 1100                     # 1100 us instead of the default
    mine[wq + 1] = 0                                             # bypass flag of the LFE EQ (dsp_runtime.c:838)
    ex.set_param(3, 1, wd, mine[wd: wd + 1])
    ex.set_param(3, 1, wq + 1, [0])
    x = synth.pcm("noise", S, T, ex.n_in, fs)
    y = ex.process(x)
    for s in range(S):
        o = oracle_lib.Oracle(mine if s == 3 else w, 2, fs, seed=s, dither=24)
        assert np.array_equal(y[s], o.process(x[s])), s
    assert not np.array_equal(y[3], oracle_lib.Oracle(w, 2, fs, seed=3, dither=24).process(x[3]))


def test_reset_to_another_rate_replans_every_variant(oracle_lib):
    """three blocks of streams on three parameter sets (the loaded program and two variants), reset through the lowest, the
    highest and again the lowest rate of a multi-rate program: every variant's plans follow the rate"""
    base = load_program("c2_testrpi_xover_f2_multifs")
    hd = wire.header(base.view(np.uint32))
    lo, hi = wire.FREQS[hd["freqMin"]], wire.FREQS[hd["freqMax"]]
    S, T, blk = 24, 400, 8
    cw = coef_words(base, 2)
    ff = cw[(np.arange(len(cw)) % 5 < 3) & (base[cw] != 0)]         # b0 b1 b2 of every section, every fs column
    rng = np.random.default_rng(29)
    progs = [base]
    for _ in range(2):
        p = base.copy()
        p[ff] += rng.integers(-64, 65, len(ff)).astype(np.int32)
        progs.append(p)
    seeds = np.arange(S, dtype=np.int32)
    ex = Executor(base, hi, 2, S, seeds=seeds, dither=24)
    for b in (1, 2):
        apply_diff(ex, b * blk, blk, base, progs[b])
    assert ex.num_variants == 3
    for fs in (lo, hi, lo):
        ex.reset(fs, seeds=seeds, dither=24)
        assert ex.num_variants == 3
        x = synth.pcm("noise", S, T, ex.n_in, fs)
        y = ex.process(x)
        for s in range(S):
            o = oracle_lib.Oracle(progs[s // blk], 2, fs, seed=s, dither=24)
            assert np.array_equal(y[s], o.process(x[s])), (fs, s)
            assert np.array_equal(ex.get_state(s)[: ex.data_size], o.data), (fs, s)
