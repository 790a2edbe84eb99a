"""Host side of the per-stream FIR table (avdsp_b200_fir_tap_words): which program words are FIR taps, in the column order
avdsp_b200_set_fir_taps takes.  Checked against the wire layout walked independently with oracle/wire.py.  No CUDA device needed."""
import ctypes as C

import numpy as np
import pytest

from conftest import load_program
import avdsp_b200
from oracle import wire


def wire_fir_tap_words(words):
    """t + 1 .. t + lw of every DSP_FIR entry, every fs column, whose length word lw is a convolution (lw > 0, lw >> 16 == 0;
    dsp_runtime.c:928-969: the opcode holds one relative pointer per fs column, 0 = skipped, then the data offset)"""
    w = np.asarray(words).view(np.uint32)
    hd = wire.header(w)
    nf = hd["freqMax"] - hd["freqMin"] + 1
    out = set()
    for p, op, skip in wire.walk(w):
        if op != wire.OP["FIR"]:
            continue
        for f in range(nf):
            rel = int(np.int32(w[p + 1 + f]))
            if rel == 0:
                continue
            lw = int(np.int32(w[p + rel]))
            if lw > 0 and (lw >> 16) == 0:
                out.update(range(p + rel + 1, p + rel + 1 + lw))
    return np.array(sorted(out), dtype=np.int32)


def fir_program(fmt, imps_per_core, fmin=48000, fmax=48000, shared=False, biquad=False):
    """one core per entry of imps_per_core: LOAD -> FIR -> SAT0DB -> STORE; shared=True: the second core's FIR points at the
    first core's impulse block; biquad=True: a BIQUADS cascade after the FIR of core 0"""
    a = wire.Asm(fmt=fmt, fmin=fmin, fmax=fmax)
    where0 = None
    for k, imps in enumerate(imps_per_core):
        a.core()
        a.param()
        where = where0 if (shared and k > 0) else a.fir_impulses(imps)
        bq = a.biquad_sections([[(0.1, 0.2, 0.1, 1.5, -0.6)] * a.nf]) if (biquad and k == 0) else None
        where0 = where0 or where
        mx = max([(l[1] + 1) if isinstance(l, tuple) else (len(l) if l is not None else 0) for l in imps] + [1])
        a.load(8 + k)
        a.fir(where, mx)
        if bq is not None:
            a.biquads(bq)
        a.sat0db()
        a.store(k)
    return a.end()


def taps(n, fmt, seed):
    v = np.random.default_rng(seed).uniform(-0.1, 0.1, n)
    return [wire.q28(x) for x in v] if fmt == 2 else [float(x) for x in v]


@pytest.mark.parametrize("name,fmt", [("c4_fir4096_f2_48k", 2), ("c4_fir4096_f3_48k", 3), *[(f"c4s_fir_f{f}_multifs", f) for f in (2, 3, 4, 5, 6)]])
def test_fir_tap_words_follow_the_wire_layout(name, fmt):
    w = load_program(name)
    got = avdsp_b200.fir_tap_words(w, fmt)
    ref = wire_fir_tap_words(w)
    assert ref.size > 0
    assert np.array_equal(got, ref)
    assert np.all(np.diff(got) > 0)                          # ascending, each word once


def test_c4_lists_both_paths():
    assert avdsp_b200.fir_tap_words(load_program("c4_fir4096_f2_48k"), 2).size == 2 * 4096


def test_plain_delay_and_skipped_entries_contribute_nothing():
    # c4s: 48k convolutions of 100 and 33 taps; 96k: channel 0 a plain delay, channel 1 skipped (make_golden.fir_program)
    w = load_program("c4s_fir_f2_multifs")
    assert avdsp_b200.fir_tap_words(w, 2).size == 100 + 33


def test_multirate_program_lists_every_fs_column():
    imps = [[taps(20, 2, 1), taps(7, 2, 2), ("delay", 5)], [None, taps(11, 2, 3), taps(3, 2, 4)]]
    w = fir_program(2, imps, fmin=48000, fmax=96000)
    got = avdsp_b200.fir_tap_words(w, 2)
    assert got.size == 20 + 7 + 11 + 3
    assert np.array_equal(got, wire_fir_tap_words(w))


def test_shared_tap_block_is_listed_once():
    imps = [[taps(24, 3, 5)], [taps(24, 3, 5)]]
    w = fir_program(3, imps, shared=True)
    fir_ops = [p for p, op, _ in wire.walk(w.view(np.uint32)) if op == wire.OP["FIR"]]
    assert len(fir_ops) == 2
    assert fir_ops[0] + int(w[fir_ops[0] + 1]) == fir_ops[1] + int(w[fir_ops[1] + 1])     # one block, two opcodes
    got = avdsp_b200.fir_tap_words(w, 3)
    assert got.size == 24
    assert np.array_equal(got, wire_fir_tap_words(w))


@pytest.mark.parametrize("fmt", [2, 3, 4])
def test_fir_and_biquad_programs_keep_the_two_lists_apart(fmt):
    w = fir_program(fmt, [[taps(16, fmt, 6)], [taps(9, fmt, 7)]], biquad=True)
    fw, cw = avdsp_b200.fir_tap_words(w, fmt), avdsp_b200.coef_words(w, fmt)
    assert fw.size == 25 and cw.size == 5
    assert np.array_equal(fw, wire_fir_tap_words(w))
    assert not set(fw.tolist()) & set(cw.tolist())


@pytest.mark.parametrize("name,fmt", [("c2_testrpi_xover_f2_192k", 2), ("c3_peq16_f3_48k", 3), ("c5_mixer8x8_f2_192k", 2)])
def test_programs_without_fir_have_no_columns(name, fmt):
    w = load_program(name)
    assert wire_fir_tap_words(w).size == 0
    assert avdsp_b200.fir_tap_words(w, fmt).size == 0


def _code(fn, *a):
    with pytest.raises(avdsp_b200.AvdspError) as e:
        fn(*a)
    return e.value.code


def test_malformed_programs_return_the_codes_of_describe():
    w = load_program("c4_fir4096_f2_48k")
    cases = []
    v = w.copy(); v[3] ^= 1; cases.append((v, 2))                              # checksum
    cases.append((w[:8].copy(), 2))                                            # shorter than its header says
    cases.append((w.copy(), 3))                                                # encoded for another DSP_FORMAT
    cases.append((w.copy(), 1))                                                # no such format
    v = w.copy(); v[0] = 0; cases.append((v, 2))                               # no header
    v = w.copy()
    p = [p for p, op, _ in wire.walk(v.view(np.uint32)) if op == wire.OP["FIR"]][0]
    v[p + 1] = 1 << 30                                                          # impulse outside the program
    cases.append((v, 2))
    for v, fmt in cases:
        code = _code(avdsp_b200.fir_tap_words, v, fmt)
        assert code < 0
        assert code == _code(avdsp_b200.describe, v, 48000, fmt)


def test_output_buffer_is_bounded():
    w = load_program("c4s_fir_f3_multifs")
    n = avdsp_b200.fir_tap_words(w, 3).size
    buf = (C.c_int32 * 4)(*([-7] * 4))
    L = avdsp_b200._lib.lib()
    assert L.avdsp_b200_fir_tap_words(w.ctypes.data, len(w), 3, buf, 3) == n
    assert list(buf)[3] == -7                                   # wrote maxOut words, not more
    assert list(buf)[:3] == avdsp_b200.fir_tap_words(w, 3)[:3].tolist()
    assert L.avdsp_b200_fir_tap_words(w.ctypes.data, len(w), 3, None, 5) == -9


def test_every_rate_is_validated():
    """a tap block that runs past the program in an fs column other than the lowest: the column list would be partial, so the
    call returns the code describe returns at that rate"""
    imps = [[taps(20, 2, 1), taps(7, 2, 2), taps(9, 2, 3)], [taps(11, 2, 4), None, None]]
    w = fir_program(2, imps, fmin=48000, fmax=96000)
    p = [p for p, op, _ in wire.walk(w.view(np.uint32)) if op == wire.OP["FIR"]][0]
    t = p + int(w[p + 3])                                       # the 96k entry's length word
    assert int(w[t]) == 9
    w[t] = 60000                                               # a convolution (lw >> 16 == 0) longer than the program
    assert _code(avdsp_b200.describe, w, 96000, 2) < 0
    assert _code(avdsp_b200.fir_tap_words, w, 2) == _code(avdsp_b200.describe, w, 96000, 2)
    avdsp_b200.describe(w, 48000, 2)                            # the lowest rate alone lowers
