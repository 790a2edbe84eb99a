"""Host side of the per-stream coefficient table (avdsp_b200_coef_words): which program words are biquad coefficients, in the
column order avdsp_b200_set_coefs takes.  Checked against the wire layout walked independently with oracle/wire.py.  No CUDA
device needed."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_program
import avdsp_b200
from avdsp_b200 import params
from oracle import wire


def wire_coef_words(words):
    """b0 b1 b2 a1 a2 of every section of every BIQUADS parameter block, every fs column (dsp_runtime.c:827-849 reads column
    fsRel at h + 5 + 6 * fsRel of each section; sections are 2 + 6 * nFreq words apart), bypassed blocks included"""
    w = np.asarray(words).view(np.uint32)
    hd = wire.header(w)
    nf = hd["freqMax"] - hd["freqMin"] + 1
    out = set()
    for p, op, skip in wire.walk(w):
        if op != wire.OP["BIQUADS"] or skip < 3:
            continue
        h = p + int(np.int32(w[p + 2]))
        num = int(np.int16(w[h] & 0xFFFF))
        for s in range(max(num, 0)):
            for f in range(nf):
                for q in range(5):
                    out.add(h + 5 + 6 * f + s * (2 + 6 * nf) + q)
    return np.array(sorted(out), dtype=np.int32)


FIXTURES = [("c2_testrpi_xover_f2_192k", 2), ("c2_testrpi_xover_f2_multifs", 2), ("c3_peq16_f2_48k", 2), ("c3_peq16_f3_48k", 3),
            ("c3_peq16_f4_48k", 4), ("c3_peq16_f5_48k", 5), ("c3_peq16_f6_48k", 6), ("c1_crossover2x2lfe_f2_48k", 2),
            ("ref_crossoverLV6", 2), ("ref_dacdiy1", 2), ("ref_dacfabriceo", 2), ("ref_lxmini_lr2", 2), ("ref_lxmini_lv8", 2),
            ("ref_win_mydspcode", 2)]


@pytest.mark.parametrize("name,fmt", FIXTURES)
def test_coef_words_follow_the_wire_layout(name, fmt):
    w = load_program(name)
    got = avdsp_b200.coef_words(w, fmt)
    ref = wire_coef_words(w)
    assert ref.size > 0
    assert np.array_equal(got, ref)
    assert np.all(np.diff(got) > 0)                          # ascending, each word once


def test_multirate_program_lists_every_fs_column():
    w = load_program("c2_testrpi_xover_f2_multifs")
    hd = wire.header(w.view(np.uint32))
    nf = hd["freqMax"] - hd["freqMin"] + 1
    assert nf > 1
    single = wire_coef_words(load_program("c2_testrpi_xover_f2_192k"))
    assert avdsp_b200.coef_words(w, 2).size == nf * single.size


def _two_way(bypass_hi=1, share=False, fmt=2, fmin=48000, fmax=48000):
    a = wire.Asm(fmt=fmt, fmin=fmin, fmax=fmax)
    nf = wire.freq_index(fmax) - wire.freq_index(fmin) + 1
    a.core()
    a.param()
    lo = a.biquad_sections([[(0.1, 0.2, 0.1, 1.5, -0.6)] * nf, [(0.2, 0.1, 0.05, 1.2, -0.4)] * nf])
    hi = lo if share else a.biquad_sections([[(0.3, -0.6, 0.3, 1.4, -0.5)] * nf], bypass_flag=bypass_hi)
    a.load(0)
    a.biquads(lo)
    a.sat0db()
    a.store(0)
    a.load(1)
    a.biquads(hi)
    a.sat0db()
    a.store(1)
    return a.end(), lo, hi, nf


def test_bypassed_block_is_listed():
    w, lo, hi, nf = _two_way(bypass_hi=0)
    got = avdsp_b200.coef_words(w, 2)
    assert np.array_equal(got, wire_coef_words(w))
    assert got.size == 5 * 3 * nf
    assert all(hi + 5 + q in got for q in range(5))            # the bypassed section's words


def test_shared_parameter_block_is_listed_once():
    w, lo, hi, nf = _two_way(share=True, fmin=44100, fmax=96000)
    assert lo == hi
    got = avdsp_b200.coef_words(w, 2)
    assert got.size == 5 * 2 * nf                               # two sections, every fs column, once
    assert np.array_equal(got, wire_coef_words(w))


def test_dump_file_biquad_symbols_land_on_listed_words():
    w = load_program("c1_crossover2x2lfe_f2_48k")
    table = params.load_dump(os.path.join(GOLDEN, "programs", "c1_crossover2x2lfe_f2_48k.dump"))
    listed = set(avdsp_b200.coef_words(w, 2).tolist())
    hd = wire.header(w.view(np.uint32))
    nf = hd["freqMax"] - hd["freqMin"] + 1
    n_blocks = 0
    for sym in table.values():
        h = params.word_index(w, sym)
        if sym.size < 2 or h >= len(w) or (int(w[h]) >> 16) != wire.OP["BIQUADS"]:
            continue                                            # (one-word symbols, such as the header's format word)
        n_blocks += 1
        num = int(w[h]) & 0xFFFF
        for s in range(num):
            for f in range(nf):
                assert {h + 5 + 6 * f + s * (2 + 6 * nf) + q for q in range(5)} <= listed, sym.name
    assert n_blocks > 0


@pytest.mark.parametrize("name,fmt", [("c4_fir4096_f2_48k", 2), ("c4_fir4096_f3_48k", 3), ("c5_mixer8x8_f2_192k", 2),
                                      ("allops_gen_f2_multifs", 2), ("allops_misc_f5_multifs", 5)])
def test_programs_without_biquads_have_no_columns(name, fmt):
    w = load_program(name)
    assert wire_coef_words(w).size == 0
    assert avdsp_b200.coef_words(w, fmt).size == 0


def _describe_code(w, fs, fmt):
    with pytest.raises(avdsp_b200.AvdspError) as e:
        avdsp_b200.describe(w, fs, fmt)
    return e.value.code


def _coef_code(w, fmt):
    with pytest.raises(avdsp_b200.AvdspError) as e:
        avdsp_b200.coef_words(w, fmt)
    return e.value.code


def test_malformed_programs_return_the_codes_of_describe():
    w = load_program("c2_testrpi_xover_f2_192k")
    cases = []
    v = w.copy(); v[3] ^= 1; cases.append((v, 2))                              # checksum
    cases.append((w[:8].copy(), 2))                                            # shorter than its header says
    cases.append((w.copy(), 3))                                                # encoded for another DSP_FORMAT
    cases.append((w.copy(), 9))                                                # no such format
    v = w.copy(); v[0] = 0; cases.append((v, 2))                               # no header
    cases.append((load_program("old_rpi_testrew"), 2))                         # encoder 0x100
    v = w.copy()
    p = [p for p, op, _ in wire.walk(v.view(np.uint32)) if op == wire.OP["BIQUADS"]][0]
    v[p + 2] = 1 << 30                                                          # parameter block outside the program
    cases.append((v, 2))
    for v, fmt in cases:
        code = _coef_code(v, fmt)
        assert code < 0
        assert code == _describe_code(v, 192000, fmt)


def test_output_buffer_is_bounded():
    import ctypes as C
    w = load_program("c3_peq16_f2_48k")
    n = avdsp_b200.coef_words(w, 2).size
    buf = (C.c_int32 * 4)(*([-7] * 4))
    L = avdsp_b200._lib.lib()
    assert L.avdsp_b200_coef_words(w.ctypes.data, len(w), 2, buf, 3) == n
    assert list(buf)[3] == -7                                   # wrote maxOut words, not more
    assert L.avdsp_b200_coef_words(w.ctypes.data, len(w), 2, None, 5) == -9
