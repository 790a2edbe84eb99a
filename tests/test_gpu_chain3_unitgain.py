"""k_chain3's unit-gain form (kernel_chain3.cu unitStep, DESIGN.md 4.2a): a part whose sections all satisfy b0 = 2^28,
b1 + a1 = -2^28, b2 + a2 = 0 runs two MACs per section on a shifted accumulator.  Against the CPU oracle, bit for bit: outputs and
state words.  The first two tests are host-only (avdsp_b200_describe)."""
import re

import numpy as np
import pytest

from conftest import load_program
import avdsp_b200
from avdsp_b200 import Executor, synth, coef_words, KERNEL_GENERIC, KERNEL_CHAIN_V3

C2, FS = "c2_testrpi_xover_f2_192k", 192000


def _v3_parts(trace):
    ln = [ln for ln in trace.splitlines() if ln.startswith("chain kernel v3 geometry")][0]
    parts = re.findall(r" (\d+):(\d+)\+(\d+)@(\d+)(u?)", ln.split("parts (chain:first+n@base):")[1].split(";")[0])
    macs = re.search(r"(\d+) IMAD.WIDE per frame executed, (\d+) algorithmic", ln)
    return [(int(c), int(f), int(n), u == "u") for c, f, n, _, u in parts], int(macs.group(1)), int(macs.group(2))


def test_c2_runs_22_sections_in_the_unit_gain_form():
    parts, macs, alg = _v3_parts(avdsp_b200.describe(load_program(C2), FS, 2, n_streams=4096, num_sms=148))
    unit = [p for p in parts if p[3]]
    assert sum(n for _, _, n, _ in unit) == 22
    assert all(n in (3, 4) for _, _, n, _ in unit)
    assert (macs, alg) == (240 - 3 * 22, 240)


@pytest.mark.parametrize("col", [0, 1, 2, 3, 4])
def test_one_lsb_off_the_identity_leaves_the_general_form(col):
    """b0, b1, b2, a1 or a2 of the first section one LSB off: the two 4-section parts that run it (one per channel) go general"""
    w = load_program(C2).copy()
    cw = coef_words(w, 2)
    w[cw[col]] += 1
    parts, macs, alg = _v3_parts(avdsp_b200.describe(w, FS, 2, n_streams=4096, num_sms=148))
    assert sum(n for _, _, n, u in parts if u) == 22 - 8
    assert (macs, alg) == (240 - 3 * 14, 240)


def _unit_rows(base, cw, n, seed):
    """n distinct coefficient rows for C2: the unit-gain sections get random stable poles (a1, a2) and the words that keep the
    identity (b1 = -2^28 - a1, b2 = -a2); the other sections keep the program's words"""
    rng = np.random.default_rng(seed)
    v = base[cw].astype(np.int64).reshape(-1, 5)
    unit = (v[:, 0] == 1 << 28) & (v[:, 1] + v[:, 3] == -(1 << 28)) & (v[:, 2] + v[:, 4] == 0)
    rows = np.repeat(v[None], n, axis=0)
    r = rng.uniform(0.90, 0.999, (n, len(v)))
    th = rng.uniform(0.001, 0.3, (n, len(v)))
    a1 = np.round((2 * r * np.cos(th) - 1) * 2.0 ** 28).astype(np.int64)        # the reference's a1 word is 2^28 (a1 - 1)
    a2 = np.round(-r * r * 2.0 ** 28).astype(np.int64)
    rows[:, unit, 3], rows[:, unit, 4] = a1[:, unit], a2[:, unit]
    rows[:, unit, 1], rows[:, unit, 2] = -(1 << 28) - a1[:, unit], -a2[:, unit]
    return np.ascontiguousarray(rows.reshape(n, -1).astype(np.int32)), np.nonzero(unit)[0]


def _check(oracle_lib, ex, progs, x, y, seeds, dither, streams):
    for s in streams:
        o = oracle_lib.Oracle(progs(s), 2, FS, seed=int(seeds[s]), dither=dither)
        assert np.array_equal(y[s], o.process(x[s])), s
        assert np.array_equal(ex.get_state(s)[: ex.data_size], o.data), s


@pytest.mark.gpu
@pytest.mark.parametrize("stim", ["noise", "full"])
def test_c2_bench_geometry_distinct_streams(oracle_lib, stim):
    """The benchmark's geometry (4096 streams, 28 per CTA), every stream its own seed and input.  Full-scale input drives the unit
    parts' inputs past the x0 bound and sections into saturation: those tiles are replayed exactly."""
    base = load_program(C2)
    S, T = 4096, 300
    seeds = (np.arange(S, dtype=np.int32) * 7919) % 100003
    ex = Executor(base, FS, 2, S, seeds=seeds, dither=24)
    ex.set_kernel(KERNEL_CHAIN_V3)
    x = synth.pcm(stim, S, T, ex.n_in, FS)
    y = ex.process(x)
    assert ex.last_chain_variant == 3
    parts, _, _ = _v3_parts(ex.trace)
    assert sum(n for _, _, n, u in parts if u) == 22
    spots = np.unique(np.concatenate([np.arange(0, 64), np.linspace(0, S - 1, 40).astype(int)]))
    _check(oracle_lib, ex, lambda s: base, x, y, seeds, 24, spots)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2])
def test_random_unit_sections_and_one_lsb_misses_per_stream(oracle_lib, seed):
    """Per-stream tables, 5 streams per CTA: every stream gets random unit-gain sections; in every other CTA one stream's row
    misses the identity by one LSB (that CTA's warps run the general form).  A second call with full-scale input saturates
    sections; a set_param then puts the missing LSB back."""
    base = load_program(C2)
    cw = coef_words(base, 2)
    S, T = 40, 700
    rows, unit = _unit_rows(base, cw, S, seed)
    rng = np.random.default_rng(seed)
    miss = []
    for cta in range(0, S // 5, 2):
        s = 5 * cta + int(rng.integers(0, 5))
        col = 5 * int(rng.choice(unit)) + int(rng.integers(0, 5))
        rows[s, col] += 1 if rng.integers(0, 2) else -1
        miss.append((s, col))
    seeds = np.arange(S, dtype=np.int32) + 3
    ex = Executor(base, FS, 2, S, seeds=seeds, dither=24)
    ex.set_kernel(KERNEL_CHAIN_V3)
    ex.set_coefs(0, rows)

    def prog(r):
        p = base.copy()
        p[cw] = r
        return p

    orcs = [oracle_lib.Oracle(prog(rows[s]), 2, FS, seed=int(seeds[s]), dither=24) for s in range(S)]
    for stim in ("noise", "full"):
        x = synth.pcm(stim, S, T, ex.n_in, FS)
        y = ex.process(x)
        assert ex.last_chain_variant == 3
        for s in range(S):
            assert np.array_equal(y[s], orcs[s].process(x[s])), (stim, s)
    for s, col in miss:                                                   # back on the identity: that CTA runs the unit form again
        k, q = divmod(col, 5)
        r = rows[s].astype(np.int64).reshape(-1, 5)[k]
        good = {0: 1 << 28, 1: -(1 << 28) - r[3], 2: -r[4], 3: -(1 << 28) - r[1], 4: -r[2]}[q]
        ex.set_param(s, 1, int(cw[col]), [int(good)])
        orcs[s].code[cw[col]] = good
    x = synth.pcm("noise", S, T, ex.n_in, FS)
    y = ex.process(x)
    for s in range(S):
        assert np.array_equal(y[s], orcs[s].process(x[s])), s
        assert np.array_equal(ex.get_state(s)[: ex.data_size], orcs[s].data), s


@pytest.mark.gpu
def test_state_round_trip_through_odd_splits_and_a_foreign_state_block():
    """Calls that end in the middle of a unit part's tiles (odd frame counts), switches to the generic interpreter between calls,
    and a foreign state block (random accumulators and histories: residues far from zero, so the unit parts enter and leave
    the z form with large d) loaded into every stream: same outputs and state as the generic interpreter."""
    w = load_program(C2)
    S, T = 11, 1600
    rng = np.random.default_rng(7)
    x = synth.pcm("noise", S, T, 2, FS)
    seeds = np.arange(S, dtype=np.int32)
    a = Executor(w, FS, 2, S, seeds=seeds); a.set_kernel(KERNEL_GENERIC)
    b = Executor(w, FS, 2, S, seeds=seeds)
    blk = a.get_state(0)
    for s in range(S):
        st = blk.copy()
        st[2:50] = rng.integers(-2 ** 30, 2 ** 30, 48)         # accumulators and histories of the two UUUU cascades (core 1)
        a.set_state(s, st); b.set_state(s, st)
    cuts = [0, 1, 37, 100, 161, 333, 334, 700, 999, 1311, T]
    ya = a.process(x)
    parts = []
    for i, (c0, c1) in enumerate(zip(cuts, cuts[1:])):
        b.set_kernel(KERNEL_GENERIC if i == 4 else KERNEL_CHAIN_V3)
        parts.append(b.process(np.ascontiguousarray(x[:, c0:c1])))
        if i != 4:
            assert b.last_chain_variant == 3
    assert np.array_equal(ya, np.concatenate(parts, axis=1))
    for s in range(S):
        assert np.array_equal(a.get_state(s), b.get_state(s)), s

