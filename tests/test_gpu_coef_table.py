"""Per-stream coefficient tables (avdsp_b200_set_coefs): every stream its own crossover / EQ in one launch.  Every case is checked
against one oracle instance per stream running that stream's own program (the loaded words with its row patched in): outputs
and data area bit-exact."""
import os

import numpy as np
import pytest

from conftest import load_program
from avdsp_b200 import (Executor, AvdspError, synth, coef_words, KERNEL_AUTO, KERNEL_GENERIC, KERNEL_CHAIN_V2, KERNEL_CHAIN_V3,
                        KERNEL_DAG)
from oracle import wire
from test_gpu_params import crossover_program

pytestmark = pytest.mark.gpu

ERR_UNSUPPORTED, ERR_ARG = -8, -9


def pcm_for(fmt):
    return synth.pcm_float if fmt >= 5 else synth.pcm


def jitter(base, cw, n, fmt, seed, lsb=64, rel=1e-4, poles=False):
    """n distinct rows close to the program's own coefficients.  The feed-forward words b0 b1 b2 (columns come in groups of
    five, b0 b1 b2 a1 a2) move by up to `lsb` LSBs (Q4.28) or by a relative `rel` (float); with poles=True a1 and a2 move too,
    by at most 2 LSBs / 2 ulps, which keeps the program's stable filters stable"""
    rng = np.random.default_rng(seed)
    v = base[cw].astype(np.int32)
    nz = v[None, :] != 0
    ff = (np.arange(len(cw)) % 5 < 3)[None, :] & nz
    if fmt == 2:
        rows = v[None, :].astype(np.int64) + rng.integers(-lsb, lsb + 1, (n, len(cw)))
        rows = np.where(ff, rows, v[None, :]).astype(np.int32)
    else:
        f = v.view(np.float32).astype(np.float64)[None, :] * (1.0 + rng.uniform(-rel, rel, (n, len(cw))))
        rows = np.where(ff, f.astype(np.float32).view(np.int32), v[None, :]).astype(np.int32)
    if poles:                         # Q4.28 LSBs or float ulps: a step of the bit pattern either way
        fb = nz & ~ff & ((np.arange(len(cw)) % 5 >= 3)[None, :])
        rows = np.where(fb, rows.astype(np.int64) + rng.integers(-2, 3, rows.shape), rows).astype(np.int32)
    return np.ascontiguousarray(rows)


def own_program(base, cw, row):
    p = base.copy()
    p[cw] = row
    return p


def check_streams(oracle_lib, y, ex, progs_of, x, fmt, fs, seeds, dither, streams, switch=0, base=None):
    """stream s ran `base` for frames [0, switch), then progs_of(s)"""
    for s in streams:
        o = oracle_lib.Oracle(base if switch else progs_of(s), fmt, fs, seed=int(seeds[s]), dither=dither)
        parts = []
        if switch:
            parts.append(o.process(x[s, :switch]))
            p = progs_of(s)
            o.code[: len(p)] = p[: len(o.code)]
        parts.append(o.process(x[s, switch:]))
        assert np.array_equal(y[s], np.concatenate(parts)), s
        assert np.array_equal(ex.get_state(s)[: ex.data_size], o.data), s


@pytest.mark.parametrize("fmt", [2, 3, 5])
@pytest.mark.parametrize("kernel", [KERNEL_AUTO, KERNEL_CHAIN_V2, KERNEL_GENERIC])
def test_64_streams_64_crossovers_one_launch(oracle_lib, kernel, fmt):
    """64 rooms, 64 different crossover frequencies (every coefficient word differs); the GAIN behind the low-pass keeps this
    program off k_chain3, which test_chain3_full_rows covers"""
    fs, S, T, cut = 48000, 64, 600, 200
    progs = [crossover_program(200.0 * 1.06 ** s, 300, 0.5, fs, fmt) for s in range(S)]
    base = progs[0]
    cw = coef_words(base, fmt)
    others = np.ones(len(base), bool)
    others[cw] = False
    assert all(np.array_equal(p[others], base[others]) for p in progs)      # only coefficient words differ
    rows = np.stack([p[cw] for p in progs])
    seeds = np.arange(S, dtype=np.int32)
    ex = Executor(base, fs, fmt, S, seeds=seeds, dither=24)
    ex.set_kernel(kernel)
    x = pcm_for(fmt)("full", S, T, ex.n_in, fs)
    l0 = ex.launch_count
    ya = ex.process(x[:, :cut])
    plain = ex.launch_count - l0
    kern, variant = ex.last_kernel, ex.last_chain_variant
    ex.set_coefs(0, rows)
    l1 = ex.launch_count
    yb = ex.process(x[:, cut:])
    assert ex.launch_count - l1 == plain                        # 64 distinct crossovers: the launches of one parameter set
    assert ex.num_variants == 1
    assert (ex.last_kernel, ex.last_chain_variant) == (kern, variant)
    y = np.concatenate([ya, yb], axis=1)
    check_streams(oracle_lib, y, ex, lambda s: progs[s], x, fmt, fs, seeds, 24, range(S), switch=cut, base=base)


@pytest.mark.parametrize("name,fmt", [("c3_peq16_f2_48k", 2), ("c3_peq16_f3_48k", 3), ("c3_peq16_f5_48k", 5),
                                      ("c2_testrpi_xover_f2_192k", 2)])
def test_chain3_full_rows(oracle_lib, name, fmt):
    """k_chain3 (fixed point and float class) with every row distinct in all five words of every section, switched in
    between two calls: the launches of one parameter set, the same kernel, bit-exact"""
    fs = 192000 if name.startswith("c2") else 48000
    S, T, cut = 256, 700, 300
    base = load_program(name)
    cw = coef_words(base, fmt)
    rows = jitter(base, cw, S, fmt, seed=41 + fmt, poles=True)
    assert len(np.unique(rows, axis=0)) == S
    fb = np.arange(len(cw)) % 5 >= 3
    assert (rows[:, fb] != base[cw][fb]).any(axis=0).sum() > fb.sum() // 2      # most a1 / a2 columns differ somewhere
    seeds = np.arange(S, dtype=np.int32)
    ex = Executor(base, fs, fmt, S, seeds=seeds, dither=24)
    ex.set_kernel(KERNEL_CHAIN_V3)
    x = pcm_for(fmt)("noise", S, T, ex.n_in, fs)
    l0 = ex.launch_count
    ya = ex.process(x[:, :cut])
    plain = ex.launch_count - l0
    assert ex.last_chain_variant == 3
    ex.set_coefs(0, rows)
    l1 = ex.launch_count
    yb = ex.process(x[:, cut:])
    assert ex.launch_count - l1 == plain and ex.last_chain_variant == 3 and ex.num_variants == 1
    y = np.concatenate([ya, yb], axis=1)
    check_streams(oracle_lib, y, ex, lambda s: own_program(base, cw, rows[s]), x, fmt, fs, seeds, 24, range(S), switch=cut,
                  base=base)


@pytest.mark.parametrize("name,fmt,kernel", [("c3_peq16_f4_48k", 4, KERNEL_AUTO), ("c3_peq16_f6_48k", 6, KERNEL_AUTO),
                                             ("c3_peq16_f5_48k", 5, KERNEL_AUTO), ("c3_peq16_f3_48k", 3, KERNEL_AUTO),
                                             ("c3_peq16_f2_48k", 2, KERNEL_AUTO), ("c3_peq16_f5_48k", 5, KERNEL_GENERIC)])
def test_peq_rows_every_format(oracle_lib, name, fmt, kernel):
    fs, S, T = 48000, 40, 400
    base = load_program(name)
    cw = coef_words(base, fmt)
    rows = jitter(base, cw, S, fmt, seed=fmt)
    seeds = np.arange(S, dtype=np.int32)
    ex = Executor(base, fs, fmt, S, seeds=seeds, dither=24)
    ex.set_kernel(kernel)
    ex.set_coefs(0, rows)
    x = pcm_for(fmt)("noise", S, T, ex.n_in, fs)
    y = ex.process(x)
    if fmt in (4, 6) or kernel == KERNEL_GENERIC:
        assert ex.last_kernel == "generic"
    check_streams(oracle_lib, y, ex, lambda s: own_program(base, cw, rows[s]), x, fmt, fs, seeds, 24, range(S))


@pytest.mark.parametrize("name,fs", [("c1_crossover2x2lfe_f2_48k", 48000), ("ref_crossoverLV6", 96000)])
def test_dag_rows(oracle_lib, name, fs):
    S, T = 48, 500
    base = load_program(name)
    cw = coef_words(base, 2)
    rows = jitter(base, cw, S, 2, seed=7)
    seeds = np.arange(S, dtype=np.int32)
    ex = Executor(base, fs, 2, S, seeds=seeds, dither=24)
    ex.set_kernel(KERNEL_DAG)
    ex.set_coefs(0, rows)
    x = synth.pcm("full", S, T, ex.n_in, fs)
    y = ex.process(x)
    assert ex.last_kernel == "dag"
    check_streams(oracle_lib, y, ex, lambda s: own_program(base, cw, rows[s]), x, 2, fs, seeds, 24, range(S))


def test_c2_4096_streams_all_rows_distinct_on_chain3(oracle_lib):
    fs, S, T = 192000, 4096, 2048
    base = load_program("c2_testrpi_xover_f2_192k")
    cw = coef_words(base, 2)
    rows = jitter(base, cw, S, 2, seed=11)
    assert len(np.unique(rows, axis=0)) == S
    seeds = np.arange(S, dtype=np.int32)
    ex = Executor(base, fs, 2, S, seeds=seeds, dither=31)
    ex.set_kernel(KERNEL_CHAIN_V3)
    ex.set_coefs(0, rows)
    x = synth.pcm("full", S, T, ex.n_in, fs)
    y = ex.process(x)
    assert ex.last_chain_variant == 3
    spots = np.unique(np.linspace(0, S - 1, 16).astype(int))
    check_streams(oracle_lib, y, ex, lambda s: own_program(base, cw, rows[s]), x, 2, fs, seeds, 31, spots)


def test_c3_float_65536_streams(oracle_lib):
    fs, S, T = 48000, 65536, 256
    base = load_program("c3_peq16_f3_48k")
    cw = coef_words(base, 3)
    rows = jitter(base, cw, S, 3, seed=13)
    seeds = np.arange(S, dtype=np.int32)
    ex = Executor(base, fs, 3, S, seeds=seeds, dither=31)
    ex.set_kernel(KERNEL_CHAIN_V3)                                # AUTO takes k_chain2 for calls this short
    l0 = ex.launch_count
    ex.process(synth.pcm("noise", S, 8, ex.n_in, fs))
    plain = ex.launch_count - l0
    ex.reset(fs, seeds=seeds, dither=31)
    ex.set_coefs(0, rows)
    x = synth.pcm("noise", S, T, ex.n_in, fs)
    l1 = ex.launch_count
    y = ex.process(x)
    assert ex.launch_count - l1 == plain
    assert ex.last_chain_variant == 3
    spots = [0, 1, 31, 32, 4095, 4096, 20000, 32767, 32768, 50001, 65535]
    check_streams(oracle_lib, y, ex, lambda s: own_program(base, cw, rows[s]), x, 3, fs, seeds, 31, spots)


@pytest.mark.parametrize("fmt", [3, 5])
def test_float_guard_takes_out_of_range_rows(oracle_lib, fmt):
    """rows with a b2 of 2^-70 or a b0 of 2^8 (feed-forward words: the cascade stays finite) are re-executed exactly; the other
    streams run the fast form; all bit-exact, and the kernel the program gets without a table is unchanged"""
    fs, S, T = 48000, 32, 600
    base = crossover_program(800.0, 300, 0.5, fs, fmt)
    cw = coef_words(base, fmt)
    ex = Executor(base, fs, fmt, S, seeds=np.arange(S, dtype=np.int32), dither=24)
    x = pcm_for(fmt)("noise", S, T, ex.n_in, fs)
    ex.process(x[:, :10])
    kern = ex.last_kernel
    ex.reset(fs, seeds=np.arange(S, dtype=np.int32), dither=24)
    rows = jitter(base, cw, S, fmt, seed=3)
    b0 = 0                                                       # columns 0..4: b0 b1 b2 a1 a2 of the first block's first section
    for s in range(0, S, 4):
        rows[s, b0 + 2] = np.float32(2.0 ** -70).view(np.int32)
    for s in range(2, S, 4):
        rows[s, b0] = np.float32(256.0).view(np.int32)
    ex.set_coefs(0, rows)
    y = ex.process(x)
    assert ex.last_kernel == kern
    check_streams(oracle_lib, y, ex, lambda s: own_program(base, cw, rows[s]), x, fmt, fs, np.arange(S), 24, range(S))


@pytest.mark.parametrize("fmt", [3, 5])
def test_float_guard_on_chain3_at_batch_width(oracle_lib, fmt):
    """the same out-of-range rows on k_chain3: C3 at 4096 streams, one stream in eight with a b2 of 2^-70, one in eight with a
    b0 of 2^8, the rest in range; flagged streams are re-executed exactly inside the call"""
    fs, S, T = 48000, 4096, 512
    base = load_program(f"c3_peq16_f{fmt}_48k")
    cw = coef_words(base, fmt)
    rows = jitter(base, cw, S, fmt, seed=53)
    rows[0::8, 2] = np.float32(2.0 ** -70).view(np.int32)
    rows[3::8, 0] = np.float32(256.0).view(np.int32)
    seeds = np.arange(S, dtype=np.int32)
    ex = Executor(base, fs, fmt, S, seeds=seeds, dither=24)
    ex.set_kernel(KERNEL_CHAIN_V3)
    ex.set_coefs(0, rows)
    x = pcm_for(fmt)("noise", S, T, ex.n_in, fs)
    y = ex.process(x)
    assert ex.last_chain_variant == 3
    spots = sorted(set(range(0, 48)) | {1024, 1027, 2048, 2051, 2053, 4088, 4091, 4095})
    check_streams(oracle_lib, y, ex, lambda s: own_program(base, cw, rows[s]), x, fmt, fs, seeds, 24, spots)


def test_set_param_interplay_reload_and_reset(oracle_lib):
    fs, S, T = 48000, 16, 300
    base = crossover_program(500.0, 300, 0.5, fs, 2)
    cw = coef_words(base, 2)
    other = crossover_program(900.0, 300, 0.5, fs, 2)
    gain_room = crossover_program(500.0, 700, 0.25, fs, 2)              # delay + gain words differ
    nc = np.nonzero(base != gain_room)[0]
    assert not np.isin(nc, cw).any()
    seeds = np.arange(S, dtype=np.int32)
    ex = Executor(base, fs, 2, S, seeds=seeds, dither=24)
    ex.set_param(0, 4, int(cw[3]), other[cw[3]: cw[3] + 1])             # before the table: a variant for streams 0..3
    assert ex.num_variants == 2
    rows = jitter(base, cw, S, 2, seed=5)
    ex.set_coefs(4, rows[4:])                                            # rows 0..3 start from their variant's words
    ex.set_param(8, 2, int(cw[0]), [int(other[cw[0]])])                 # after: into the rows, no variant
    assert ex.num_variants == 2
    for r in (nc[0], nc[-1]):
        ex.set_param(12, 4, int(r), [int(gain_room[r])])                # non-coefficient words: variants, combined with the rows
    assert ex.num_variants == 3
    expect = []
    for s in range(S):
        p = base.copy()
        if s < 4:
            p[cw[3]] = other[cw[3]]
        else:
            p[cw] = rows[s]
        if s in (8, 9):
            p[cw[0]] = other[cw[0]]
        if s >= 12:
            p[nc[0]], p[nc[-1]] = gain_room[nc[0]], gain_room[nc[-1]]
        expect.append(p)
    x = synth.pcm("noise", S, T, ex.n_in, fs)
    y = ex.process(x)
    check_streams(oracle_lib, y, ex, lambda s: expect[s], x, 2, fs, seeds, 24, range(S))
    # reset at the same rate keeps the table
    ex.reset(fs, seeds=seeds, dither=24)
    y = ex.process(x)
    check_streams(oracle_lib, y, ex, lambda s: expect[s], x, 2, fs, seeds, 24, range(S))
    # reload_params drops it (and every variant)
    ex.reload_params(base)
    ex.reset(fs, seeds=seeds, dither=24)
    assert ex.num_variants == 1
    y = ex.process(x)
    check_streams(oracle_lib, y, ex, lambda s: base, x, 2, fs, seeds, 24, range(S))


def test_reset_to_another_rate_reads_that_rate_columns(oracle_lib):
    base = load_program("c2_testrpi_xover_f2_multifs")
    hd = wire.header(base.view(np.uint32))
    rates = [wire.FREQS[hd["freqMin"]], wire.FREQS[hd["freqMax"]]]
    S, T = 24, 400
    cw = coef_words(base, 2)
    rows = jitter(base, cw, S, 2, seed=17)
    seeds = np.arange(S, dtype=np.int32)
    ex = Executor(base, rates[0], 2, S, seeds=seeds, dither=24)
    ex.set_coefs(0, rows)
    for fs in rates + [rates[0]]:
        ex.reset(fs, seeds=seeds, dither=24)
        x = synth.pcm("noise", S, T, ex.n_in, fs)
        y = ex.process(x)
        check_streams(oracle_lib, y, ex, lambda s: own_program(base, cw, rows[s]), x, 2, fs, seeds, 24, range(S))


def test_call_paths(oracle_lib):
    """device rows written by a kernel just before set_coefs; set_coefs between two process_async calls without a host sync;
    any split of the frames; process_range; the host path; process_pcm; plugin order"""
    import torch
    fs, S, T = 48000, 96, 1200
    base = crossover_program(600.0, 300, 0.5, fs, 2)
    cw = coef_words(base, 2)
    rows = jitter(base, cw, S, 2, seed=19)
    rows2 = jitter(base, cw, S, 2, seed=23)
    seeds = np.arange(S, dtype=np.int32)
    x = synth.pcm("full", S, T, Executor(base, fs, 2, 1).n_in, fs)
    ref_first = [own_program(base, cw, rows[s]) for s in range(S)]

    def oracle_two(s, cut, p1, p2, xx):
        o = oracle_lib.Oracle(p1, 2, fs, seed=int(seeds[s]), dither=24)
        a = o.process(xx[s, :cut])
        o.code[: len(p2)] = p2
        return np.concatenate([a, o.process(xx[s, cut:])]), o.data.copy()

    # device rows: computed on the GPU, handed over without a host round trip, and swapped between two async calls
    ex = Executor(base, fs, 2, S, seeds=seeds, dither=24)
    src = torch.from_numpy(rows).cuda()
    src2 = torch.from_numpy(rows2).cuda()
    torch.cuda.synchronize()
    dev = torch.empty_like(src)
    torch.add(src, 0, out=dev)                                   # a kernel on the current stream writes the rows
    ex.set_coefs(0, dev)
    xd = torch.from_numpy(x).cuda()
    ya = ex.process(xd[:, :500].contiguous())
    dev2 = torch.empty_like(src2)
    torch.add(src2, 0, out=dev2)
    ex.set_coefs(0, dev2)
    yb = ex.process(xd[:, 500:].contiguous())
    torch.cuda.synchronize()
    y = torch.cat([ya, yb], dim=1).cpu().numpy()
    for s in range(S):
        r, d = oracle_two(s, 500, ref_first[s], own_program(base, cw, rows2[s]), x)
        assert np.array_equal(y[s], r), s
        assert np.array_equal(ex.get_state(s)[: ex.data_size], d), s
    # any split of the frames, process_range over two halves, host path: identical output
    ref = np.stack([oracle_lib.Oracle(ref_first[s], 2, fs, seed=int(seeds[s]), dither=24).process(x[s]) for s in range(S)])
    for cuts in ([T], [1, 63, 700, T], [257, T]):
        ex = Executor(base, fs, 2, S, seeds=seeds, dither=24)
        ex.set_coefs(0, rows)
        parts, a = [], 0
        for b in cuts:
            parts.append(ex.process(x[:, a:b]))
            a = b
        assert np.array_equal(np.concatenate(parts, axis=1), ref)
    ex = Executor(base, fs, 2, S, seeds=seeds, dither=24)
    ex.set_coefs(0, rows)
    h = S // 3
    y1 = ex.process_range(xd[:h].contiguous(), 0)
    y2 = ex.process_range(xd[h:].contiguous(), h)
    torch.cuda.synchronize()
    assert np.array_equal(torch.cat([y1, y2]).cpu().numpy(), ref)
    # process_pcm (S16 frames, widened on the device)
    ex = Executor(base, fs, 2, S, seeds=seeds, dither=24)
    ex.set_coefs(0, rows)
    raw = (x >> 16).astype(np.int16)
    yp = ex.process_pcm(raw, 1, T)
    xw = raw.astype(np.int32) << 16
    for s in (0, 17, S - 1):
        assert np.array_equal(yp[s], oracle_lib.Oracle(ref_first[s], 2, fs, seed=int(seeds[s]), dither=24).process(xw[s])), s
    # plugin order
    ex = Executor(base, fs, 2, S, seeds=seeds, dither=24)
    ex.set_order(64)
    ex.set_coefs(0, rows)
    yo = ex.process(x)
    for s in (0, 5, S - 1):
        o = oracle_lib.Oracle(ref_first[s], 2, fs, seed=int(seeds[s]), dither=24)
        assert np.array_equal(yo[s], o.process_plugin_order(x[s], 64, ex.n_in, ex.n_out)), s


def test_refusals_change_nothing(oracle_lib):
    import ctypes as C
    from avdsp_b200 import _lib
    fs, S, T = 48000, 8, 200
    mix = load_program("c5_mixer8x8_f2_192k")
    exm = Executor(mix, 192000, 2, 2)
    with pytest.raises(AvdspError) as e:
        exm.set_coefs(0, np.zeros((2, 0), np.int32))
    assert e.value.code == ERR_UNSUPPORTED
    base = crossover_program(700.0, 300, 0.5, fs, 2)
    cw = coef_words(base, 2)
    rows = jitter(base, cw, S, 2, seed=29)
    seeds = np.arange(S, dtype=np.int32)
    ex = Executor(base, fs, 2, S, seeds=seeds, dither=24)
    ex.set_coefs(0, rows)
    for first, r in ((-1, rows), (1, rows), (S, rows[:1])):
        with pytest.raises(AvdspError) as e:
            ex.set_coefs(first, r)
        assert e.value.code == ERR_ARG
    L = _lib.lib()
    assert L.avdsp_b200_set_coefs(ex._h, 0, 1, None, 0, None) == ERR_ARG
    assert L.avdsp_b200_set_coefs(ex._h, 0, 1, rows.ctypes.data, 7, None) == ERR_ARG
    # rows of the wrong width never reach the library (it reads n * nCoef words)
    import torch
    for bad in (rows[:, :-1], np.concatenate([rows, rows[:, :1]], axis=1)):
        with pytest.raises(ValueError):
            ex.set_coefs(0, np.ascontiguousarray(bad))
    with pytest.raises(ValueError):
        ex.set_coefs(0, torch.from_numpy(np.ascontiguousarray(rows[:, :-1])).cuda())
    # a set_param that would move the table's words (a block's section count) is refused before it changes anything: no variant,
    # no row written, not even the coefficient word the same call carries
    p = [p for p, op, _ in wire.walk(base.view(np.uint32)) if op == wire.OP["BIQUADS"]][0]
    h = p + int(base[p + 2])
    assert h + 5 == cw[0]
    patch = base[h: h + 6].copy()
    patch[0] = (int(base[h]) & ~0xFFFF) | ((int(base[h]) & 0xFFFF) - 1)
    patch[5] = int(base[h + 5]) + 12345
    with pytest.raises(AvdspError) as e:
        ex.set_param(0, 2, h, patch)
    assert e.value.code == ERR_UNSUPPORTED
    assert ex.num_variants == 1
    ex.set_coefs(S - 1, rows[S - 1:])                              # the table still takes rows
    x = synth.pcm("noise", S, T, ex.n_in, fs)
    y = ex.process(x)
    check_streams(oracle_lib, y, ex, lambda s: own_program(base, cw, rows[s]), x, 2, fs, seeds, 24, range(S))


def test_multi_device_host_rows(oracle_lib):
    import torch
    fs, S, T = 48000, 40, 300
    base = crossover_program(700.0, 300, 0.5, fs, 2)
    cw = coef_words(base, 2)
    rows = jitter(base, cw, S, 2, seed=31)
    seeds = np.arange(S, dtype=np.int32)
    ndev = torch.cuda.device_count()
    old = os.environ.get("AVDSP_B200_MULTI_REPLICATE")
    if ndev < 2:
        os.environ["AVDSP_B200_MULTI_REPLICATE"] = "2"           # two shards on the one GPU there is
    try:
        ex = Executor(base, fs, 2, S, seeds=seeds, dither=24, devices=list(range(min(ndev, 4))))
    finally:
        if old is None:
            os.environ.pop("AVDSP_B200_MULTI_REPLICATE", None)
        else:
            os.environ["AVDSP_B200_MULTI_REPLICATE"] = old
    assert ex.n_devices >= 2
    with pytest.raises(AvdspError) as e:
        ex.set_coefs(0, torch.from_numpy(rows).cuda())
    assert e.value.code == ERR_UNSUPPORTED
    ex.set_coefs(3, rows[3:])
    x = synth.pcm("noise", S, T, ex.n_in, fs)
    y = ex.process(x)
    check_streams(oracle_lib, y, ex, lambda s: own_program(base, cw, rows[s]) if s >= 3 else base, x, 2, fs, seeds, 24, range(S))
