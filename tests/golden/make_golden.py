#!/usr/bin/env python
"""Regenerates everything under tests/golden/ from the REAL reference, run in the authoring container.

  programs/*.bin|.h : produced by the unchanged reference encoder (oracle/_ref/dspcreate, built from
                      /root/reference by oracle/Makefile) with the command lines below.  The three
                      checked-in fixtures of the reference that regenerate byte-identically
                      (osx/crossoverLV6.bin, osx/dacdiy1.bin, osx/dsptest1.bin, osx/dac8prodsp.h; commands from
                      osx/oktodac.mak:19-41) are asserted to do so.
  vectors/*.npz     : input PCM + output PCM + final data area produced by the reference runtime itself
                      (oracle/_ref/libavdspruntime<fmt>_strict.so through oracle/refdriver.py), canonical
                      order (frame-major, cores ascending).
  reference_digests.json : not written here; AVDSP_RECORD_REFERENCE_DIGESTS=1 python -m pytest
                      tests/test_oracle_golden.py -k compiled_reference  rewrites it (see AgainstReference there).

Nothing here runs on the GPU box: /root/reference does not exist there; the committed files do.
Usage:  python tests/golden/make_golden.py         (from the repo root, after `make -C oracle`)
"""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import refdriver, wire          # noqa: E402
from avdsp_b200 import synth                 # noqa: E402

REFDIR = os.path.join(ROOT, "oracle", "_ref")
PROGDIR = os.path.join(ROOT, "tests", "golden", "programs")
VECDIR = os.path.join(ROOT, "tests", "golden", "vectors")
REF_OSX = "/root/reference/module_avdsp/osx"

PROGDIR_EARLY = os.path.join(ROOT, "tests", "golden", "programs")   # the symbol table dspcreate -dumpfile writes for C1 is a fixture too
# name -> (program .so, output kind, dspcreate arguments)
PROGRAMS = {
    "c1_crossover2x2lfe_f2_48k":   ("crossover2x2lfe", "bin", "-dspformat 2 -fsmin 48000 -fsmax 48000 -dumpfile " + os.path.join(PROGDIR_EARLY, "c1_crossover2x2lfe_f2_48k.dump")),
    "c2_testrpi_xover_f2_192k":    ("testrpi", "bin", "-dspformat 2 -fsmin 192000 -fsmax 192000 -crossover"),
    "c2_testrpi_xover_f2_multifs": ("testrpi", "bin", "-dspformat 2 -fsmax 192000 -crossover"),
    "c3_peq16_f3_48k":             ("c3_peq16", "bin", "-dspformat 3 -fsmin 48000 -fsmax 48000"),
    "c3_peq16_f4_48k":             ("c3_peq16", "bin", "-dspformat 4 -fsmin 48000 -fsmax 48000"),
    "c3_peq16_f5_48k":             ("c3_peq16", "bin", "-dspformat 5 -fsmin 48000 -fsmax 48000"),
    "c3_peq16_f6_48k":             ("c3_peq16", "bin", "-dspformat 6 -fsmin 48000 -fsmax 48000"),
    "c3_peq16_f2_48k":             ("c3_peq16", "bin", "-dspformat 2 -fsmin 48000 -fsmax 48000"),
    "c5_mixer8x8_f2_192k":         ("c5_mixer8x8", "bin", "-dspformat 2 -fsmin 192000 -fsmax 192000"),
    # the reference's own fixtures (osx/oktodac.mak)
    "ref_crossoverLV6":            ("crossoverLV6", "bin", "-dspformat 2 -fsmax 96000 -fx 800"),
    "ref_dacdiy1":                 ("oktodac_diy", "bin", "-dspformat 2 -fsmax 192000 -prog 1 -dither 24"),
    "ref_dsptest1":                ("testfunction", "bin", "-dspformat 3 -fsmax 96000 -test1 -dither 26"),
    "ref_dac8prodsp":              ("oktodac", "hex", "-dspformat 2 -dac8prodsp -dither 24"),
}
# our own all-opcode programs (oracle/progs/allops_*.c) on the unchanged encoder: every `case` of the runtime's switch
# (runtime/dsp_runtime.c:319-1305) executes at least once in every DSP_FORMAT
for _f in (2, 3, 4, 5, 6):
    PROGRAMS[f"allops_alu_f{_f}_48k"] = ("allops_alu", "bin", f"-dspformat {_f} -fsmin 48000 -fsmax 48000" + (" -int" if _f == 2 else ""))
    PROGRAMS[f"allops_gen_f{_f}_multifs"] = ("allops_gen", "bin", f"-dspformat {_f} -fsmin 44100 -fsmax 192000")
MUST_MATCH = {"ref_crossoverLV6": "crossoverLV6.bin", "ref_dacdiy1": "dacdiy1.bin",
              "ref_dsptest1": "dsptest1.bin", "ref_dac8prodsp": "dac8prodsp.h"}

# checked-in fixtures of the reference that its current sources no longer regenerate byte for byte (uninitialised MEM words
# in dacfabriceo*.bin, SURVEY.md App. C #7; the LXmini sources moved on): taken as they are, as test vectors.
# name -> path under /root/reference/module_avdsp
COPIED = {
    "ref_dacfabriceo":      "osx/dacfabriceo.bin",
    "ref_dacfabriceo_oppo": "osx/dacfabriceo_oppo.bin",
    "ref_lxmini_lr2":       "osx/dacfabriceo_LXmini_LR2.bin",
    "ref_lxmini_lv8":       "osx/dacfabriceo_LXmini_LV8.bin",
    "ref_win_mydspcode":    "windows/mydspcode.bin",
    # encoder 0x100 files: 11-word header, other opcode layouts (the reference runtime crashes on the first): decoder must reject
    "old_rpi_dacfabriceo":  "rpi/dacfabriceo.bin",
    "old_rpi_testrew":      "rpi/testrew.bin",
    "old_osx_mydspcode":    "osx/mydspcode.bin",
}


def asm_misc_program(fmt):
    """Opcodes the encoder has no emitter for (LOAD_MEM_DATA, runtime/dsp_runtime.c:1277-1281) or only WIP ones, in the layout
    the runtime decodes; plus the 32-bit DELAY_1 / DELAY forms next to their 64-bit twins."""
    a = wire.Asm(fmt=fmt, fmin=44100, fmax=96000)
    a.core()
    tp = a.tpdf_calc(24)
    a.store(0)
    a.load_mem_data(tp)                 # X = the 64-bit TPDF value TPDF_CALC left in the data area
    a.store(1)
    a.load_gain(8, 0.5)
    a.delay_1()
    a.load_mem_data(a.data - 2)         # reads back what DELAY_1 just stored
    a.sat0db()
    a.store(2)
    a.core()
    a.load_gain(9, 0.5)
    a.delay_fixed_us(250, 96000, dp=True)
    a.delay_fixed_us(100, 96000, dp=False)
    a.sat0db()
    a.store(3)
    a.load_gain(8, 0.25)
    a.dcblock([-0.003, -0.0025, -0.0015, -0.00125])
    a.clip(0.1)
    a.sat0db_tpdf()
    a.store(4)
    return a.end()


def fir_taps(n, seed):
    """Room-correction-like impulse: a main tap followed by exponentially decaying noise; sum(|c|) ~ 1.3."""
    r = np.random.default_rng(seed)
    k = np.arange(n)
    c = r.standard_normal(n) * np.exp(-k / (n / 6.0))
    c *= 0.6 / np.abs(c).sum()
    c[0] += 0.7
    return c.astype(np.float32)


def fir_program(fmt, lens, fmin=48000, fmax=48000, nch=2, variants=None):
    """C4 (SURVEY.md 8): one core per channel, LOAD_GAIN -> FIR -> SAT0DB -> STORE, ALSA io convention (in 8+k, out k).
    Assembled with oracle/wire.py in the layout the RUNTIME decodes (dsp_runtime.c:928-969) because the reference
    encoder's dsp_FIR emission is broken (SURVEY.md App. C #4-5).  lens[k][fsIndex] = taps of channel k at that fs,
    ('delay', n) for the plain-delay form, or None (FIR skipped at that fs)."""
    a = wire.Asm(fmt=fmt, fmin=fmin, fmax=fmax)
    for k in range(nch):
        a.core()
        a.param()
        imps = []
        for fi, ln in enumerate(lens[k]):
            if ln is None or isinstance(ln, tuple):
                imps.append(ln)
            else:
                t = fir_taps(ln, 1000 * k + fi + 17)
                imps.append([wire.q28(float(v)) for v in t] if fmt == 2 else [float(v) for v in t])
        where = a.fir_impulses(imps)
        mx = max([(l[1] + 1) if isinstance(l, tuple) else (l or 0) for l in lens[k]] + [1])
        a.load_gain(8 + k, 0.9 - 0.2 * k)
        a.fir(where, mx)
        if variants and variants[k] == "gain":
            a.gain(1.25)
            a.sat0db()
        elif variants and variants[k] == "satgain":
            a.sat0db_gain(0.8)
        else:
            a.sat0db()
        a.store(k)
        if variants and variants[k] == "gain":
            a.store(nch + k)
    return a.end()


# programs assembled here (no reference encoder involved): name -> (DSP_FORMAT, builder)
ASM_PROGRAMS = {}
for _f in (2, 3):
    ASM_PROGRAMS[f"c4_fir4096_f{_f}_48k"] = (_f, lambda f=_f: fir_program(f, [[4096], [4096]]))
for _f in (2, 3, 4, 5, 6):
    ASM_PROGRAMS[f"allops_misc_f{_f}_multifs"] = (_f, lambda f=_f: asm_misc_program(f))
for _f in (2, 3, 4, 5, 6):
    # two sampling rates: 48k convolution (ragged lengths), 96k: channel 0 plain delay, channel 1 skipped
    ASM_PROGRAMS[f"c4s_fir_f{_f}_multifs"] = (_f, lambda f=_f: fir_program(
        f, [[100, None, ("delay", 37)], [33, None, None]], fmin=48000, fmax=96000, variants=["gain", "satgain"]))

# vector name -> (program, DSP_FORMAT, fs, seed, defaultDither, stimulus, frames)
VECTORS = {}
for stim in ("noise", "full", "impulse", "sine"):
    VECTORS[f"c1_{stim}"] = ("c1_crossover2x2lfe_f2_48k", 2, 48000, 0, 31, stim, 1024)
    VECTORS[f"c2_{stim}"] = ("c2_testrpi_xover_f2_192k", 2, 192000, 0, 31, stim, 1024)
    VECTORS[f"c5_{stim}"] = ("c5_mixer8x8_f2_192k", 2, 192000, 3, 31, stim, 2048)
for fmt in (3, 4, 5, 6):
    VECTORS[f"c3_f{fmt}_noise"] = (f"c3_peq16_f{fmt}_48k", fmt, 48000, 0, 31, "noise", 1024)
    VECTORS[f"c3_f{fmt}_impulse"] = (f"c3_peq16_f{fmt}_48k", fmt, 48000, 0, 31, "impulse", 2048)
VECTORS["c3_f2_noise"] = ("c3_peq16_f2_48k", 2, 48000, 0, 31, "noise", 1024)
VECTORS["c2_multifs_96k"] = ("c2_testrpi_xover_f2_multifs", 2, 96000, 7, 24, "noise", 1024)
VECTORS["c2_multifs_44k"] = ("c2_testrpi_xover_f2_multifs", 2, 44100, 7, 24, "full", 1024)
VECTORS["lv6_48k"] = ("ref_crossoverLV6", 2, 48000, 0, 24, "noise", 1024)
VECTORS["lv6_96k"] = ("ref_crossoverLV6", 2, 96000, 11, 31, "full", 1024)
VECTORS["dacdiy1_192k"] = ("ref_dacdiy1", 2, 192000, 0, 24, "noise", 1024)
VECTORS["dacdiy1_48k"] = ("ref_dacdiy1", 2, 48000, 5, 31, "sine", 1024)
VECTORS["dsptest1_48k"] = ("ref_dsptest1", 3, 48000, 0, 26, "noise", 1024)
# DSP_FIR: the reference's FLOAT kernel is a correct direct form (dsp_firSTD.h:38-52) -> golden vectors for formats 3..6;
# its fixed-point kernel is not a convolution (SURVEY.md App. C #3) -> no golden for format 2 (oracle-defined semantics)
for fmt in (3, 4, 5, 6):
    VECTORS[f"c4s_f{fmt}_48k_noise"] = (f"c4s_fir_f{fmt}_multifs", fmt, 48000, 0, 31, "noise", 512)
    VECTORS[f"c4s_f{fmt}_96k_full"] = (f"c4s_fir_f{fmt}_multifs", fmt, 96000, 0, 24, "full", 256)
VECTORS["c4_f3_noise"] = ("c4_fir4096_f3_48k", 3, 48000, 0, 31, "noise", 640)
VECTORS["dac8prodsp_96k"] = ("ref_dac8prodsp", 2, 96000, 0, 24, "noise", 1024)
# every opcode, every DSP_FORMAT
for fmt in (2, 3, 4, 5, 6):
    VECTORS[f"allops_alu_f{fmt}_noise"] = (f"allops_alu_f{fmt}_48k", fmt, 48000, 0, 31, "noise", 512)
    VECTORS[f"allops_alu_f{fmt}_full"] = (f"allops_alu_f{fmt}_48k", fmt, 48000, 5, 24, "full", 512)
    VECTORS[f"allops_gen_f{fmt}_48k"] = (f"allops_gen_f{fmt}_multifs", fmt, 48000, 0, 31, "noise", 1536)
    VECTORS[f"allops_gen_f{fmt}_96k"] = (f"allops_gen_f{fmt}_multifs", fmt, 96000, 9, 24, "full", 1536)
    VECTORS[f"allops_misc_f{fmt}_44k"] = (f"allops_misc_f{fmt}_multifs", fmt, 44100, 2, 24, "noise", 512)
VECTORS["allops_gen_f2_192k_sine"] = ("allops_gen_f2_multifs", 2, 192000, 0, 20, "sine", 2048)
# the remaining fixtures of the reference (osx/*.bin, windows/mydspcode.bin): DELAY_DP, SHIFT, SAT0DB_GAIN, X/Y crossovers
VECTORS["dacfabriceo_48k"] = ("ref_dacfabriceo", 2, 48000, 0, 24, "noise", 1024)
VECTORS["dacfabriceo_96k"] = ("ref_dacfabriceo", 2, 96000, 3, 31, "full", 1024)
VECTORS["dacfabriceo_oppo_88k"] = ("ref_dacfabriceo_oppo", 2, 88200, 0, 24, "noise", 1024)
VECTORS["lxmini_lr2_192k"] = ("ref_lxmini_lr2", 2, 192000, 0, 23, "noise", 1024)
VECTORS["lxmini_lr2_44k"] = ("ref_lxmini_lr2", 2, 44100, 1, 31, "full", 1024)
VECTORS["lxmini_lv8_96k"] = ("ref_lxmini_lv8", 2, 96000, 0, 23, "noise", 1024)
VECTORS["lxmini_lv8_176k"] = ("ref_lxmini_lv8", 2, 176400, 4, 24, "sine", 1024)
VECTORS["win_mydspcode_48k"] = ("ref_win_mydspcode", 2, 48000, 0, 24, "noise", 1024)
VECTORS["win_mydspcode_192k"] = ("ref_win_mydspcode", 2, 192000, 8, 31, "full", 1024)


def prog_path(name):
    if name in ASM_PROGRAMS or name in COPIED:
        return os.path.join(PROGDIR, name + ".bin")
    kind = PROGRAMS[name][1]
    return os.path.join(PROGDIR, name + (".bin" if kind == "bin" else ".h"))


def load_prog(name):
    from avdsp_b200 import program
    return program.load(prog_path(name))


def make_programs():
    os.makedirs(PROGDIR, exist_ok=True)
    env = dict(os.environ, LD_LIBRARY_PATH=REFDIR)
    for name, (so, kind, args) in PROGRAMS.items():
        out = prog_path(name)
        cmd = [os.path.join(REFDIR, "dspcreate"), "-dspprog", os.path.join(REFDIR, so + ".so"),
               "-binfile" if kind == "bin" else "-hexfile", out] + args.split()
        r = subprocess.run(cmd, env=env, capture_output=True, text=True, cwd=REFDIR)
        if r.returncode or not os.path.exists(out):
            raise SystemExit(f"{name}: dspcreate failed\n{r.stdout[-2000:]}{r.stderr[-2000:]}")
        if name in MUST_MATCH and os.path.exists(os.path.join(REF_OSX, MUST_MATCH[name])):
            a = open(out, "rb").read()
            b = open(os.path.join(REF_OSX, MUST_MATCH[name]), "rb").read()
            assert a == b, f"{name}: regenerated file differs from the reference's checked-in {MUST_MATCH[name]}"
            print(f"  {name}: byte-identical to osx/{MUST_MATCH[name]}")
        print(f"  wrote {os.path.relpath(out, ROOT)} ({os.path.getsize(out)} bytes)")


def copy_fixtures():
    for name, rel in COPIED.items():
        raw = open(os.path.join("/root/reference/module_avdsp", rel), "rb").read()
        open(prog_path(name), "wb").write(raw)
        print(f"  copied {rel} -> {os.path.relpath(prog_path(name), ROOT)} ({len(raw)} bytes)")


def make_asm_programs():
    os.makedirs(PROGDIR, exist_ok=True)
    for name, (fmt, build) in ASM_PROGRAMS.items():
        w = build()
        w.astype("<i4").tofile(prog_path(name))
        print(f"  wrote {os.path.relpath(prog_path(name), ROOT)} ({w.size * 4} bytes, assembled)")


def make_vectors():
    os.makedirs(VECDIR, exist_ok=True)
    only = sys.argv[1:]          # optional name prefixes: regenerate just those vectors (npz files are not byte-reproducible)
    for vname, (prog, fmt, fs, seed, dither, stim, frames) in VECTORS.items():
        if only and not any(vname.startswith(o) for o in only):
            continue
        w = load_prog(prog)
        ins, outs = wire.io_maps(w)
        gen = synth.pcm_float if fmt >= 5 else synth.pcm
        x = gen(stim, 1, frames, len(ins), fs)[0]
        r = refdriver.RefProgram(w, fmt, fs, seed=seed, dither=dither, strict=True)
        assert r.rc > 0, (vname, r.rc)
        y = r.process(x)
        np.savez_compressed(os.path.join(VECDIR, vname + ".npz"), x=x, y=y, data=r.data.copy(),
                            code=r.buf[: r.total].copy(),
                            meta=np.array([fmt, fs, seed, dither, frames], dtype=np.int64), program=prog, stimulus=stim)
        print(f"  {vname}: {prog} fmt{fmt} fs={fs} {stim} x{x.shape} -> y{y.shape} nonzero={np.count_nonzero(y)}")


if __name__ == "__main__":
    if not os.path.exists(os.path.join(REFDIR, "dspcreate")):
        raise SystemExit("oracle/_ref is not built: run `make -C oracle` where /root/reference exists")
    if not sys.argv[1:]:
        make_programs()
        copy_fixtures()
    make_asm_programs()
    make_vectors()
