#!/usr/bin/env python
"""Time k_chain3 warp placements of one program (DESIGN.md 4.2a, "Warp placement").

The part list, the per-item prices and the planner's own placement come from the `chain kernel v3 placement` line of
`describe`.  Every placement that is distinct up to interchangeable items (same trace token: sections, form, finish,
source gain) and sub-partition relabelling is enumerated and counted by the IMAD.WIDE per frame of its busiest
sub-partition.  With --time, the placements at or below --max-macs plus a seeded sample of the rest run on the GPU,
each forced through AVDSP_B200_BINS3 on a fresh instance and timed with CUDA events; the planner's placement (or --baseline) is
timed again every --default-every placements to give the run-to-run spread.  One JSON line per timed placement.

  python tools/chain3_placement_sweep.py                       # count only (no GPU)
  python tools/chain3_placement_sweep.py --time --out sweep.jsonl [--general]

--general adds one LSB to b2 of every unit-gain section, so every part runs the general form: the placement a CTA gets
when a per-stream coefficient row breaks the identity.
"""
import argparse
import json
import os
import random
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import avdsp_b200  # noqa: E402

PROGRAMS = {"c2": ("c2_testrpi_xover_f2_192k", 2, 192000), "c3": ("c3_peq16_f2_48k", 2, 48000), "c3f": ("c3_peq16_f3_48k", 3, 48000)}


def placement_line(trace):
    """(items [(token, macs, other)], planner's sub-partition of each item) from the trace"""
    ln = [ln for ln in trace.splitlines() if ln.startswith("chain kernel v3 placement")][0]
    items = [(t, int(m), int(o)) for t, m, o in re.findall(r" ([0-9]+[uTg]*|d|s):(\d+)\+(\d+)", ln.split("per frame:")[1].split(";")[0])]
    bins = [int(b) for b in re.search(r"sub-partition of each item ([0-9,]+)", ln).group(1).split(",")]
    return items, bins


def general_form(words, fmt):
    """the program with b2 of every unit-gain section one LSB up: no part keeps the unit-gain form"""
    w = np.array(words, dtype=np.int32)
    cw = avdsp_b200.coef_words(w, fmt).reshape(-1, 5)
    for c in cw:
        b0, b1, b2, a1, a2 = (int(w[i]) for i in c)
        if b0 == 1 << 28 and b1 + a1 == -(1 << 28) and b2 + a2 == 0:
            w[c[2]] += 1
    return w


def enumerate_placements(items, nbins=4):
    """every assignment of items to bins, distinct up to interchangeable items and relabelling of equal-size bins;
    yields the sub-partition of each item"""
    total = len(items)
    slots = [(total - q + 3) // 4 for q in range(nbins)]
    kinds = sorted({t for t, _, _ in items})
    count = [sum(t == k for t, _, _ in items) for k in kinds]

    def contents(left, size):                               # count vectors of `size` items drawn from `left`, descending
        def rec(i, size):
            if i == len(left):
                if size == 0:
                    yield ()
                return
            for c in range(min(left[i], size), -1, -1):
                for rest in rec(i + 1, size - c):
                    yield (c,) + rest
        return rec(0, size)

    def rec(q, left, prev):
        if q == nbins:
            yield []
            return
        for c in contents(left, slots[q]):
            if prev is not None and slots[q] == slots[q - 1] and c > prev:    # equal bins in descending order
                continue
            for rest in rec(q + 1, [a - b for a, b in zip(left, c)], c):
                yield [c] + rest

    for binc in rec(0, count, None):
        pool = {k: [i for i, (t, _, _) in enumerate(items) if t == k] for k in kinds}
        out = [0] * total
        for q, c in enumerate(binc):
            for k, n in zip(kinds, c):
                for _ in range(n):
                    out[pool[k].pop(0)] = q
        yield out


def per_bin(items, bins, what):
    s = [0, 0, 0, 0]
    for (t, m, o), q in zip(items, bins):
        s[q] += {"macs": m, "general": 5 * int(re.match(r"\d*", t).group() or 0), "other": o}[what]
    return s


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except Exception as e:
        return f"nvidia-smi failed: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c2", choices=sorted(PROGRAMS))
    ap.add_argument("--streams", type=int, default=4096)
    ap.add_argument("--frames", type=int, default=12288)
    ap.add_argument("--reps", type=int, default=4, help="timed calls per placement (median)")
    ap.add_argument("--general", action="store_true")
    ap.add_argument("--max-macs", type=int, default=56, help="time every placement whose busiest sub-partition executes at most this")
    ap.add_argument("--sample", type=int, default=300, help="plus this many of the others (seeded)")
    ap.add_argument("--extra", action="append", default=[], help="a placement to time as well (AVDSP_B200_BINS3 form)")
    ap.add_argument("--baseline", default=None, help="the placement timed repeatedly for the spread (default: the planner's)")
    ap.add_argument("--default-every", type=int, default=100)
    ap.add_argument("--time", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    name, fmt, fs = PROGRAMS[args.workload]
    words = avdsp_b200.load_bin(os.path.join(ROOT, "tests", "golden", "programs", name + ".bin"))
    if args.general:
        words = general_form(words, fmt)
    os.environ.pop("AVDSP_B200_BINS3", None)
    items, default = placement_line(avdsp_b200.describe(words, fs, fmt, n_streams=args.streams, num_sms=148))
    if args.baseline:
        default = [int(c) for c in args.baseline.split(",")]
    allp = list(enumerate_placements(items))
    key = lambda b: max(per_bin(items, b, "macs"))
    hist = {}
    for b in allp:
        hist[key(b)] = hist.get(key(b), 0) + 1
    cum, acc = {}, 0
    for m in sorted(hist):
        acc += hist[m]
        cum[m] = acc
    print(f"{args.workload}{' (general form)' if args.general else ''}: items {' '.join(t for t, _, _ in items)}, "
          f"{len(allp)} distinct placements; busiest sub-partition IMAD.WIDE -> placements at or below: {cum}", file=sys.stderr)
    print(f"planner's placement {','.join(map(str, default))}: IMAD.WIDE {per_bin(items, default, 'macs')}, "
          f"every part general {per_bin(items, default, 'general')}", file=sys.stderr)
    if not args.time:
        return

    import torch
    from avdsp_b200 import synth
    rng = random.Random(0)
    sel = [b for b in allp if key(b) <= args.max_macs]
    rest = [b for b in allp if key(b) > args.max_macs]
    sel += rng.sample(rest, min(args.sample, len(rest)))
    sel += [[int(c) for c in e.split(",")] for e in args.extra]
    rng.shuffle(sel)
    dev = torch.device("cuda", 0)
    S, T = args.streams, args.frames
    seeds = np.arange(S, dtype=np.int32)
    probe = avdsp_b200.Executor(words, fs, fmt, S, seeds=seeds, dither=31, device=0)
    x = synth.pcm_torch("noise", S, T, probe.n_in, dev)
    y = torch.empty((S, T, probe.n_out), dtype=torch.int32, device=dev)
    probe.close()
    info0 = gpu_info()
    out = open(args.out, "w") if args.out else sys.stdout

    def run(bins, tag):
        os.environ["AVDSP_B200_BINS3"] = ",".join(map(str, bins))
        ex = avdsp_b200.Executor(words, fs, fmt, S, seeds=seeds, dither=31, device=0)
        try:
            ex.set_kernel(avdsp_b200.KERNEL_CHAIN_V3)
            got = placement_line(ex.trace)[1]
            assert got == list(bins), (got, bins)
            ex.process(x, out=y)
            ms = []
            for _ in range(args.reps):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                ex.process(x, out=y)
                b.record()
                b.synchronize()
                ms.append(a.elapsed_time(b))
            assert ex.last_chain_variant == 3
        finally:
            ex.close()
        rec = {"workload": args.workload, "general_form": args.general, "tag": tag, "placement": ",".join(map(str, bins)),
               "imad_per_smsp": per_bin(items, bins, "macs"), "imad_per_smsp_all_general": per_bin(items, bins, "general"),
               "issue_per_smsp": [m + o for m, o in zip(per_bin(items, bins, "macs"), per_bin(items, bins, "other"))],
               "ms_per_call": float(np.median(ms)), "ms_all": [round(v, 4) for v in ms], "streams": S, "frames": T}
        print(json.dumps(rec), file=out, flush=True)

    t0 = time.time()
    run(default, "baseline")
    for i, b in enumerate(sel):
        run(b, "sweep")
        if (i + 1) % args.default_every == 0:
            run(default, "baseline")
    run(default, "baseline")
    info1 = gpu_info()
    print(json.dumps({"workload": args.workload, "general_form": args.general, "tag": "gpu", "items": [t for t, _, _ in items],
                      "distinct_placements": len(allp), "at_or_below": cum, "timed": len(sel),
                      "gpu_before (name, power.limit, clocks.sm, clocks.max.sm)": info0, "gpu_after": info1,
                      "seconds": round(time.time() - t0, 1)}), file=out, flush=True)
    os.environ.pop("AVDSP_B200_BINS3", None)


if __name__ == "__main__":
    main()
