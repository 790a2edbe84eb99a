"""Cost of the per-stream FIR table (avdsp_b200_set_fir_taps): python tools/fir_table_bench.py [out.jsonl]

One GPU run, CUDA events around each call, warm-ups first, cases interleaved rep by rep so that clocks and neighbours affect them
alike.  At the C4 shape (1024 streams x 65536 frames, two paths of 4096 taps), DSP_FORMAT 2 and 3, on the exact FIR kernel
(k_fir, which runs the table):
  the program as loaded ("none") against a table whose rows are all distinct ("table");
and, for contrast, 16 and 64 streams with taps of their own through set_param variants (one launch per run of streams; variants
of FIR programs are not forked onto side streams because they share the FIR workspace).  For format 2, the tensor-core
kernel that AUTO picks at this size: with shared taps ("none_tc") and in its per-stream form with the table ("table_tc").
The GPU name, power limit and SM clock are read in the same run and written beside the numbers."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

from avdsp_b200 import Executor, synth, fir_tap_words, load_bin, KERNEL_AUTO, KERNEL_FIR  # noqa: E402

PROG = os.path.join(ROOT, "tests", "golden", "programs")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm", "--format=csv,noheader"], capture_output=True, text=True)
    f = ((q.stdout.strip().splitlines() or ["?, ?, ?"])[0].split(",") + ["?"] * 3)[:3]
    return {"gpu": f[0].strip(), "power_limit": f[1].strip(), "sm_clock": f[2].strip()}


def rows_for(base, fmt, n, seed):
    """n distinct impulse responses near the program's own: every tap moved by up to 64 LSBs (Q4.28) or by a relative 1e-4
    (float), which keeps them above 2^-60 (no stream leaves the FIR kernel)"""
    tw = fir_tap_words(base, fmt)
    rng = np.random.default_rng(seed)
    v = base[tw].astype(np.int32)
    if fmt == 2:
        return tw, (v[None, :].astype(np.int64) + rng.integers(-64, 65, (n, len(tw)))).astype(np.int32)
    f = v.view(np.float32).astype(np.float64)[None, :] * (1.0 + rng.uniform(-1e-4, 1e-4, (n, len(tw))))
    return tw, np.ascontiguousarray(f.astype(np.float32).view(np.int32))


class Case:
    def __init__(self, name, fmt, S, T, kernel=KERNEL_FIR, table=False, variants=0):
        base = load_bin(os.path.join(PROG, f"c4_fir4096_f{fmt}_48k.bin"))
        self.name, self.S, self.T = name, S, T
        self.ex = Executor(base, 48000, fmt, S, seeds=np.arange(S, dtype=np.int32), dither=31)
        self.ex.set_kernel(kernel)
        tw, rows = rows_for(base, fmt, S, seed=S + fmt)
        if table:
            self.ex.set_fir_taps(0, rows)
        for s in range(variants):                     # a variant of its own for each of the first `variants` streams
            self.ex.set_param(s, 1, int(tw[0]), rows[s, :len(tw) // 2])
        self.x = synth.pcm_torch("noise", S, T, self.ex.n_in, "cuda")
        self.y = torch.empty((S, T, self.ex.n_out), dtype=torch.int32, device="cuda")
        self.ms = []
        self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def run(self, timed):
        l0 = self.ex.launch_count
        self.e0.record()
        self.ex.process(self.x, out=self.y)
        self.e1.record()
        torch.cuda.synchronize()
        self.launches = self.ex.launch_count - l0
        if timed:
            self.ms.append(self.e0.elapsed_time(self.e1))

    def result(self):
        ms = sorted(self.ms)
        return {"case": self.name, "streams": self.S, "frames": self.T, "kernel": self.ex.last_kernel,
                "variants": self.ex.num_variants, "launches_per_call": self.launches, "ms_median": round(ms[len(ms) // 2], 3),
                "ms_min": round(ms[0], 3), "ms_max": round(ms[-1], 3), "reps": len(ms)}


def main():
    out = open(sys.argv[1], "w") if len(sys.argv) > 1 else None
    S, T = 1024, 65536
    for fmt in (2, 3):
        cases = [Case(f"c4f{fmt}/none", fmt, S, T), Case(f"c4f{fmt}/table", fmt, S, T, table=True)]
        cases += [Case(f"c4f{fmt}/variants{v}", fmt, S, T, variants=v) for v in (16, 64)]
        if fmt == 2:
            cases += [Case("c4f2/none_tc", fmt, S, T, kernel=KERNEL_AUTO), Case("c4f2/table_tc", fmt, S, T, kernel=KERNEL_AUTO, table=True)]
        for c in cases:                                # warm-up: module loads, first-touch of every buffer
            c.run(False)
            c.run(False)
        for _ in range(5):
            for c in cases:
                c.run(True)
        info = gpu_info()
        res = [c.result() for c in cases]
        base = res[0]["ms_median"]
        for r in res:
            r["vs_none_k_fir"] = round(r["ms_median"] / base, 4)
            r.update(info)
            line = json.dumps(r)
            print(line, flush=True)
            if out:
                print(line, file=out, flush=True)
        for c in cases:
            c.ex.close()
        del cases
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
