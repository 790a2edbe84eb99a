"""Cost of the per-stream coefficient table (avdsp_b200_set_coefs): python tools/coef_table_bench.py [out.jsonl]

One GPU run, CUDA events around each call, warm-ups first, cases interleaved rep by rep so that clocks and neighbours affect them
alike.  Pairs: the program as loaded ("none") against a table whose rows are all distinct ("table"), for
  C2 (4096 x 48000, the bench.py shape) on the kernel AUTO picks (k_chain3) and on k_chain2, C3-float at 65536 streams,
  k_dag (C1, 4096 streams) and, for the record, k_generic (C2, 4096 x 4800);
and, for contrast, C2 with 64 and 512 streams on set_param variants of their own (one launch per run of streams).
The GPU name and power limit are read in the same run and written beside the numbers."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

from avdsp_b200 import Executor, synth, coef_words, load_bin, KERNEL_AUTO, KERNEL_CHAIN_V2, KERNEL_GENERIC  # noqa: E402

PROG = os.path.join(ROOT, "tests", "golden", "programs")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(",")[:2]
    return {"gpu": name.strip(), "power_limit": power.strip()}


def rows_for(base, fmt, n, seed):
    """n distinct rows: the feed-forward words (b0 b1 b2: columns 0..2 of each group of five) moved a little, so every filter
    keeps the program's poles, its stability and its float-class guard behaviour"""
    cw = coef_words(base, fmt)
    rng = np.random.default_rng(seed)
    v = base[cw].astype(np.int32)
    ff = (np.arange(len(cw)) % 5 < 3)[None, :] & (v[None, :] != 0)
    if fmt == 2:
        r = v[None, :].astype(np.int64) + rng.integers(-64, 65, (n, len(cw)))
        return cw, np.where(ff, r, v[None, :]).astype(np.int32)
    f = v.view(np.float32).astype(np.float64)[None, :] * (1.0 + rng.uniform(-1e-4, 1e-4, (n, len(cw))))
    return cw, np.where(ff, f.astype(np.float32).view(np.int32), v[None, :]).astype(np.int32)


class Case:
    def __init__(self, name, prog, fmt, fs, S, T, kernel=KERNEL_AUTO, table=False, variants=0):
        base = load_bin(os.path.join(PROG, prog + ".bin"))
        self.name, self.S, self.T = name, S, T
        self.ex = Executor(base, fs, fmt, S, seeds=np.arange(S, dtype=np.int32), dither=31)
        self.ex.set_kernel(kernel)
        cw, rows = rows_for(base, fmt, S, seed=S + fmt)
        if table:
            self.ex.set_coefs(0, rows)
        for s in range(variants):                     # a variant of its own for each of the first `variants` streams
            self.ex.set_param(s, 1, int(cw[0]), [int(base[cw[0]]) + 1 + s])
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
        return {"case": self.name, "streams": self.S, "frames": self.T, "kernel": self.ex.last_kernel + str(self.ex.last_chain_variant or ""),
                "variants": self.ex.num_variants, "launches_per_call": self.launches, "ms_median": round(ms[len(ms) // 2], 3),
                "ms_min": round(ms[0], 3), "ms_max": round(ms[-1], 3), "reps": len(ms)}


def pair(label, prog, fmt, fs, S, T, kernel=KERNEL_AUTO):
    return [Case(f"{label}/none", prog, fmt, fs, S, T, kernel), Case(f"{label}/table", prog, fmt, fs, S, T, kernel, table=True)]


def main():
    out = open(sys.argv[1], "w") if len(sys.argv) > 1 else None
    info = gpu_info()
    groups = [
        pair("c2_chain3", "c2_testrpi_xover_f2_192k", 2, 192000, 4096, 48000)
        + [Case(f"c2_variants{v}", "c2_testrpi_xover_f2_192k", 2, 192000, 4096, 48000, variants=v) for v in (64, 512)],
        pair("c2_chain2", "c2_testrpi_xover_f2_192k", 2, 192000, 4096, 48000, KERNEL_CHAIN_V2),
        pair("c3f", "c3_peq16_f3_48k", 3, 48000, 65536, 4096),
        pair("c1_dag", "c1_crossover2x2lfe_f2_48k", 2, 48000, 4096, 48000),
        pair("c2_generic", "c2_testrpi_xover_f2_192k", 2, 192000, 4096, 4800, KERNEL_GENERIC),
    ]
    for cases in groups:
        for c in cases:                                # warm-up: module loads, first-touch of every buffer
            c.run(False)
            c.run(False)
        for _ in range(7):
            for c in cases:
                c.run(True)
        res = [c.result() for c in cases]
        base = res[0]["ms_median"]
        for r in res:
            r["vs_none"] = round(r["ms_median"] / base, 4)
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
