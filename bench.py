#!/usr/bin/env python
"""bench.py -- the headline measurement (BASELINE.json `metric`): channel-samples/s of the batched AVDSP
executor on B200, with the roofline of the dominant kernel and the reference runtime timed on the host
cores in the same run.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c5|c3]
                  [--streams S] [--frames T] [--dump-outputs DIR]

Workload at N=1 (config.workload): BASELINE.json configs[1] -- "DAC8PRO-style 8-ch 3-way crossover,
fixed-point int64 format, 192 kHz, 4096 independent streams batched on 1xB200" = program
tests/golden/programs/c2_testrpi_xover_f2_192k.bin (reference dspprogs/testrpi.c -crossover, encoded by the
unchanged reference encoder), 4096 streams x 48000 frames (0.25 s of audio) per step.
A "step" = one pass of the hot path over that batch: every stream advances by T frames.  For N>1 every
rank owns 4096 streams of its own (weak scaling, no data-path collective; SURVEY.md 8e).

One JSON line on stdout (rank 0).  `value` = whole-job channel-samples/s with PCM resident in HBM;
`e2e` = the same through the C-ABI host call (avdsp_b200_process, HOST memspace) on pinned host buffers,
host<->device copies inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: no __pycache__ written into it
DUMP_BYTES = 64 * 10**6             # cap of --dump-outputs

WORKLOADS = {
    # name: (program, DSP_FORMAT, fs, default streams, default frames, MACs/frame, description)
    "c2": ("c2_testrpi_xover_f2_192k", 2, 192000, 4096, 48000, 240,
           "C2 DAC8PRO-style 8-ch 3-way crossover (testrpi -crossover), int64 fixed point, 192 kHz"),
    "c5": ("c5_mixer8x8_f2_192k", 2, 192000, 4096, 48000, 72,
           "C5 8x8 matrix mixer + per-channel delays + gain/TPDF dither, int64 fixed point, 192 kHz"),
    "c3": ("c3_peq16_f2_48k", 2, 48000, 65536, 4096, 160,
           "C3 16-section parametric EQ per channel x2 (fixed-point encoding), 48 kHz"),
    "c3f": ("c3_peq16_f3_48k", 3, 48000, 65536, 4096, 160,
            "C3 16-section parametric EQ per channel x2, float format (DSP_FORMAT 3), 48 kHz"),
    "c4": ("c4_fir4096_f2_48k", 2, 48000, 1024, 65536, 8192,
           "C4 4096-tap room-correction FIR per channel x2, fixed point (direct tiled, int64 accumulation), 48 kHz"),
    "c4f": ("c4_fir4096_f3_48k", 3, 48000, 1024, 65536, 8192,
            "C4 4096-tap room-correction FIR per channel x2, float format (DSP_FORMAT 3, reference tap order), 48 kHz"),
}


def workload_config(desc, prog, S, T, fs, n_in, n_out):
    """`config` of the JSON line: the same keys and values in both arms (ours / reference)"""
    return {"workload": desc, "program": prog, "streams_per_gpu": S, "frames_per_step": T, "fs": fs, "n_in": n_in, "n_out": n_out,
            "layout": "interleaved [stream][frame][channel] int32"}


def prog_file(name):
    return os.path.join(ROOT, "tests", "golden", "programs", name + ".bin")


def dump_outputs(d, y, first):
    """--dump-outputs: what the last timed step returned (int32 PCM [S, T, n_out] on the device) as float64, which holds every
    int32 exactly.  Every stream when that fits DUMP_BYTES, else a fixed seeded sample of streams (and only the leading frames
    when one stream alone is larger): outputs.npy [k, t, n_out] and outputs_streams.npy [k], the job's stream numbers."""
    import numpy as np
    import torch
    S, T, n_out = y.shape
    room = DUMP_BYTES - 1024                                  # two .npy headers
    t = min(T, (room - 8) // (n_out * 8))
    k = min(S, room // (t * n_out * 8 + 8))
    idx = np.arange(S) if k == S else np.sort(np.random.default_rng(0).choice(S, k, replace=False))
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "outputs.npy"), y[torch.from_numpy(idx).to(y.device), :t].cpu().numpy().astype(np.float64))
    np.save(os.path.join(d, "outputs_streams.npy"), (idx + first).astype(np.float64))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU while the timed region runs (nvidia-smi, 200 ms)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 6 for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def cpu_reference_rate(prog, fmt, fs, frames, workers, streams_per_worker=1):
    """Time the reference's own CPU implementation on the host cores (oracle/_ref, compiled from
    /root/reference by oracle/Makefile); falls back to the C restatement (oracle/liboracle_avdsp.so)."""
    refdir = os.path.join(ROOT, "oracle", "_ref")
    exe, lib = os.path.join(refdir, "refbench"), os.path.join(refdir, f"libavdspruntime{fmt}.so")
    # fixed-point DSP_FIR: the reference's int kernel is not a convolution (SURVEY.md App. C #3) and does a fraction of the
    # work, so timing it would be meaningless: the oracle restatement ("port", one core) is the CPU baseline there
    broken_ref = fmt == 2 and "fir" in prog
    if os.path.exists(exe) and os.path.exists(lib) and not broken_ref:
        out = subprocess.run([exe, lib, prog_file(prog), str(fmt), str(fs), str(workers), str(streams_per_worker), str(frames)],
                             capture_output=True, text=True, timeout=900)
        if out.returncode == 0:
            r = json.loads(out.stdout.strip().splitlines()[-1])
            r.update(kind="reference", cores=workers)
            return r
    # "port": the oracle restatement, one core
    import numpy as np
    from oracle import pyoracle
    from avdsp_b200 import program, synth
    w = program.load(prog_file(prog))
    o = pyoracle.Oracle(w, fmt, fs, seed=0)
    x = synth.pcm("noise", 1, frames, len(o.ins), fs)[0]
    t0 = time.perf_counter()
    o.process(x)
    dt = time.perf_counter() - t0
    return {"frames": frames, "seconds": dt, "frames_per_s": frames / dt, "n_in": len(o.ins), "n_out": len(o.outs),
            "kind": "port", "cores": 1, "workers": 1}


def run_reference(args, wl):
    prog, fmt, fs, S, T, macs, desc = wl
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    # bounded sample of the workload per step: one stream per host core, `fr` frames each (~1-2 s per step)
    fr = max(1500000 * 240 // wl[5] // 1000 * 1000, 1000) if args.frames is None else args.frames   # bounded sample: ~0.6 s per host thread per step
    for _ in range(args.warmup):
        cpu_reference_rate(prog, fmt, fs, max(1000, fr // 20), cores)
    tot_frames, tot_s, kind, n_out, n_in = 0.0, 0.0, "reference", 8, 2
    for _ in range(args.steps):
        r = cpu_reference_rate(prog, fmt, fs, fr, cores)
        tot_frames += r["frames"]; tot_s += r["seconds"]; kind = r["kind"]; n_out = r["n_out"]; n_in = r.get("n_in", n_in); used = r["cores"]
    val = tot_frames * n_out / tot_s / 1e6
    sample = f"{used} streams x {fr} frames per step (one stream per host thread), stream-major, canonical core order"
    line = {"impl": "reference", "metric": "channel-samples/sec", "value": val, "unit": "Msps", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64" if fmt == 2 else "f32",
            "data": "synthetic",
            "config": workload_config(desc, prog, S if args.streams is None else args.streams, T, fs, n_in, n_out),
            "cpu_baseline": {"value": val, "unit": "Msps", "cores": used, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": "Msps", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--streams", type=int, default=None)
    ap.add_argument("--frames", type=int, default=None)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every rank owns --streams streams of its own (default); strong: --streams is the whole job, sharded over the ranks "
                         "(BASELINE configs[2]: 65536 float streams sharded across 2/4/8)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-multi", action="store_true", help="skip the one-call multi-device arm (avdsp_b200_create_multi) at N > 1")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--kernel", default="auto", choices=["auto", "generic", "chain", "chain_v2", "chain_v3", "mix", "fir", "fir_tc", "dag"],
                    help="force a kernel (diagnostics; the default is what the product picks)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last one to DIR/*.npy (float64, at most 64 MB: a fixed "
                         "sample of streams when larger; rank 0's streams when N > 1), to compare builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        return run_reference(args, wl)

    # rank 0 prints ONE JSON line on stdout: whatever native libraries write to file descriptor 1 (NCCL's "NCCL version ..."
    # banner) goes to stderr instead
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    import numpy as np
    import torch
    import avdsp_b200
    from avdsp_b200 import synth

    prog, fmt, fs, S, T, macs, desc = wl
    S = args.streams or S
    T = args.frames or T
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (avdsp_b200 has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    words = avdsp_b200.load_bin(prog_file(prog))
    S_job = S * world if args.scaling == "weak" else S
    if args.scaling == "strong":                       # the job's streams sharded over the ranks (contiguous balanced ranges)
        first, S = avdsp_b200.shard_range(S_job, rank, world)
    else:
        first = rank * S                               # weak scaling: rank r owns streams [r*S, (r+1)*S)
    seeds = np.arange(first, first + S, dtype=np.int32)
    ex = avdsp_b200.Executor(words, fs, fmt, S, seeds=seeds, dither=31, device=local)
    if args.kernel != "auto":
        ex.set_kernel({"generic": avdsp_b200.KERNEL_GENERIC, "chain": avdsp_b200.KERNEL_CHAIN, "mix": avdsp_b200.KERNEL_MIX,
                       "fir": avdsp_b200.KERNEL_FIR, "fir_tc": avdsp_b200.KERNEL_FIR_TC,
                       "chain_v2": avdsp_b200.KERNEL_CHAIN_V2, "chain_v3": avdsp_b200.KERNEL_CHAIN_V3, "dag": avdsp_b200.KERNEL_DAG}[args.kernel])
    n_in, n_out = ex.n_in, ex.n_out
    x = synth.pcm_torch("noise", S, T, n_in, dev, first_stream=first)       # synthetic PCM, resident in HBM
    y = torch.empty((S, T, n_out), dtype=torch.int32, device=dev)

    # ---- device-resident timing: K steps bracketed by barrier+sync, CUDA events on the launch stream
    for _ in range(args.warmup):
        ex.process(x, out=y)
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    l0 = ex.launch_count
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for a, b in evs:
        a.record()
        ex.process(x, out=y)
        b.record()
    e1.record()
    barrier()
    total_ms = e0.elapsed_time(e1)
    launches = ex.launch_count - l0
    launches_per_step = max(launches // max(args.steps, 1), 1)
    kernel_ms = sum(a.elapsed_time(b) for a, b in evs) / max(args.steps, 1)      # all launches of one step (1 for the chain kernel, 3 for the mix path)
    timed_kernel, timed_variant = ex.last_kernel, ex.last_chain_variant            # of the device-resident step (the e2e leg runs other sizes)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, y, first)
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    frames_job = float(S_job) * T * args.steps
    value = frames_job * n_out / (total_ms * 1e-3) / 1e6

    # ---- end to end through the host-facing C-ABI call: pinned host PCM in, pinned host PCM out
    e2e = None
    if not args.no_e2e:
        # page-locked host PCM placed on the NUMA node next to this rank's GPU (avdsp_b200_host_alloc)
        xh = ex.alloc_pcm(T, n_in)
        yh = ex.alloc_pcm(T, n_out)
        xh[:] = x.cpu().numpy()
        torch.cuda.synchronize()

        def timed(fn, reps):
            barrier()
            t0 = time.perf_counter()
            for _ in range(reps):
                fn()                               # synchronous: returns when the outputs are in host memory
            torch.cuda.synchronize()
            dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            if dist is not None:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            return float(dt.item())

        for _ in range(2):
            ex.process_pinned(xh, yh)
        dt = timed(lambda: ex.process_pinned(xh, yh), args.steps)
        chk = int(yh[0, :64].astype(np.int64).sum())
        # the same DMA schedule without the kernel: what PCIe + host memory allow for this call on this box
        ex.copy_only(xh, yh)
        dtc = timed(lambda: ex.copy_only(xh, yh), max(2, args.steps // 2)) / max(2, args.steps // 2) * args.steps
        e2e = {"value": frames_job * n_out / dt / 1e6, "unit": "Msps",
               "h2d_bytes_per_step": S * T * n_in * 4, "d2h_bytes_per_step": S * T * n_out * 4,
               "ms_per_step": 1e3 * dt / args.steps, "checksum": chk,
               "host_buffers": "avdsp_b200_host_alloc: page-locked, on the NUMA node next to the GPU",
               "numa_node": ex.shards()[0][3],
               "roofline": {"bound": "pcie+host memory (copy-only run of the same call: same buffers, same 2-D chunked DMA schedule, no kernel)",
                            "achieved": (S * T * (n_in + n_out) * 4) * world / (dt / args.steps) / 1e9,
                            "peak": (S * T * (n_in + n_out) * 4) * world / (dtc / args.steps) / 1e9, "unit": "GB/s (both directions, whole job)",
                            "frac": dtc / dt}}
        # one C call over all GPUs of the box (avdsp_b200_create_multi), timed on rank 0 while the other ranks idle
        if world > 1 and not args.no_multi:
            ex_m = None
            barrier()
            if rank == 0:
                ex_m = avdsp_b200.Executor(words, fs, fmt, S_job, seeds=np.arange(S_job, dtype=np.int32), dither=31, devices=list(range(world)))
                xm = ex_m.alloc_pcm(T, n_in)
                ym = ex_m.alloc_pcm(T, n_out)
                for a0 in range(0, S_job, S):            # synthetic PCM: rank 0's block repeated
                    nn = min(S, S_job - a0)
                    xm[a0:a0 + nn] = xh[:nn]
                ex_m.process(xm, out=ym)
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    ex_m.process(xm, out=ym)
                dtm = time.perf_counter() - t0
                e2e["multi_device_call"] = {"value": frames_job * n_out / dtm / 1e6, "unit": "Msps", "ms_per_step": 1e3 * dtm / args.steps,
                                            "api": "avdsp_b200_create_multi + avdsp_b200_process(HOST): one process, one call, one staging thread per GPU",
                                            "devices": world, "shards": ex_m.shards()}
                ex_m.close()
            barrier()
        del xh, yh

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peaks, peak_src = measured_peaks()
    alg_bytes = float(S) * T * (n_in + n_out) * 4               # read every input once + write every output once
    # DRAM bytes per launch of the dominant kernel, from the committed `ncu --set full` capture of this exact workload + kernel
    traffic = None
    kname = timed_kernel + (str(timed_variant) if timed_kernel == "chain" else "")       # chain2 / chain3
    prof_name = {("c2", "chain2"): "r1_chain2_c2", ("c2", "chain3"): "r1_chain3_c2", ("c5", "mix"): "r1_mix_c5", ("c4", "fir_tc"): "r1_firtc_i8_c4",
                 ("c4f", "fir_tc"): "r1_firtc_tf32_c4f", ("c4f", "fir"): "r1_fir_f32_c4f"}.get((args.workload, kname))
    prof = os.path.join(ROOT, "profiles", f"{prof_name}_ncu_summary.txt") if prof_name else None
    if prof and S == wl[3] and T == wl[4] and os.path.exists(prof):
        tot = 0.0
        for ln in open(prof):
            f = ln.split()
            if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                tot += float(f[2]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[f[1]]
        traffic = tot or None
    # `traffic` (DRAM bytes per launch) cannot be measured inside an un-profiled run: null here, and the figure of the committed
    # ncu capture of this workload + kernel is quoted beside it with its source (it does not follow code changes by itself)
    traffic_ncu = {"value": traffic, "source": f"profiles/{prof_name}_ncu_summary.txt (committed `ncu --set full` capture, not this run)"} if traffic else None
    traffic = None
    common = {"traffic": traffic, "traffic_ncu": traffic_ncu, "kernel": f"k_{kname}", "kernel_ms": kernel_ms, "launches_per_step": launches_per_step}
    hbm = {"bound": "hbm", "achieved": alg_bytes / (kernel_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
           "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, **common}
    hbm["frac"] = hbm["achieved"] / hbm["peak"]
    alg_macs = float(S) * T * macs
    if fmt == 2:
        int_peak = avdsp_b200.measure_int_peak(local, 4096)
        pipe = {"bound": "int_pipe", "achieved": alg_macs / (kernel_ms * 1e-3) / 1e12, "peak": int_peak / 1e12,
                "unit": "T mad.wide.s32/s", "peak_source": "measured live (avdsp_b200_measure_int_peak)",
                "algorithmic_macs_per_launch": alg_macs, **common}
    else:
        # DSP_FORMAT 3: a MAC is a truncating multiply + a rounded add (no FMA: the reference rounds each product)
        int_peak = avdsp_b200.measure_f32_peak(local, 4096, False)
        packed = avdsp_b200.measure_f32_peak(local, 4096, True)
        pipe = {"bound": "fp32_pipe", "achieved": alg_macs / (kernel_ms * 1e-3) / 1e12, "peak": int_peak / 1e12,
                "unit": "T (mul.rz + add.rn)/s", "peak_source": "measured live (avdsp_b200_measure_f32_peak, scalar FMUL+FADD)",
                "peak_packed_f32x2": packed / 1e12, "algorithmic_macs_per_launch": alg_macs, **common}
    pipe["frac"] = pipe["achieved"] / pipe["peak"] if int_peak else None
    tensor = None
    if timed_kernel == "fir_tc":
        # Toeplitz GEMM on tcgen05: dense MMA operations issued per launch (kernel_fir_tc.cu geometry: 128-output blocks,
        # Hc + 128 samples of K per block; int8: 16 limb products per MAC, TF32: 3 passes)
        taps, paths = 4096, n_out
        hc = (taps + 127) // 128 * 128
        blocks = (T + 127) // 128
        if fmt == 2:
            tiles, ns, passes, kind, peak_tc = (S + 63) // 64, 64, 16, "int8 (kind::i8)", 2.0 * peaks["bf16_tflops"]
        else:
            tiles, ns, passes, kind, peak_tc = (S + 255) // 256, 256, 3, "tf32 (kind::tf32)", 0.5 * peaks["bf16_tflops"]
        ops = 2.0 * blocks * tiles * paths * passes * 128.0 * ns * (hc + 128)
        tensor = {"bound": "tensor", "achieved": ops / (kernel_ms * 1e-3) / 1e12, "peak": peak_tc, "unit": "TOP/s" if fmt == 2 else "TFLOP/s",
                  "peak_source": f"{peak_src}: dense bf16 x {'2' if fmt == 2 else '0.5'} for {kind} on the same tensor datapath",
                  "mma_ops_per_launch": ops, "useful_macs_per_launch": alg_macs,
                  "note": "kernel_ms covers pack + GEMM + delay-line update (3 launches)", **common}
        tensor["frac"] = tensor["achieved"] / tensor["peak"]
    # `roofline` is the BINDING one for the workload + kernel; the HBM figure is always kept beside it
    binding = tensor if tensor else (hbm if args.workload == "c5" else pipe)

    cpu = None
    if not args.no_cpu:
        cores = os.cpu_count() or 1
        fr = max(3000000 * 240 // macs // 1000 * 1000, 2000)     # ~1-1.5 s per host thread, ~20 core-seconds in total
        r = cpu_reference_rate(prog, fmt, fs, fr, cores)
        cpu = {"value": r["frames_per_s"] * r["n_out"] / 1e6, "unit": "Msps", "cores": r["cores"], "kind": r["kind"],
               "sample": f"{r['workers']} streams x {fr} frames of the same program and PCM recipe, one stream per host thread, "
                         f"{r['seconds']:.2f} s"}

    line = {"metric": "channel-samples/sec", "value": value, "unit": "Msps", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "int64" if fmt == 2 else "f32", "data": "synthetic",
            "config": workload_config(desc, prog, S if args.scaling == "weak" else S_job, T, fs, n_in, n_out),
            "run": {"l2": f"inputs+outputs {alg_bytes / 1e9:.2f} GB per step >> 126 MB L2 (no flush needed)",
                    "kernel": kname, "frames_per_s": frames_job / (total_ms * 1e-3), "streams_job": S_job, "streams_this_rank": S},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": binding, "roofline_hbm": hbm, ("roofline_int" if fmt == 2 else "roofline_fp32"): pipe, "cpu_baseline": cpu}
    print(json.dumps(line), file=json_out, flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
