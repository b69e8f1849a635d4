"""Throughput of the power-spectrum block (qdsp_spectrum_process) on one GPU.

Input: 2^28 device-resident cf32 samples (2 GiB, larger than L2) of config 4's wideband comb. For each FFT size N in
{1024, 4096, 16384} and hop in {N, N/2}, at average = 64: warm-up calls, then a timed region of at least 0.7 s of
back-to-back calls over the whole input on one handle, timed with CUDA events. One JSON line per size:

  gsps             samples per second / 1e9
  alg_bytes_per_sample  8 min(1, N / hop) (samples read) + 4 N / (A hop) (rows written)
  alg_flop_per_sample   (5 N log2 N + 8 N) / hop (FFT, window and power)
  hbm_frac, fp32_frac   achieved algorithmic bytes/s over the HBM copy peak (bench.measured_peaks()), flop/s over
                        nominal FP32 (bench.FP32_NOMINAL_TFLOPS); `bound` names the larger of the two least times
  gpu, power_limit_w, sm_clock_mhz, sm_clock_max_mhz   nvidia-smi, read right after the timed region

  python tools/spectrum_bench.py [--out FILE.jsonl]
  python tools/spectrum_bench.py --profile [--out FILE.jsonl]
        one call per size under torch.profiler (CUDA activities) instead: device time and launches per kernel, and the
        frames kernel's algorithmic input bandwidth (8 min(1, N / hop) bytes per sample over its device time)
  python tools/spectrum_bench.py --format cs16,cs8,cu8 [--reps R] [--out FILE.jsonl]
        integer input instead: the same comb quantised to each format (synth.quantize_iq, usual scale / offset), 2^28
        pairs per call, N in {1024, 4096, 16384} x hop in {N, 8N} x average in {1, 64}. Three arms per point, each a timed
        region of at least 0.7 s of back-to-back calls (CUDA events), alternated R times (default 2) in this order:
          native   qdsp_spectrum_process on the integer pairs after set_input_format: what the handle runs, which is
                   the frames kernel reading them, except at N = 16384 with hop <= N, where the handle converts first
                   (`path` in the record: "native" or "convert first")
          convert  qdsp_iq_convert_process into a cf32 buffer, then qdsp_spectrum_process on that
          cf32     qdsp_spectrum_process on the comb itself (the reference rate; the same for every format)
        One JSON line per point: the input rate of each arm in GS/s (every repetition, and the median), and
        native_over_convert, the ratio of the medians.
"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_SAMPLES = 1 << 28
AVERAGE = 64
MIN_SECONDS = 0.7


def smi():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, pl, sm, smax = [v.strip() for v in out.split(",")]
    return {"gpu": name, "power_limit_w": float(pl), "sm_clock_mhz": float(sm), "sm_clock_max_mhz": float(smax)}


def profile_call(torch, h, x, out, N, hop, hbm_gbs):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        h.process_device(x.ptr, out.ptr, N_SAMPLES)
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = getattr(ev, "device_time_total", None)
        if us is None:
            us = ev.cuda_time_total
        k = kern.setdefault(ev.name, [0, 0.0])
        k[0] += 1
        k[1] += us
    rec = {"block": "spectrum", "profile": "torch.profiler, CUDA activities, one call", "fftSize": N, "hop": hop,
           "average": AVERAGE, "samples_per_call": N_SAMPLES,
           "kernels": {n: {"launches": c, "us": round(t, 1)} for n, (c, t) in sorted(kern.items(), key=lambda kv: -kv[1][1])}}
    frames_us = sum(t for n, (c, t) in kern.items() if "spectrum_frames_kernel" in n)
    total_us = sum(t for c, t in kern.values())
    if frames_us > 0:
        in_bytes = 8.0 * min(1.0, N / hop) * N_SAMPLES
        rec["frames_kernel_share"] = round(frames_us / total_us, 4)
        rec["frames_kernel_input_gbs"] = round(in_bytes / (frames_us * 1e-6) / 1e9, 1)
        rec["frames_kernel_hbm_frac"] = round(rec["frames_kernel_input_gbs"] / hbm_gbs, 4)
    return rec


def timed_gsps(torch, stream, call):
    """Warm-up, then back-to-back calls for at least MIN_SECONDS between two CUDA events: samples per second / 1e9."""
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    call()
    e1.record(stream)
    e1.synchronize()
    iters = max(3, math.ceil(MIN_SECONDS / (e0.elapsed_time(e1) * 1e-3)))
    e0.record(stream)
    for _ in range(iters):
        call()
    e1.record(stream)
    e1.synchronize()
    return N_SAMPLES * iters / (e0.elapsed_time(e1) * 1e-3) / 1e9


def bench_formats(torch, args, L, B, x):
    """Integer input: the native read against convert-then-cf32, with the cf32 rate beside them (module docstring)."""
    import numpy as np

    from qdsp_b200 import lib, synth

    stream = torch.cuda.current_stream()
    fmts = args.format.split(",")
    chunk = 1 << 24
    raws = {}
    for fmt in fmts:
        # the comb quantised on the host in chunks, as a radio front end would deliver it
        dt = synth.IQ_FORMATS[fmt][0]
        host = np.empty(2 * N_SAMPLES, dt)
        for c0 in range(0, N_SAMPLES, chunk):
            host[2 * c0:2 * (c0 + chunk)] = synth.quantize_iq(x.to_numpy(np.complex64, chunk, offset_bytes=8 * c0), fmt)
        raws[fmt] = B.DevBuf.from_numpy(host)
        del host
    conv = B.DevBuf(N_SAMPLES * 8)
    records = []
    for N in (1024, 4096, 16384):
        for hop in (N, 8 * N):
            for A in (1, AVERAGE):
                rows_max = N_SAMPLES // (hop * A) + 2
                out = B.DevBuf(rows_max * N * 4)
                ref = B.Spectrum(N, None, hop, A)
                hs = {}
                for fmt in fmts:
                    hs[fmt] = (B.Spectrum(N, None, hop, A), B.Spectrum(N, None, hop, A))
                    hs[fmt][0].set_input_format(fmt)
                arms = {("cf32", None): []}
                for fmt in fmts:
                    arms[("native", fmt)] = []
                    arms[("convert", fmt)] = []

                def run(arm, fmt):
                    if arm == "cf32":
                        return lambda: ref.process_device(x.ptr, out.ptr, N_SAMPLES)
                    if arm == "native":
                        return lambda: hs[fmt][0].process_device(raws[fmt].ptr, out.ptr, N_SAMPLES)
                    _, code, sc, off = B._iq_format(fmt)

                    def call():
                        lib.check(L.qdsp_iq_convert_process(code, sc, off, raws[fmt].ptr, conv.ptr, N_SAMPLES, None))
                        hs[fmt][1].process_device(conv.ptr, out.ptr, N_SAMPLES)
                    return call

                for _ in range(args.reps):
                    for (arm, fmt) in arms:
                        arms[(arm, fmt)].append(round(timed_gsps(torch, stream, run(arm, fmt)), 2))
                gpu = smi()
                cf = arms[("cf32", None)]
                for fmt in fmts:
                    nat, cvt = arms[("native", fmt)], arms[("convert", fmt)]
                    rec = {"block": "spectrum", "format": fmt, "fftSize": N, "hop": hop, "average": A,
                           "path": "native" if N // 16 <= 512 or hop > N else "convert first",
                           "samples_per_call": N_SAMPLES, "min_seconds_per_arm": MIN_SECONDS,
                           "native_gsps": nat, "convert_gsps": cvt, "cf32_gsps": cf,
                           "native_gsps_median": float(np.median(nat)), "convert_gsps_median": float(np.median(cvt)),
                           "cf32_gsps_median": float(np.median(cf)),
                           "native_over_convert": round(float(np.median(nat) / np.median(cvt)), 4)}
                    rec.update(gpu)
                    records.append(rec)
                    print(json.dumps(rec), flush=True)
                for a, b in hs.values():
                    a.close()
                    b.close()
                ref.close()
                out.free()
    return records


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="append the JSON lines to this file as well")
    ap.add_argument("--profile", action="store_true", help="device time per kernel of one call per size instead")
    ap.add_argument("--format", help="integer input: comma-separated cs16 / cs8 / cu8 (module docstring)")
    ap.add_argument("--reps", type=int, default=2, help="--format: repetitions of the alternated arms")
    args = ap.parse_args()

    import torch

    import bench
    from qdsp_b200 import blocks as B, lib

    lib.require_device()
    L = lib.load()
    hbm_gbs, hbm_src = bench.measured_peaks()
    fp32_gflops = bench.FP32_NOMINAL_TFLOPS * 1e3
    x = B.DevBuf(N_SAMPLES * 8)
    lib.check(L.qdsp_synth_comb_cf32(x.ptr, 0, N_SAMPLES, 61_440_000, 256, 240_000, 5e3, 1.0 / 64.0, 0.001, 4, None))
    stream = torch.cuda.current_stream()
    if args.format:
        records = bench_formats(torch, args, L, B, x)
        if args.out:
            with open(args.out, "a") as f:
                for r in records:
                    f.write(json.dumps(r) + "\n")
        return
    records = []
    for N in (1024, 4096, 16384):
        for hop in (N, N // 2):
            h = B.Spectrum(N, None, hop, AVERAGE)
            rows_max = N_SAMPLES // (hop * AVERAGE) + 2
            out = B.DevBuf(rows_max * N * 4)
            for _ in range(2):
                h.process_device(x.ptr, out.ptr, N_SAMPLES)
            torch.cuda.synchronize()
            if args.profile:
                rec = profile_call(torch, h, x, out, N, hop, hbm_gbs)
                rec.update(smi())
                records.append(rec)
                print(json.dumps(rec), flush=True)
                h.close()
                out.free()
                continue
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            h.process_device(x.ptr, out.ptr, N_SAMPLES)
            e1.record(stream)
            e1.synchronize()
            iters = max(3, math.ceil(MIN_SECONDS / (e0.elapsed_time(e1) * 1e-3)))
            e0.record(stream)
            for _ in range(iters):
                h.process_device(x.ptr, out.ptr, N_SAMPLES)
            e1.record(stream)
            e1.synchronize()
            sec = e0.elapsed_time(e1) * 1e-3
            gsps = N_SAMPLES * iters / sec / 1e9
            bps = 8.0 * min(1.0, N / hop) + 4.0 * N / (AVERAGE * hop)
            fps = (5.0 * N * math.log2(N) + 8.0 * N) / hop
            rec = {"block": "spectrum", "fftSize": N, "hop": hop, "average": AVERAGE, "samples_per_call": N_SAMPLES,
                   "calls": iters, "seconds": round(sec, 4), "gsps": round(gsps, 2),
                   "alg_bytes_per_sample": round(bps, 4), "alg_flop_per_sample": round(fps, 2),
                   "hbm_gbs": round(gsps * bps, 1), "hbm_peak_gbs": hbm_gbs, "hbm_peak_source": hbm_src,
                   "hbm_frac": round(gsps * bps / hbm_gbs, 4), "fp32_frac": round(gsps * fps / fp32_gflops, 4),
                   "bound": "hbm" if bps / hbm_gbs >= fps / fp32_gflops else "fp32"}
            rec.update(smi())
            records.append(rec)
            print(json.dumps(rec), flush=True)
            h.close()
            out.free()
    if args.out:
        with open(args.out, "a") as f:
            for r in records:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
