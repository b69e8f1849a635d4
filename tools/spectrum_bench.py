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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="append the JSON lines to this file as well")
    ap.add_argument("--profile", action="store_true", help="device time per kernel of one call per size instead")
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
