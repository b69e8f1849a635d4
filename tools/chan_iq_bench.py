"""Cost of the channelizer's complex-baseband output (qdsp_channelizer_process_iq) on one GPU, at config 4's geometry.

Input: 2^26 device-resident cf32 samples of config 4's 256-channel comb (61.44 MS/s, 10 241 taps, D = 1280), run() blocks of
819 200 samples, one handle per arm, each seeked to 0 as bench.py's cfg4 does at N = 1. Arms:

  fft_audio       FFT polyphase form, audio only (qdsp_channelizer_process: bench.py configs.cfg4's path)
  fft_iq_audio    FFT polyphase form, IQ + audio
  fft_iq          FFT polyphase form, IQ only (audio_out_dev = NULL)
  direct_iq_audio direct form (variant 2), IQ + audio

The arms alternate: `--rounds` rounds, each timing every arm over at least 0.7 s of back-to-back calls with CUDA events
after warm-up calls. One JSON line per (round, arm):

  gsps                 wideband input samples per second / 1e9 (all 256 channels produced)
  store_bytes_per_sample  bytes the arm stores per input sample: 256 x (4 audio + 8 IQ) / 1280
  gpu, power_limit_w, sm_clock_mhz, sm_clock_max_mhz   nvidia-smi, read right after the timed region

  python tools/chan_iq_bench.py [--rounds R] [--out FILE.jsonl]
"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_SAMPLES = 1 << 26
BLOCK = 819_200
NCH, FS, SPACING, D = 256, 61_440_000, 240_000, 1280
MIN_SECONDS = 0.7


def smi():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, pl, sm, smax = [v.strip() for v in out.split(",")]
    return {"gpu": name, "power_limit_w": float(pl), "sm_clock_mhz": float(sm), "sm_clock_max_mhz": float(smax)}


def timed(torch, step, warmup=3):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    step()
    e1.record()
    e1.synchronize()
    k = max(3, math.ceil(MIN_SECONDS * 1e3 / max(e0.elapsed_time(e1), 1e-3)))
    e0.record()
    for _ in range(k):
        step()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / k, k


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    from qdsp_b200 import blocks as B, lib, synth

    L = lib.load()
    lib.require_device()
    torch.cuda.init()
    n = N_SAMPLES
    x = B.DevBuf(n * 8)
    lib.check(L.qdsp_synth_comb_cf32(x.ptr, 0, n, FS, NCH, SPACING, 5e3, 1.0 / 64.0, 0.001, 4, None))
    stride = n // D + 64
    audio = B.DevBuf(NCH * stride * 4)
    iq = B.DevBuf(NCH * stride * 8)
    offs = synth.cfg4_offsets(NCH, SPACING)

    def handle(variant):
        ch = B.Channelizer(offs, float(FS), 48e3, 48e3, 5e3)
        ch.set_variant(variant)
        ch.seek(0)
        return ch

    hs = {"fft_audio": handle(0), "fft_iq_audio": handle(0), "fft_iq": handle(0), "direct_iq_audio": handle(2)}
    arms = {
        "fft_audio": (lambda: hs["fft_audio"].process_device(x.ptr, audio.ptr, n, stride, BLOCK), 4),
        "fft_iq_audio": (lambda: hs["fft_iq_audio"].process_device_iq(x.ptr, iq.ptr, audio.ptr, n, stride, BLOCK), 12),
        "fft_iq": (lambda: hs["fft_iq"].process_device_iq(x.ptr, iq.ptr, None, n, stride, BLOCK), 8),
        "direct_iq_audio": (lambda: hs["direct_iq_audio"].process_device_iq(x.ptr, iq.ptr, audio.ptr, n, stride, BLOCK), 12),
    }
    out = open(args.out, "a") if args.out else None
    for r in range(args.rounds):
        for name, (step, per_out) in arms.items():
            ms, k = timed(torch, step)
            rec = {"tool": "chan_iq_bench", "round": r, "arm": name, "samples_per_call": n, "block": BLOCK, "calls": k,
                   "ms_per_call": round(ms, 4), "gsps": round(n / ms / 1e6, 2),
                   "store_bytes_per_sample": round(NCH * per_out / D, 2)}
            rec.update(smi())
            line = json.dumps(rec)
            print(line, flush=True)
            if out:
                out.write(line + "\n")
    if out:
        out.close()


if __name__ == "__main__":
    main()
