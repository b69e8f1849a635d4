"""tools/bench_extra.py — device-resident throughput of the non-headline BASELINE configs (1a, 1b, 3, 4, 5) and of the
element-wise "next" rows (pw).
One JSON line per config. Inputs are generated on the device; timing = CUDA events over `steps` passes.
    python tools/bench_extra.py [--configs 1a,1b,3,4,5] [--steps 5]"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from qdsp_b200 import blocks as B, lib  # noqa: E402

L = lib.load()
FS = 2.4e6


def timed(fn, steps, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="1a,1b,3,4,5,pw")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--n3", type=int, default=1 << 26, help="samples for config 3 (full config: 2^30)")
    ap.add_argument("--n4", type=int, default=1 << 24, help="wideband samples for config 4 (full: 2^26)")
    ap.add_argument("--nch", type=int, default=32, help="channels on this GPU for config 4 (256 / 8 GPUs)")
    args = ap.parse_args()
    cfgs = args.configs.split(",")
    sp = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    hbm = 6549.1
    fp32 = L.qdsp_measure_fp32_peak(1, 20000)
    print(json.dumps({"probe": "fp32_peak_ffma2_tflops", "value": fp32, "ffma_tflops": L.qdsp_measure_fp32_peak(0, 20000)}), flush=True)

    def uniform(n, seed):
        x = torch.empty(n, dtype=torch.complex64, device="cuda")
        lib.check(L.qdsp_synth_uniform_cf32(x.data_ptr(), seed, 0, n, sp))
        return x

    if "1a" in cfgs or "1b" in cfgs:
        n = 1 << 24
        x = uniform(n, 1)
        win = B.BlackmanWindow(300e3, 4 * FS / 127, FS)
        if "1a" in cfgs:
            f = B.FIR(win)
            y = torch.empty(n, dtype=torch.complex64, device="cuda")
            ms = timed(lambda: f.process_device(x.data_ptr(), y.data_ptr(), n, stream=sp), args.steps)
            print(json.dumps({"config": "1a FIR 127 taps, 2^24 cf32", "ms": ms, "Msamples_s": n / ms / 1e3,
                              "tflops": 508 * n / ms / 1e9, "frac_fp32_measured": 508 * n / ms / 1e9 / fp32,
                              "hbm_gbs": 16 * n / ms / 1e6}), flush=True)
        if "1b" in cfgs:
            r = B.PolyphaseResampler(win, FS, FS / 4)
            y = torch.empty(n // 4 + 64, dtype=torch.complex64, device="cuda")
            ms = timed(lambda: r.process_device(x.data_ptr(), y.data_ptr(), n, 524288, stream=sp), args.steps)
            print(json.dumps({"config": "1b FIR 127 taps + decimate 4 (PolyphaseResampler I=1,D=4), 2^24 cf32, blocks of 524288",
                              "ms": ms, "Msamples_s": n / ms / 1e3, "tflops": 127 * n / ms / 1e9,
                              "hbm_gbs": 10 * n / ms / 1e6, "frac_hbm_measured": 10 * n / ms / 1e6 / hbm}), flush=True)
        del x
    if "3" in cfgs:
        n = args.n3
        x = uniform(n, 3)
        f = B.FIR(B.BlackmanWindow(100e3, 4 * FS / 4095, FS))
        y = torch.empty(n, dtype=torch.complex64, device="cuda")
        ms = timed(lambda: f.process_device(x.data_ptr(), y.data_ptr(), n, stream=sp), max(2, args.steps // 2), warmup=1)
        print(json.dumps({"config": f"3 FIR 4095 taps, {n} cf32 (one shard)", "ms": ms, "Msamples_s": n / ms / 1e3,
                          "tflops": 16380 * n / ms / 1e9, "frac_fp32_measured": 16380 * n / ms / 1e9 / fp32,
                          "frac_fp32_nominal_74.4": 16380 * n / ms / 1e9 / 74.4}), flush=True)
        del x, y
    if "4" in cfgs:
        n, nch = args.n4, args.nch
        x = uniform(n, 4)
        offs = np.asarray([(2 * k - 255) * 240e3 / 2 for k in range(nch)], np.float32)
        ch = B.Channelizer(offs, 61.44e6, 48e3, 48e3, 5e3)
        stride = n // 1280 + 64
        y = torch.empty(nch * stride, dtype=torch.float32, device="cuda")
        ms = timed(lambda: ch.process_device(x.data_ptr(), y.data_ptr(), n, stride, 819200, stream=sp), max(2, args.steps // 2), warmup=1)
        print(json.dumps({"config": f"4 channelizer {nch} ch/GPU, 61.44 MS/s -> 48 kS/s (10241 taps, D=1280), {n} wideband cf32",
                          "ms": ms, "wideband_Msamples_s": n / ms / 1e3, "channel_Msamples_s": nch * n / ms / 1e3,
                          "tflops": 38.0 * nch * n / ms / 1e9, "frac_fp32_measured": 38.0 * nch * n / ms / 1e9 / fp32}), flush=True)
        del x, y
    if "5" in cfgs:
        n = 1 << 26
        x = uniform(n, 5)
        y = torch.empty(n, dtype=torch.complex64, device="cuda")
        for name, blk, bytes_per in [("BFMDeemp", B.BFMDeemp(48e3, 50e-6), 16), ("ComplexAGC", B.ComplexAGC(1.0, 65535.0, 1e-3), 16),
                                     ("CostasLoop<4> chunk 2048 warmup 2048", B.CostasLoop(4, 0.004), 16),
                                     ("FeedForwardAGC", B.FeedForwardAGC(), 16), ("FrequencyXlator", B.FrequencyXlator(FS, -250e3), 16)]:
            if "Costas" in name:
                blk.set_chunking(2048, 2048)
            ms = timed(lambda: blk.process_device(x.data_ptr(), y.data_ptr(), n, stream=sp), args.steps, warmup=1)
            print(json.dumps({"config": f"5 {name}, {n} elements", "ms": ms, "Msamples_s": n / ms / 1e3,
                              "hbm_gbs": bytes_per * n / ms / 1e6, "frac_hbm_measured": bytes_per * n / ms / 1e6 / hbm}), flush=True)
        xf = x.view(torch.float32)
        yf = y.view(torch.float32)
        agc = B.AGC(20.0, 48e3)
        ms = timed(lambda: agc.process_device(xf.data_ptr(), yf.data_ptr(), 2 * n, 1000000, stream=sp), args.steps, warmup=1)
        print(json.dumps({"config": f"5 AGC, {2 * n} floats, run() blocks of 1e6", "ms": ms, "Msamples_s": 2 * n / ms / 1e3,
                          "hbm_gbs": 8 * 2 * n / ms / 1e6, "frac_hbm_measured": 8 * 2 * n / ms / 1e6 / hbm}), flush=True)
    if "pw" in cfgs:
        # element-wise / layout / per-block-statistic rows: all HBM-bound, algorithmic bytes per sample in the table
        n = 1 << 26
        x = uniform(n, 6)
        x2 = uniform(n, 7)
        y = torch.empty(n, dtype=torch.complex64, device="cuda")
        Lc = lib.load()
        xp, x2p, yp = x.data_ptr(), x2.data_ptr(), y.data_ptr()
        am, sq, ssb, di = B.AMDemod(), B.Squelch(-30.0), B.SSBDemod(48e3, 3e3, 0), B.DelayImag()
        rows = [
            ("Add<complex_t>", 24, lambda: Lc.qdsp_math_process(0, 1, xp, x2p, yp, n, sp)),
            ("Multiply<complex_t>", 24, lambda: Lc.qdsp_math_process(2, 1, xp, x2p, yp, n, sp)),
            ("StereoToMono", 12, lambda: Lc.qdsp_layout_process(2, xp, None, yp, None, n, sp)),
            ("StereoToChannels", 16, lambda: Lc.qdsp_layout_process(3, xp, None, yp, yp + 4 * n, n, sp)),
            ("Volume<stereo_t>", 16, lambda: Lc.qdsp_volume_process(1, 0.49, 0, xp, yp, n, sp)),
            ("DelayImag", 16, lambda: di.process_device(xp, yp, n, stream=sp)),
            ("AMDemod, run() blocks of 1e6 (12 B algorithmic, 20 B moved)", 12, lambda: am.process_device(xp, yp, n, 1000000, stream=sp)),
            ("Squelch, run() blocks of 1e6 (16 B algorithmic, 24 B moved)", 16, lambda: sq.process_device(xp, yp, n, 1000000, stream=sp)),
            ("SSBDemod", 12, lambda: ssb.process_device(xp, yp, n, stream=sp)),
        ]
        # Mueller & Mueller clock recovery: sequential-exact, one warp per stream (latency bound by construction)
        try:
            taps = np.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                                        "reference_vectors.npz"))["interp_taps"]
            nm = 1 << 22
            mm = B.MMClockRecovery(4.0, (0.01 * 0.01) / 4, 0.01, 0.005, taps)
            ms = timed(lambda: mm.process_device(xp, yp, nm, 1000000, stream=sp), 3, warmup=1)
            print(json.dumps({"config": f"pw MMClockRecovery<complex_t> omega=4, {nm} samples (one stream, sequential-exact)", "ms": ms,
                              "Msamples_s": nm / ms / 1e3, "Msymbols_s": nm / 4 / ms / 1e3}), flush=True)
        except Exception as e:  # noqa: BLE001
            print(json.dumps({"config": "pw MMClockRecovery", "error": str(e)}), flush=True)
        for name, bytes_per, fn in rows:
            ms = timed(fn, args.steps, warmup=1)
            print(json.dumps({"config": f"pw {name}, {n} elements", "ms": ms, "Msamples_s": n / ms / 1e3,
                              "hbm_gbs": bytes_per * n / ms / 1e6, "frac_hbm_measured": bytes_per * n / ms / 1e6 / hbm}), flush=True)


if __name__ == "__main__":
    main()
