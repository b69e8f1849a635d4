"""tools/vfofm_trace.py — torch.profiler trace of back-to-back calls of the fused VFO -> FM chain (bench.py's timed pattern:
one handle, the same input and the same audio buffer every call, the per-launch timing ring on). Prints one JSON line per
kernel (start, end, and how long it ran alongside its predecessor) and writes the Chrome trace next to it.

    python tools/vfofm_trace.py [--calls 5] [--out DIR]      (DIR defaults to a new temporary directory)"""
import argparse
import ctypes as C
import json
import os
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from qdsp_b200 import blocks as B, lib  # noqa: E402

N, BLOCK = 1 << 28, 819_200
FS, FC, FM, DEV = 2_400_000, 250_000, 1_000, 5e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    a.out = a.out or tempfile.mkdtemp(prefix="vfofm_trace_")
    os.makedirs(a.out, exist_ok=True)
    L = lib.load()
    sp = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    x = torch.empty(N, dtype=torch.complex64, device="cuda")
    lib.check(L.qdsp_synth_fm_cf32(x.data_ptr(), 0, N, FS, FC, FM, DEV, 0.5, 0.005, 2, sp))
    chain = B.VFOFM(float(FC), float(FS), 48e3, 48e3, DEV)
    n_out = chain.out_count(N, BLOCK)
    audio = torch.empty(n_out + 64, dtype=torch.float32, device="cuda")

    def step():
        assert L.qdsp_vfofm_process(chain.h, x.data_ptr(), audio.data_ptr(), None, N, None, 0, BLOCK, None, sp) == n_out

    for _ in range(5):
        step()
    torch.cuda.synchronize()
    lib.check(L.qdsp_vfofm_enable_timing_ring(chain.h, a.calls), "enable_timing_ring")
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(a.calls):
            step()
        torch.cuda.synchronize()
    nrec = C.c_int(0)
    ring_ms = L.qdsp_vfofm_kernel_ms_mean(chain.h, C.byref(nrec))
    path = os.path.join(a.out, "vfofm_calls.pt.trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        ev = json.load(f)["traceEvents"]
    ks = sorted((e for e in ev if e.get("cat") == "kernel" and "decim_rowlane" in e.get("name", "")), key=lambda e: e["ts"])
    prev_end = None
    for i, e in enumerate(ks):
        start, end = float(e["ts"]), float(e["ts"]) + float(e["dur"])
        rec = {"kernel": i, "start_us": round(start - ks[0]["ts"], 2), "end_us": round(end - ks[0]["ts"], 2),
               "dur_us": round(float(e["dur"]), 2)}
        if prev_end is not None:
            rec["overlap_with_previous_us"] = round(prev_end - start, 2)
        print(json.dumps(rec))
        prev_end = end
    span = (float(ks[-1]["ts"]) + float(ks[-1]["dur"]) - float(ks[0]["ts"])) if ks else 0.0
    print(json.dumps({"kernels": len(ks), "first_start_to_last_end_us": round(span, 2), "us_per_call": round(span / max(len(ks), 1), 2),
                      "ring_us_mean": round(ring_ms * 1e3, 2), "ring_launches": nrec.value, "trace": path}))


if __name__ == "__main__":
    main()
