"""tools/vfofm_formats.py — the fused VFO -> FM chain (config 2's step) fed cf32, cs16, cs8 and cu8 input.

    python tools/vfofm_formats.py [--out FILE.jsonl] [--rounds 5] [--samples 268435456] [--steps 100] [--e2e-samples 67108864]

Device-resident: every format gets its own handle and input buffer (2^28 samples per call by default: every format's
input exceeds the 126 MB L2), and bench.py's burst pattern -- warm-up calls, then `--steps` calls on the same input and
audio buffers with the per-launch timing ring on, one CUDA event pair around the burst. An integer call is the
conversion (qdsp_iq_convert_process) and the cf32 kernel; the `*_convert_only` arms time the conversion alone (TB/s
of its read + write). End to end: process_host from
pinned host memory, next to a plain pinned H2D copy of the same bytes (the bus ceiling for that format). The formats
alternate `--rounds` times in one process. The card's name, power limit and SM clocks are recorded in the same run.
One JSON line per measurement, then one summary line per format (medians). Without --out the lines go to stdout only."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, REPO)
BLOCK = 819_200
FS, FC, FM, DEV = 2_400_000, 250_000, 1_000, 5e3
OUT_SR, BW = 48e3, 48e3
FORMATS = ["cf32", "cs16", "cs8", "cu8"]
CODES = {"cs16": 2, "cs8": 3, "cu8": 4}
SCALE = {"cs16": (1 / 32768, 0.0), "cs8": (1 / 128, 0.0), "cu8": (1 / 128, -127.5)}


def smi():
    q = "name,power.limit,clocks.sm,clocks.max.sm,temperature.gpu"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unavailable"


def quantize(torch, x, fmt):
    """cf32 device tensor -> interleaved integer pairs (synth.quantize_iq on the GPU)."""
    r = torch.view_as_real(x).reshape(-1)
    if fmt == "cs16":
        return torch.round(r * 32768.0).clamp_(-32768, 32767).to(torch.int16)
    if fmt == "cs8":
        return torch.round(r * 128.0).clamp_(-128, 127).to(torch.int8)
    return torch.round(r * 128.0 + 127.5).clamp_(0, 255).to(torch.uint8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--samples", type=int, default=1 << 28)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--e2e-samples", type=int, default=1 << 26)
    ap.add_argument("--e2e-steps", type=int, default=3)
    a = ap.parse_args()

    import torch
    from qdsp_b200 import blocks as B, lib

    L = lib.load()
    lib.require_device()
    dev = torch.device("cuda:0")
    sp = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    lines = []

    def emit(rec):
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)

    card = smi()
    emit({"kind": "card", "nvidia_smi": card, "query": "name, power.limit, clocks.sm, clocks.max.sm, temperature.gpu"})

    # ---- device-resident ------------------------------------------------------------------------------------------
    n = a.samples
    x = torch.empty(n, dtype=torch.complex64, device=dev)
    lib.check(L.qdsp_synth_fm_cf32(x.data_ptr(), 0, n, FS, FC, FM, DEV, 0.5, 0.005, 2, sp))
    inputs = {"cf32": x}
    for f in FORMATS[1:]:
        inputs[f] = quantize(torch, x, f)
    chains, audio = {}, {}
    for f in FORMATS:
        chains[f] = B.VFOFM(float(FC), float(FS), OUT_SR, BW, DEV)
        if f != "cf32":
            chains[f].set_input_format(f)
    n_out = chains["cf32"].out_count(n, BLOCK)
    for f in FORMATS:
        audio[f] = torch.empty(n_out + 64, dtype=torch.float32, device=dev)
    torch.cuda.synchronize()

    conv = torch.empty(n, dtype=torch.complex64, device=dev)

    def step(f):
        if f.endswith("_convert_only"):   # qdsp_iq_convert_process alone: the conversion's share of an integer call
            g = f.split("_")[0]
            lib.check(L.qdsp_iq_convert_process(CODES[g], *SCALE[g], inputs[g].data_ptr(), conv.data_ptr(), n, sp), "convert")
            return
        m = L.qdsp_vfofm_process(chains[f].h, inputs[f].data_ptr(), audio[f].data_ptr(), None, n, None, 0, BLOCK, None, sp)
        if m != n_out:
            raise SystemExit(f"{f}: process returned {m}, expected {n_out}: {lib.last_error()}")

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    arms = FORMATS + [f + "_convert_only" for f in FORMATS[1:]]
    dev_rates = {f: [] for f in arms}
    for r in range(a.rounds):
        for f in arms:
            for _ in range(a.warmup):
                step(f)
            torch.cuda.synchronize()
            ring = not f.endswith("_convert_only")
            if ring:
                lib.check(L.qdsp_vfofm_enable_timing_ring(chains[f].h, a.steps), "ring")
            launches0 = L.qdsp_launch_count()
            e0.record()
            for _ in range(a.steps):
                step(f)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            nrec = C.c_int(0)
            k_ms = float(L.qdsp_vfofm_kernel_ms_mean(chains[f].h, C.byref(nrec))) if ring else None
            gs = n * a.steps / (ms * 1e-3) / 1e9
            dev_rates[f].append(gs)
            in_b = inputs[f.split("_")[0]].numel() * inputs[f.split("_")[0]].element_size() / n
            rec = {"kind": "device", "round": r, "format": f, "samples_per_call": n, "calls": a.steps, "ms": ms,
                   "gsps": gs, "kernel_ms_mean": k_ms, "launches": L.qdsp_launch_count() - launches0, "in_bytes_per_sample": in_b}
            if not ring:   # read + write of the conversion
                rec["tbps"] = n * (in_b + 8) * a.steps / (ms * 1e-3) / 1e12
            emit(rec)
    del inputs, x, conv
    torch.cuda.synchronize()
    torch.cuda.empty_cache()

    # ---- end to end -----------------------------------------------------------------------------------------------
    ne = a.e2e_samples
    xe = torch.empty(ne, dtype=torch.complex64, device=dev)
    lib.check(L.qdsp_synth_fm_cf32(xe.data_ptr(), 0, ne, FS, FC, FM, DEV, 0.5, 0.005, 2, sp))
    host = {"cf32": torch.empty(ne, dtype=torch.complex64, pin_memory=True)}
    host["cf32"].copy_(xe)
    for f in FORMATS[1:]:
        q = quantize(torch, xe, f)
        host[f] = torch.empty(q.numel(), dtype=q.dtype, pin_memory=True)
        host[f].copy_(q)
        del q
    del xe
    ne_out = chains["cf32"].out_count(ne, BLOCK)
    yh = torch.empty(ne_out + 64, dtype=torch.float32, pin_memory=True)
    torch.cuda.synchronize()
    e2e_chains = {}
    for f in FORMATS:
        e2e_chains[f] = B.VFOFM(float(FC), float(FS), OUT_SR, BW, DEV)
        if f != "cf32":
            e2e_chains[f].set_input_format(f)
    e2e_rates = {f: [] for f in FORMATS}
    e2e_frac = {f: [] for f in FORMATS}
    for r in range(a.rounds):
        for f in FORMATS:
            h = host[f]
            nbytes = h.numel() * h.element_size()
            dcopy = torch.empty(h.numel(), dtype=h.dtype, device=dev)
            m = L.qdsp_vfofm_process_host(e2e_chains[f].h, h.data_ptr(), yh.data_ptr(), ne, BLOCK, sp)   # warm
            if m != ne_out:
                raise SystemExit(f"{f}: process_host returned {m}: {lib.last_error()}")
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(a.e2e_steps):
                L.qdsp_vfofm_process_host(e2e_chains[f].h, h.data_ptr(), yh.data_ptr(), ne, BLOCK, sp)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            dcopy.copy_(h, non_blocking=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(a.e2e_steps):
                dcopy.copy_(h, non_blocking=True)
            torch.cuda.synchronize()
            dtc = time.perf_counter() - t0
            del dcopy
            gs = ne * a.e2e_steps / dt / 1e9
            frac = (nbytes * a.e2e_steps / dt) / (nbytes * a.e2e_steps / dtc)
            e2e_rates[f].append(gs)
            e2e_frac[f].append(frac)
            emit({"kind": "e2e", "round": r, "format": f, "samples_per_call": ne, "calls": a.e2e_steps, "gsps": gs,
                  "h2d_bytes_per_call": nbytes, "h2d_gbs": nbytes * a.e2e_steps / dt / 1e9,
                  "copy_alone_gbs": nbytes * a.e2e_steps / dtc / 1e9, "frac_of_h2d_copy": frac})
    card_after = smi()
    for f in arms:
        emit({"kind": "summary", "format": f, "device_gsps_median": statistics.median(dev_rates[f]),
              "device_gsps_spread": max(dev_rates[f]) - min(dev_rates[f]),
              "device_vs_cf32": statistics.median(dev_rates[f]) / statistics.median(dev_rates["cf32"])})
    for f in FORMATS:
        emit({"kind": "summary_e2e", "format": f,
              "e2e_gsps_median": statistics.median(e2e_rates[f]), "e2e_frac_of_h2d_copy_median": statistics.median(e2e_frac[f]),
              "nvidia_smi_before": card, "nvidia_smi_after": card_after})
    if a.out:
        with open(a.out, "w") as fo:
            fo.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
