#!/usr/bin/env python
"""bench.py — benchmark of qdsp_b200 on the BASELINE.json configurations.

Headline (`value`, `e2e`, `roofline`): BASELINE.json configs[1] — the fused NCO xlator -> polyphase resampler
(2.4 MS/s -> 48 kS/s, 401 taps, I=1, D=50) -> FM quadrature demod chain on 2^28 synthetic cf32 samples per GPU, cut into
the reference's run() blocks of 819 200 samples. Metric: Msamples/s of INPUT cf32 consumed.

  python bench.py [--gpus N] [--steps K] [--warmup W]        our arm (one process per GPU under torchrun)
  python bench.py ... --dump-outputs DIR                      also write the output of the last timed step, DIR/audio.npy
  python bench.py --impl reference ...                        the reference's own CPU chain, same metric

One JSON line on stdout (rank 0). `value` = whole-job throughput with the input resident in HBM; `e2e` = the same chain
through the C-ABI host-buffer entry point (pinned host in/out, H2D + D2H timed); `roofline` = the fused kernel's
algorithmic bytes / its own CUDA-event duration vs the measured HBM peak; `cpu_baseline` = the unmodified reference
headers (oracle/_ref) timed on this box's host cores; `parity` = the timed run's own output checked against the CPU
oracle on windows (outside every timed region); `configs` = the other BASELINE configurations, each with its own
clocks sample and oracle check:
  cfg1a / cfg1b   127-tap FIR, and FIR + decimate-by-4, 2^24 samples                     (N = 1 only)
  cfg3            4095-tap FIR on 2^30 samples, TIME-SHARDED over the N ranks; the (taps-1)-sample halo is read by the
                  FIR kernel straight from the neighbour's memory over NVLink (CUDA IPC peer mapping)   (strong scaling)
  cfg4            256-channel channelizer off a 61.44 MS/s stream, FFT polyphase form (the default path for this geometry): all
                  256 channels on every GPU, the stream TIME-SHARDED (2^26 samples + lead-in per rank), no collective  (weak scaling)
  cfg4_direct     the same channelizer in direct form (the reference's algorithm), 2^26 samples, channels PARTITIONED over
                  the N ranks, no collective                                                             (strong scaling)
  cfg5            recurrent blocks (de-emphasis, ComplexAGC, AGC, FeedForwardAGC, Costas) on 2^28 samples (N = 1 only)
"""
import argparse
import ctypes as C
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_SAMPLES = 1 << 28          # per GPU (config 2)
BLOCK = 819_200              # reference-sized run() block with count*I % D == 0 (SURVEY Q4)
FS, FC, FM, DEV = 2_400_000, 250_000, 1_000, 5e3
OUT_SR, BW = 48e3, 48e3
ALG_BYTES_PER_SAMPLE = 8.0 + 4.0 / 50.0   # cf32 in + f32 audio out per input sample (SURVEY §8d, cfg 2)
ALG_FLOP_PER_SAMPLE = 6 + 401 * 4 / 50 + 0.4
FP32_NOMINAL_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12     # 74.4: SMs x FP32 lanes x 2 flop x max clock
FUSED_NCU_SUMMARY = os.path.join(ROOT, "profiles", "r02_fused_rowlane_ncu_full.txt")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(path):
    """dram__bytes_read.sum + dram__bytes_write.sum of the committed ncu --set full summary (tools/ncu_summary.py)."""
    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    try:
        tot, seen = 0.0, 0
        with open(path) as f:
            for line in f:
                t = line.split()
                if len(t) >= 3 and t[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    tot += float(t[1]) * mult[t[2]]
                    seen += 1
        return tot if seen == 2 else None
    except OSError:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING a timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                          str(self.index), "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def mark(self):
        return len(self.rows)

    def summary(self, lo=0, hi=None):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows[lo:hi]:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        return self.summary()


# =================================================================================================
# reference arm / cpu_baseline: the UNMODIFIED reference chain on host cores
# =================================================================================================
_CPU_INPUTS = {}


def cpu_reference_run(sample: int, replicas: int):
    """Time `replicas` independent copies of the reference chain (VFO -> FloatFMDemod, 3 worker threads
    each, as the reference schedules them) over disjoint shards of a `sample`-long synthetic stream.
    Returns (Msamples/s, cores, kind, description)."""
    from oracle import loader
    from qdsp_b200 import synth

    per = (sample // replicas // BLOCK) * BLOCK
    per = max(per, BLOCK)
    key = (per, replicas)
    if _CPU_INPUTS.get("key") != key:   # synthetic input generated once, outside every timed region
        _CPU_INPUTS["key"] = key
        _CPU_INPUTS["xs"] = [synth.cfg2_input(r * per, per) for r in range(replicas)]
    xs = _CPU_INPUTS["xs"]
    if loader.have_ref("fast"):
        R = loader.ref("fast")
        kind, what = "reference", "unmodified reference headers (VFO + FloatFMDemod, 3 threads/chain) + VOLK shim, -O3 -march=x86-64-v3"

        def run(x):
            return R.vfo_fm(float(FC), float(FS), OUT_SR, BW, DEV, x, BLOCK, timing=True)[2]
    else:
        P = loader.port()
        kind, what = "port", "oracle/port.c restatement (single thread per chain)"

        def run(x):
            t0 = time.perf_counter()
            P.vfo_fm(float(FC), float(FS), OUT_SR, BW, DEV, x, BLOCK)
            return time.perf_counter() - t0
    results = [None] * replicas

    def worker(i):
        results[i] = run(xs[i])

    t0 = time.perf_counter()
    th = [threading.Thread(target=worker, args=(i,)) for i in range(replicas)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    wall = time.perf_counter() - t0
    cores = replicas * (3 if kind == "reference" else 1)
    return per * replicas / wall / 1e6, cores, kind, f"{replicas} x {per} samples of the config-2 stream in {BLOCK}-sample blocks; {what}"


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncpu = os.cpu_count() or 1
    replicas = max(1, min(ncpu // 3, 16))
    sample = replicas * 8 * BLOCK       # ~6.5 M samples per chain per step
    vals = []
    for i in range(args.warmup + args.steps):
        v, cores, kind, desc = cpu_reference_run(sample, replicas)
        if i >= args.warmup:
            vals.append(v)
    v = float(np.mean(vals))
    n_per_step = (sample // replicas // BLOCK) * BLOCK * replicas
    line = {
        "impl": "reference", "metric": "Msamples/s cf32 through xlate-resample-demod chain", "value": v, "unit": "Msamples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": n_per_step / v / 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "cfg2: NCO xlator + polyphase resampler 2.4MS/s->48kS/s (401 taps, I=1, D=50) + FM demod; "
                               "bounded CPU sample per step", "samples_per_step": n_per_step, "block": BLOCK},
        "cpu_baseline": {"value": v, "unit": "Msamples/s", "cores": cores, "kind": kind, "sample": desc},
        "e2e": {"value": v, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# =================================================================================================
# our arm
# =================================================================================================
class Ctx:
    """Per-process bench context: ranks, device, streams, the clock sampler, timing helpers."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        from qdsp_b200 import lib

        self.torch, self.dist, self.args = torch, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; qdsp_b200 has no CPU fallback")
        torch.cuda.set_device(self.local)
        self.L = lib.load()
        self.lib = lib
        lib.check(self.L.qdsp_set_device(self.local))
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        self.dev = torch.device("cuda", self.local)
        self.stream = torch.cuda.current_stream()
        self.sp = C.c_void_p(self.stream.cuda_stream)
        self.sampler = ClockSampler(self.local).start() if self.rank == 0 else None
        self.hbm_peak, self.hbm_src = measured_peaks()

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def allmax(self, v: float) -> float:
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def allmin(self, v: float) -> float:
        return -self.allmax(-v)

    def timed(self, step, min_seconds=0.7, warmup=3, max_steps=100000):
        """W warm-up calls, then K calls bracketed by barrier + synchronize and CUDA events on the launching stream; K is
        chosen (identically on every rank) so that the region lasts >= min_seconds: long enough for several 100 ms
        nvidia-smi samples. Returns (ms per call, max over ranks; K; clocks summary of exactly that region)."""
        torch = self.torch
        for _ in range(warmup):
            step()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        step()
        e1.record(self.stream)
        self.barrier()
        est = self.allmax(e0.elapsed_time(e1))
        k = int(min(max_steps, max(3, math.ceil(min_seconds * 1e3 / max(est, 1e-3)))))
        mark = self.sampler.mark() if self.sampler else 0
        self.barrier()
        e0.record(self.stream)
        for _ in range(k):
            step()
        e1.record(self.stream)
        self.barrier()
        ms = self.allmax(e0.elapsed_time(e1)) / k
        clocks = None
        if self.sampler:
            time.sleep(0.12)
            clocks = self.sampler.summary(mark)
        return ms, k, clocks


def dev_window(buf_ptr, lo, hi, dtype=np.complex64):
    """D2H copy of elements [lo, hi) of a device array of `dtype` (used by the oracle checks only)."""
    from qdsp_b200 import lib
    L = lib.load()
    out = np.empty(hi - lo, dtype)
    if out.nbytes:
        lib.check(L.qdsp_copy_d2h(out.ctypes.data, buf_ptr + lo * out.itemsize, out.nbytes, None), "d2h")
        lib.check(L.qdsp_stream_sync(None), "sync")
    return out


# ---- config 2 (headline) ----------------------------------------------------------------------------------
def run_cfg2(cx: Ctx):
    torch, L, lib, args = cx.torch, cx.L, cx.lib, cx.args
    from qdsp_b200 import blocks as B

    n = args.samples
    x = torch.empty(n, dtype=torch.complex64, device=cx.dev)
    # each rank: its own stream = an independent channel (weak scaling, no collective)
    lib.check(L.qdsp_synth_fm_cf32(x.data_ptr(), cx.rank * n, n, FS, FC, FM, DEV, 0.5, 0.005, 2, cx.sp))
    chain = B.VFOFM(float(FC), float(FS), OUT_SR, BW, DEV)
    n_out = chain.out_count(n, BLOCK)
    audio = torch.empty(n_out + 64, dtype=torch.float32, device=cx.dev)
    L.qdsp_vfofm_enable_timing(chain.h, 1)

    def step():
        m = L.qdsp_vfofm_process(chain.h, x.data_ptr(), audio.data_ptr(), None, n, None, 0, BLOCK, None, cx.sp)
        if m != n_out:
            raise SystemExit(f"process returned {m}, expected {n_out}: {lib.last_error()}")

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step()
    cx.barrier()
    mark = cx.sampler.mark() if cx.sampler else 0
    launches0 = L.qdsp_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # one CUDA event pair per launch of the fused kernel, recorded on the launching stream inside the timed region
    lib.check(L.qdsp_vfofm_enable_timing_ring(chain.h, args.steps), "enable_timing_ring")
    cx.barrier()
    e0.record(cx.stream)
    for _ in range(args.steps):
        step()
    e1.record(cx.stream)
    cx.barrier()
    ms = e0.elapsed_time(e1)
    launches = L.qdsp_launch_count() - launches0
    nrec = C.c_int(0)
    k_ms = float(L.qdsp_vfofm_kernel_ms_mean(chain.h, C.byref(nrec)))
    assert nrec.value == args.steps, (nrec.value, args.steps)
    ms_max = cx.allmax(ms)
    value = cx.world * n * args.steps / (ms_max * 1e-3) / 1e6
    # the audio of the last timed step, read back before the passes below reuse `audio` and the chain's stream position
    last_audio = audio[:n_out].cpu().numpy() if args.dump_outputs else None

    # ---- parity of THIS run's output (device path) and of the host-buffer path, against the CPU oracle ----
    parity = None
    audio_host = None
    if not args.no_parity:
        audio_host = audio[:n_out].cpu().numpy()

    # ---- end to end: pinned host in -> C-ABI host entry point -> pinned host out ---------------------
    e2e = None
    host_equal = None
    if not args.no_e2e:
        xh = torch.empty(n, dtype=torch.complex64, pin_memory=True)
        xh.copy_(x)
        yh = torch.empty(n_out + 64, dtype=torch.float32, pin_memory=True)
        torch.cuda.synchronize()
        chain2 = B.VFOFM(float(FC), float(FS), OUT_SR, BW, DEV)

        def e2e_step():
            m = L.qdsp_vfofm_process_host(chain2.h, xh.data_ptr(), yh.data_ptr(), n, BLOCK, cx.sp)
            if m != n_out:
                raise SystemExit(f"process_host returned {m}, expected {n_out}: {lib.last_error()}")

        e2e_step()          # first call from a fresh handle: same stream position as the device path's first step
        yh_first = yh[:n_out].numpy().copy() if audio_host is not None else None
        if audio_host is not None:
            first_dev = B.VFOFM(float(FC), float(FS), OUT_SR, BW, DEV)
            tmp = torch.empty(n_out + 64, dtype=torch.float32, device=cx.dev)
            L.qdsp_vfofm_process(first_dev.h, x.data_ptr(), tmp.data_ptr(), None, n, None, 0, BLOCK, None, cx.sp)
            torch.cuda.synchronize()
            host_equal = bool(np.array_equal(yh_first.view(np.uint32), tmp[:n_out].cpu().numpy().view(np.uint32)))
            audio_first = tmp[:n_out].cpu().numpy()
            del tmp
        cx.barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            e2e_step()          # synchronises the stream internally: result is in host memory on return
        torch.cuda.synchronize()
        dt = cx.allmax(time.perf_counter() - t0)
        e2e = {"value": cx.world * n * args.e2e_steps / dt / 1e6, "unit": "Msamples/s",
               "h2d_bytes_per_step": n * 8, "d2h_bytes_per_step": n_out * 4, "steps": args.e2e_steps,
               "h2d_gbs_per_gpu": n * 8 * args.e2e_steps / dt / 1e9,
               "checksum": float(yh[:n_out].double().abs().sum())}
        # the PCIe ceiling of this box for the same bytes: a plain pinned H2D copy of the input, timed alone
        xd2 = torch.empty(n, dtype=torch.complex64, device=cx.dev)
        xd2.copy_(xh, non_blocking=True)
        cx.barrier()
        t0 = time.perf_counter()
        for _ in range(2):
            xd2.copy_(xh, non_blocking=True)
        torch.cuda.synchronize()
        dt2 = cx.allmax(time.perf_counter() - t0)
        e2e["h2d_copy_alone_gbs_per_gpu"] = n * 8 * 2 / dt2 / 1e9
        e2e["frac_of_h2d_copy_alone"] = e2e["h2d_gbs_per_gpu"] / e2e["h2d_copy_alone_gbs_per_gpu"]
        del xd2

    time.sleep(0.12)
    clocks = cx.sampler.summary(mark) if cx.sampler else None     # the K timed steps + the end-to-end passes
    # ---- sustained variant: the same step repeated for >= 2 s (the headline region above is a burst of K steps) ----
    L.qdsp_vfofm_enable_timing(chain.h, 0)
    sus_ms, sus_k, sus_clocks = cx.timed(step, min_seconds=2.0, warmup=0)
    sustained = {"value": cx.world * n / (sus_ms * 1e-3) / 1e6, "unit": "Msamples/s", "steps": sus_k, "ms_per_step": sus_ms,
                 "clocks": sus_clocks}

    if audio_host is not None and cx.rank == 0:
        from oracle import windows
        seams = [c * 10 * BLOCK for c in range(1, n // (10 * BLOCK) + 1)]      # process_host's 8 192 000-sample chunks
        centres = windows.pick_windows(n, BLOCK, 16, 65536, seams)

        def get_in(lo, hi):
            return x[lo:hi].cpu().numpy()

        # the timed steps continue ONE stream (handle state carried): step s starts at absolute sample s*n, so the last
        # step's output is checked with the NCO phase of that position; the first-call output of a fresh handle too
        t0 = time.perf_counter()
        parity = {"oracle": "oracle/port.c, reference chain with the drift-free (float64) rotator, recomputed per window",
                  "tolerance_abs": 1e-4, "windows": len(centres), "window_samples": 65536,
                  "seams_checked": len(seams)}
        if not args.no_e2e:
            wd, cnt = windows.check_vfofm_windows(get_in, audio_first, n, BLOCK, centres, 65536, float(FC), float(FS), OUT_SR, BW,
                                                  DEV, 50, 401)
            wh, _ = windows.check_vfofm_windows(get_in, yh_first, n, BLOCK, centres, 65536, float(FC), float(FS), OUT_SR,
                                                BW, DEV, 50, 401)
            parity.update({"max_abs_err_device_path": wd, "max_abs_err_host_path": wh, "outputs_compared": cnt,
                           "host_path_bit_equal_to_device_path": host_equal,
                           "ok": bool(wd <= 1e-4 and wh <= 1e-4 and host_equal)})
        else:
            parity.update({"note": "run without --no-e2e for the device/host path comparison"})
        parity["seconds"] = time.perf_counter() - t0
    if not args.no_e2e:
        del xh, yh

    achieved = ALG_BYTES_PER_SAMPLE * n / (k_ms * 1e-3) / 1e9
    traffic = ncu_traffic(FUSED_NCU_SUMMARY) if n == N_SAMPLES else None
    roof = {"bound": "hbm", "achieved": achieved, "peak": cx.hbm_peak, "unit": "GB/s", "frac": achieved / cx.hbm_peak,
            "traffic": traffic, "traffic_source": os.path.relpath(FUSED_NCU_SUMMARY, ROOT) if traffic else None,
            "peak_source": cx.hbm_src,
            "note": "peak is the driver-measured COPY bandwidth (read+write); this kernel is 99 % reads, which HBM3e serves faster",
            "kernel": "qdsp::decim_rowlane_kernel<9,50,402,2,ROT,DEMOD> (fused xlate+resample+demod, history advance folded in)",
            "kernel_ms": k_ms, "alg_bytes_per_launch": ALG_BYTES_PER_SAMPLE * n,
            "fp32_tflops": ALG_FLOP_PER_SAMPLE * n / (k_ms * 1e-3) / 1e12}
    del x, audio
    torch.cuda.empty_cache()
    return {"value": value, "ms_per_step": ms_max / args.steps, "warm": warm, "launches": int(launches), "e2e": e2e,
            "clocks": clocks, "roofline": roof, "parity": parity, "sustained": sustained, "n": n, "last_audio": last_audio}


DUMP_BYTES_MAX = 60_000_000     # what --dump-outputs writes stays below 64 MB, .npy headers included


def dump_output(out_dir, name, a):
    """Write a as out_dir/<name>.npy. Above DUMP_BYTES_MAX a fixed seeded sample of its elements (in stream order) is
    written instead, with their positions as <name>_index.npy, so that two runs with the same arguments stay comparable."""
    os.makedirs(out_dir, exist_ok=True)
    if a.nbytes > DUMP_BYTES_MAX:
        idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_BYTES_MAX // (a.itemsize + 8), replace=False))
        a = a[idx]
        np.save(os.path.join(out_dir, name + "_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, name + ".npy"), a)


# ---- config 1: 127-tap FIR (1a) and FIR + decimate-by-4 (1b), 2^24 samples ---------------------------------
def run_cfg1(cx: Ctx, fp32_peak):
    from oracle import loader, windows
    from qdsp_b200 import blocks as B

    L, lib = cx.L, cx.lib
    n, nbuf = 1 << 24, 4          # 4 x 128 MiB inputs used round robin: every pass reads a buffer that is not in L2 (126 MB)
    xs = [B.DevBuf(n * 8) for _ in range(nbuf)]
    for i, b in enumerate(xs):
        lib.check(L.qdsp_synth_uniform_cf32(b.ptr, 1, i * n, n, cx.sp))
    ys = [B.DevBuf(n * 8) for _ in range(nbuf)]
    win = B.BlackmanWindow(300e3, 4 * 2.4e6 / 127, 2.4e6)
    P = loader.port()
    taps = P.blackman_taps(300e3, 4 * 2.4e6 / 127, 2.4e6)
    out = {}
    # 1a
    f = B.FIR(win)
    it = [0]

    def step_a():
        i = it[0] % nbuf
        it[0] += 1
        f.process_device(xs[i].ptr, ys[i].ptr, n, stream=cx.sp)

    ms, k, clocks = cx.timed(step_a)
    f0 = B.FIR(win)
    f0.process_device(xs[0].ptr, ys[0].ptr, n, stream=cx.sp)
    cx.torch.cuda.synchronize()
    centres = windows.pick_windows(n, 1 << 19, 6, 16384, [])
    rel, mx, cnt = windows.check_fir_windows(lambda lo, hi: dev_window(xs[0].ptr, lo, hi), None,
                                             lambda lo, hi: dev_window(ys[0].ptr, lo, hi), n, taps, centres, 16384)
    tf = 508.0 * n / ms / 1e9
    out["cfg1a"] = {"workload": "FIR<complex_t>, 127 taps, 2^24 cf32 (4 rotating inputs > L2)", "value": n / ms / 1e3, "unit": "Msamples/s",
                    "ms_per_step": ms, "steps": k, "clocks": clocks,
                    "roofline": {"bound": "fp32", "achieved": tf, "unit": "TFLOP/s", "peak_nominal": FP32_NOMINAL_TFLOPS,
                                 "frac_nominal": tf / FP32_NOMINAL_TFLOPS, "peak_probe_ffma2": fp32_peak, "frac_probe": tf / fp32_peak,
                                 "hbm_gbs": 16.0 * n / ms / 1e6},
                    "parity": {"oracle": "oracle/port.c fir_cf32", "windows": len(centres), "outputs_compared": cnt, "rel_l2_worst": rel,
                               "tolerance_rel_l2": 1e-5, "ok": bool(rel <= 1e-5)}}
    # 1b
    r = B.PolyphaseResampler(win, 2.4e6, 0.6e6)

    def step_b():
        i = it[0] % nbuf
        it[0] += 1
        r.process_device(xs[i].ptr, ys[i].ptr, n, 524288, stream=cx.sp)

    ms, k, clocks = cx.timed(step_b)
    r0 = B.PolyphaseResampler(win, 2.4e6, 0.6e6)
    m = r0.process_device(xs[0].ptr, ys[0].ptr, n, 524288, stream=cx.sp)
    cx.torch.cuda.synchronize()
    rel, cnt = 0.0, 0
    for c in windows.pick_windows(n, 524288, 6, 32768, [524288, 524288 * 7]):
        lo = max(0, (c - 16384) // 4 * 4 - 128 * 4)
        hi = min(n, lo + 128 * 4 + 32768)
        cuts = [lo] + list(range((lo // 524288 + 1) * 524288, hi, 524288)) + [hi]
        yo, _ = P.resamp_cf32(taps, 1, 4, dev_window(xs[0].ptr, lo, hi), [b - a for a, b in zip(cuts[:-1], cuts[1:])])
        first = 0 if lo == 0 else 40
        g = dev_window(ys[0].ptr, lo // 4 + first, lo // 4 + len(yo))
        rel = max(rel, float(np.linalg.norm(g - yo[first:]) / np.linalg.norm(yo[first:])))
        cnt += len(g)
    gbs = 10.0 * n / ms / 1e6
    tf = 127.0 * n / ms / 1e9
    out["cfg1b"] = {"workload": "PolyphaseResampler<complex_t> fs -> fs/4 (I=1, D=4, 127 taps), 2^24 cf32, run() blocks of 524288",
                    "value": n / ms / 1e3, "unit": "Msamples/s", "ms_per_step": ms, "steps": k, "clocks": clocks,
                    "roofline": {"bound": "hbm~fp32 (ridge)", "achieved": gbs, "unit": "GB/s", "peak": cx.hbm_peak, "frac": gbs / cx.hbm_peak,
                                 "fp32_tflops": tf, "frac_fp32_nominal": tf / FP32_NOMINAL_TFLOPS},
                    "parity": {"oracle": "oracle/port.c resamp_cf32", "outputs_compared": cnt, "rel_l2_worst": rel, "tolerance_rel_l2": 1e-5,
                               "out_count_exact": bool(m == n // 4), "ok": bool(rel <= 1e-5 and m == n // 4)}}
    for b in xs + ys:
        b.free()
    return out


# ---- config 3: 4095-tap FIR, one 2^30-sample stream time-sharded over the ranks ------------------------------
def run_cfg3(cx: Ctx, fp32_peak):
    from oracle import loader, windows
    from qdsp_b200 import blocks as B, shard

    torch, dist, L, lib = cx.torch, cx.dist, cx.L, cx.lib
    total = cx.args.n3
    win = B.BlackmanWindow(100e3, 4 * 2.4e6 / 4095, 2.4e6)
    P = loader.port()
    taps = P.blackman_taps(100e3, 4 * 2.4e6 / 4095, 2.4e6)
    T = len(taps)
    shards = shard.time_shards(total, cx.world, 1 << 20, T - 1)
    me = shards[cx.rank]
    x = B.DevBuf(me.count * 8)
    y = B.DevBuf(me.count * 8)
    lib.check(L.qdsp_synth_uniform_cf32(x.ptr, 3, me.start, me.count, cx.sp))
    # ---- halo: map the previous rank's shard into this process (CUDA IPC) and let the FIR kernel read the last T-1
    # samples straight out of it over NVLink; fallback (IPC unavailable): one NCCL send/recv of the tail per step
    halo_ptr, halo_path, mapped, halo_buf = None, "none (single shard: zero history)", None, None
    if cx.world > 1:
        hnd = np.zeros(64, np.uint8)
        lib.check(L.qdsp_ipc_export(x.ptr, hnd.ctypes.data), "ipc_export")
        allh = [torch.empty(64, dtype=torch.uint8, device=cx.dev) for _ in range(cx.world)]
        dist.all_gather(allh, torch.from_numpy(hnd).to(cx.dev))
        ok = 1
        if cx.rank > 0:
            prev = shards[cx.rank - 1]
            ph = allh[cx.rank - 1].cpu().numpy().copy()
            mapped = L.qdsp_ipc_open(ph.ctypes.data)
            if mapped and prev.count >= T - 1:
                halo_ptr = mapped + (prev.count - (T - 1)) * 8
            else:
                ok = 0
        ok = int(cx.allmin(float(ok)))
        if ok:
            halo_path = "p2p-direct-read: FIR kernel loads the neighbour's tail through a CUDA-IPC peer mapping (NVLink), no copy, no collective"
        else:
            halo_path = "nccl-sendrecv fallback (CUDA IPC unavailable): tail sent with one point-to-point message per step"
            halo_ptr = None
            halo_buf = torch.zeros(2 * (T - 1), dtype=torch.float32, device=cx.dev)

            class _Raw:   # zero-copy torch view of the DevBuf tail
                def __init__(self, ptr, nfloat):
                    self.__cuda_array_interface__ = {"shape": (nfloat,), "typestr": "<f4", "data": (ptr, False), "version": 2}
            tail_view = torch.as_tensor(_Raw(x.ptr + (me.count - (T - 1)) * 8, 2 * (T - 1)), device=cx.dev)
    fir = B.FIR(win)

    def step():
        hp = halo_ptr
        if halo_buf is not None:
            reqs = []
            if cx.rank + 1 < cx.world:
                reqs.append(dist.isend(tail_view, dst=cx.rank + 1))
            if cx.rank > 0:
                reqs.append(dist.irecv(halo_buf, src=cx.rank - 1))
            for q in reqs:
                q.wait()
            hp = halo_buf.data_ptr() if cx.rank > 0 else None
        m = fir.process_halo_device(hp, x.ptr, y.ptr, me.count, stream=cx.sp)
        assert m == me.count

    cx.barrier()       # every shard's input is generated before any neighbour reads it
    ms, k, clocks = cx.timed(step, min_seconds=1.0, warmup=1)
    # ---- oracle check: every shard boundary (the window straddles it) + random windows + both ends -------------------
    centres = [c for c in windows.pick_windows(total, 1 << 20, 6, 8192, [s.start for s in shards[1:]])
               if me.start <= c - 4096 and c + 4096 <= me.start + me.count] if me.count >= 16384 else []
    if cx.rank > 0 and me.count >= 8192:
        centres.append(me.start + 4096)         # outputs [start, start + 8192): their windows reach into the previous shard
    in_scratch = B.DevBuf((8192 + T) * 8)

    def get_in(lo, hi):    # any window of the stream, regenerated (counter-based generator): crosses shard boundaries freely
        lib.check(L.qdsp_synth_uniform_cf32(in_scratch.ptr, 3, lo, hi - lo, None))
        return dev_window(in_scratch.ptr, 0, hi - lo)

    rel, mx, cnt = windows.check_fir_windows(get_in, None, lambda lo, hi: dev_window(y.ptr, lo - me.start, hi - me.start), total, taps,
                                             sorted(set(centres)), 8192) if centres else (0.0, 0.0, 0)
    rel = cx.allmax(rel)
    cnt_all = int(cx.allmax(float(cnt)))
    tf = 4.0 * T * total / ms / 1e9
    res = {"workload": f"FIR<complex_t>, 4095 taps, one stream of {total} cf32 time-sharded over {cx.world} GPU(s) in run() blocks of 2^20",
           "value": total / ms / 1e3, "unit": "Msamples/s", "scaling": "strong", "ms_per_step": ms, "steps": k, "clocks": clocks,
           "halo": {"samples": T - 1, "bytes_per_boundary": (T - 1) * 8, "path": halo_path},
           "roofline": {"bound": "fp32", "achieved": tf, "unit": "TFLOP/s (all GPUs)", "per_gpu": tf / cx.world,
                        "peak_nominal_per_gpu": FP32_NOMINAL_TFLOPS, "frac_nominal": tf / cx.world / FP32_NOMINAL_TFLOPS,
                        "peak_probe_ffma2_per_gpu": fp32_peak, "frac_probe": tf / cx.world / fp32_peak},
           "parity": {"oracle": "oracle/port.c fir_cf32 on windows: every shard boundary (outputs start .. start+8192), both ends, random",
                      "windows_this_rank_max": len(centres), "outputs_compared_max_rank": cnt_all, "rel_l2_worst": rel,
                      "tolerance_rel_l2": 1e-5, "ok": bool(rel <= 1e-5)}}
    cx.barrier()
    if mapped:
        L.qdsp_ipc_close(mapped)
    cx.barrier()
    x.free()
    y.free()
    in_scratch.free()
    return res


# ---- config 4: 256-channel channelizer, channels partitioned over the ranks -----------------------------------
def run_cfg4(cx: Ctx, fp32_peak):
    """Two records. `cfg4`: the product's default path for this geometry -- the FFT polyphase channelizer (k_chanfft.cu), all
    256 channels on every GPU, the STREAM time-sharded at N > 1 (weak: 2^26 samples per GPU, each shard fed 16 output rows of
    lead-in it drops; no collective). `cfg4_direct`: the direct form (every channel its own VFO, the reference's algorithm
    unchanged), channels partitioned over the GPUs (strong) -- round 1's record, kept for continuity and the FP32 roofline."""
    out = {"cfg4_direct": _cfg4_direct(cx, fp32_peak)}
    if not (cx.args.cfg4_world and cx.world == 1):
        out["cfg4"] = _cfg4_fft(cx)
    return out


def _cfg4_fft(cx: Ctx):
    from oracle import windows
    from qdsp_b200 import blocks as B, shard, synth

    L, lib = cx.L, cx.lib
    n, nch = cx.args.n4, 256
    fs, spacing, D, blk = 61_440_000, 240_000, 1280, 819200
    # shard r = [s_r, s_{r+1}) of the N * 2^26-sample stream, s_r on the decimation grid (2^26 is not a multiple of 1280);
    # lead-in: history (10 240 samples) + one row for the demodulator's previous angle + margin = 16 rows
    total = cx.world * n
    me = shard.lead_in_shards(n, cx.world, D, 10241, extra_rows=6)[cx.rank]
    lo, hi, lead = me.start, me.start + me.count, me.lead
    g0 = lo - lead                               # stream position of this rank's first local sample
    n = me.count
    offs = synth.cfg4_offsets(nch, spacing)
    x = B.DevBuf((n + lead) * 8)
    lib.check(L.qdsp_synth_comb_cf32(x.ptr, g0, n + lead, fs, nch, spacing, 5e3, 1.0 / 64.0, 0.001, 4, cx.sp))
    ch = B.Channelizer(offs, float(fs), 48e3, 48e3, 5e3)
    assert (ch.tapCount, ch._interp, ch._decim) == (10241, 1, D)
    stride = (n + lead) // D + 64
    y = B.DevBuf(nch * stride * 4)
    ch.seek(g0)

    def step():
        ch.process_device(x.ptr, y.ptr, n + lead, stride, blk, stream=cx.sp)

    l0 = L.qdsp_launch_count()
    step()
    launches = L.qdsp_launch_count() - l0
    ms, k, clocks = cx.timed(step, min_seconds=0.7, warmup=3)
    # ---- oracle check on a fresh handle at this shard's stream position
    ch0 = B.Channelizer(offs, float(fs), 48e3, 48e3, 5e3)
    ch0.seek(g0)
    m = ch0.process_device(x.ptr, y.ptr, n + lead, stride, blk, stream=cx.sp)
    cx.torch.cuda.synchronize()
    worst, cnt = 0.0, 0
    rng = np.random.default_rng(300 + cx.rank)
    picks = sorted(set([0, nch - 1] + [int(c) for c in rng.integers(0, nch, size=4)]))
    local = windows.pick_windows(n, blk, 2, 65536, [blk, blk * (n // blk)])
    centres = [lo + c for c in local]            # incl. the shard's first and last window: the seams between ranks
    for c in picks:
        a = np.zeros(total // D, dtype=np.float32)          # the whole stream's output axis; this rank fills its shard
        got = dev_window(y.ptr, c * stride, c * stride + m, np.float32)
        a[lo // D:lo // D + n // D] = got[lead // D:lead // D + n // D]
        w, k2 = windows.check_vfofm_windows(lambda l, h: dev_window(x.ptr, l - g0, h - g0), a, hi, blk, centres, 65536,
                                            float(offs[c]), float(fs), 48e3, 48e3, 5e3, D, 10241)
        worst = max(worst, w)
        cnt += k2
    worst = cx.allmax(worst)
    alg = (n + lead) * 8 + nch * ((n + lead) // D) * 4
    gbs = alg / ms / 1e6
    res = {"workload": f"256-channel channelizer (VFO + FloatFMDemod per channel: 10241 taps, I=1, D=1280), FFT polyphase form: all 256 "
                       f"channels on every GPU, a 61.44 MS/s stream of {total} cf32 time-sharded over {cx.world} GPU(s) "
                       f"({n} samples + {lead} lead-in on this rank), no collective",
           "value": total / ms / 1e3, "unit": "Msamples/s (wideband input, all 256 channels produced)", "scaling": "weak",
           "channel_msamples_s": nch * total / ms / 1e3, "ms_per_step": ms, "steps": k, "launches_per_step": int(launches), "clocks": clocks,
           "roofline": {"bound": "hbm", "achieved": gbs, "unit": "GB/s", "peak": cx.hbm_peak, "frac": gbs / cx.hbm_peak,
                        "alg_bytes_per_launch": alg, "note": "algorithmic bytes: the wideband input once + the 256 audio rows; the U/V "
                        "planes between the two kernels (2 x 16 B per output row and channel) are extra traffic",
                        "direct_form_equivalent_tflops_per_gpu": 38.0 * nch * (n + lead) / ms / 1e9},
           "parity": {"oracle": "oracle/port.c reference chain (float64 rotator) per channel, windows incl. run() boundaries and both ends "
                                "of this rank's shard (the seams between ranks)",
                      "channels_checked_per_rank": len(picks), "outputs_compared_this_rank": cnt, "max_abs_err": worst, "tolerance_abs": 1e-4,
                      "ok": bool(worst <= 1e-4)}}
    x.free()
    y.free()
    return res


def _cfg4_direct(cx: Ctx, fp32_peak):
    from oracle import loader, windows
    from qdsp_b200 import blocks as B, shard, synth

    L, lib = cx.L, cx.lib
    n, nch_total = cx.args.n4, 256
    fs, spacing = 61_440_000, 240_000
    # --cfg4-world W (development aid): take rank 0's share of a W-way partition on this one GPU (32 channels for W = 8)
    eworld = cx.args.cfg4_world if (cx.args.cfg4_world and cx.world == 1) else cx.world
    sl = shard.channel_slice(nch_total, eworld, cx.rank)
    offs_all = synth.cfg4_offsets(nch_total, spacing)
    offs = offs_all[sl]
    nch = len(offs)
    x = B.DevBuf(n * 8)     # every rank holds the same wideband stream (generated in place: no broadcast on the timed path)
    lib.check(L.qdsp_synth_comb_cf32(x.ptr, 0, n, fs, nch_total, spacing, 5e3, 1.0 / 64.0, 0.001, 4, cx.sp))
    ch = B.Channelizer(offs, float(fs), 48e3, 48e3, 5e3)
    ch.set_variant(2)
    assert (ch.tapCount, ch._interp, ch._decim) == (10241, 1, 1280)
    blk = 819200
    stride = n // 1280 + 64
    y = B.DevBuf(nch * stride * 4)

    def step():
        ch.process_device(x.ptr, y.ptr, n, stride, blk, stream=cx.sp)

    ms, k, clocks = cx.timed(step, min_seconds=1.0, warmup=1)
    # ---- oracle check on a fresh handle (first call of a stream), a few (channel, window) pairs incl. this rank's edge channels
    ch0 = B.Channelizer(offs, float(fs), 48e3, 48e3, 5e3)
    ch0.set_variant(2)
    m = ch0.process_device(x.ptr, y.ptr, n, stride, blk, stream=cx.sp)
    cx.torch.cuda.synchronize()
    worst, cnt = 0.0, 0
    rng = np.random.default_rng(100 + cx.rank)
    picks = sorted(set([0, nch - 1] + [int(c) for c in rng.integers(0, nch, size=4)]))
    centres = windows.pick_windows(n, blk, 2, 65536, [blk, blk * (n // blk)])
    for c in picks:
        a = dev_window(y.ptr, c * stride, c * stride + m, np.float32)
        w, k2 = windows.check_vfofm_windows(lambda lo, hi: dev_window(x.ptr, lo, hi), a, n, blk, centres, 65536, float(offs[c]), float(fs),
                                            48e3, 48e3, 5e3, 1280, 10241)
        worst = max(worst, w)
        cnt += k2
    worst = cx.allmax(worst)
    if eworld != cx.world:      # emulated share: report this GPU's channels only
        nch_total = nch
    tf = 38.0 * nch_total * n / ms / 1e9
    res = {"workload": f"{nch_total}-channel channelizer (VFO + FloatFMDemod per channel: 10241 taps, I=1, D=1280) off one 61.44 MS/s stream of "
                       f"{n} cf32, DIRECT form; {nch} channels on each of {cx.world} GPU(s), no collective",
           "value": n / ms / 1e3, "unit": "Msamples/s (wideband input, all 256 channels produced)", "scaling": "strong",
           "channel_msamples_s": nch_total * n / ms / 1e3, "ms_per_step": ms, "steps": k, "clocks": clocks,
           "roofline": {"bound": "fp32", "achieved": tf, "unit": "TFLOP/s (all GPUs)", "per_gpu": tf / cx.world,
                        "peak_nominal_per_gpu": FP32_NOMINAL_TFLOPS, "frac_nominal": tf / cx.world / FP32_NOMINAL_TFLOPS,
                        "peak_probe_ffma2_per_gpu": fp32_peak, "frac_probe": tf / cx.world / fp32_peak,
                        "fp32_bound_wideband_gsps_per_gpu_at_32ch": FP32_NOMINAL_TFLOPS * 1e3 / (38.0 * 32)},
           "parity": {"oracle": "oracle/port.c reference chain (float64 rotator) per channel, windows incl. run() boundaries and both ends",
                      "channels_checked_per_rank": len(picks), "outputs_compared_this_rank": cnt, "max_abs_err": worst, "tolerance_abs": 1e-4,
                      "ok": bool(worst <= 1e-4)}}
    x.free()
    y.free()
    return res


# ---- config 5: recurrent blocks on 2^28 samples ----------------------------------------------------------------
def run_cfg5(cx: Ctx):
    from oracle import loader
    from qdsp_b200 import blocks as B

    L, lib = cx.L, cx.lib
    n = cx.args.n5
    P = loader.port()
    x = B.DevBuf(n * 8)
    y = B.DevBuf(n * 8)
    pre = 1 << 21          # recurrences are causal: the first 2^21 outputs depend on the first 2^21 inputs only
    out = {}

    def record(name, ms, k, clocks, bytes_per, err, tol, kind, extra=None, count=None):
        count = n if count is None else count
        gbs = bytes_per * count / ms / 1e6
        out[name] = {"value": count / ms / 1e3, "unit": "Msamples/s", "ms_per_step": ms, "steps": k, "clocks": clocks,
                     "roofline": {"bound": "hbm", "achieved": gbs, "unit": "GB/s", "peak": cx.hbm_peak, "frac": gbs / cx.hbm_peak,
                                  "alg_bytes_per_sample": bytes_per},
                     "parity": {"oracle": f"oracle/port.c on the first {pre} samples", kind: err, "tolerance": tol, "ok": bool(err <= tol)}}
        if extra:
            out[name].update(extra)

    # (i) BFMDeemp on stereo U(5, n)
    lib.check(L.qdsp_synth_uniform_cf32(x.ptr, 5, 0, n, cx.sp))
    blk = B.BFMDeemp(48e3, 50e-6)
    ms, k, clocks = cx.timed(lambda: blk.process_device(x.ptr, y.ptr, n, stream=cx.sp))
    b0 = B.BFMDeemp(48e3, 50e-6)
    b0.process_device(x.ptr, y.ptr, n, stream=cx.sp)
    xo = dev_window(x.ptr, 0, pre)
    yo = P.deemp(48e3, 50e-6, xo.view(np.float32).reshape(-1, 2)).reshape(-1).view(np.complex64)
    g = dev_window(y.ptr, 0, pre)
    record("cfg5_deemp", ms, k, clocks, 16, float(np.abs(g - yo).max()), 0.0, "max_abs_err",
           {"workload": f"BFMDeemp(48 kHz, 50 us), {n} stereo samples", "bit_exact": bool(np.array_equal(g.view(np.uint32), yo.view(np.uint32)))})
    # (iv) AGC(20, fs) on the same data viewed as floats, run() blocks of 1e6
    agc = B.AGC(20.0, 48e3)
    ms, k, clocks = cx.timed(lambda: agc.process_device(x.ptr, y.ptr, 2 * n, 1000000, stream=cx.sp))
    a0 = B.AGC(20.0, 48e3)
    a0.process_device(x.ptr, y.ptr, 2 * n, 1000000, stream=cx.sp)
    xf = dev_window(x.ptr, 0, 2 * pre - (2 * pre) % 1000000, np.float32)
    yo = P.agc(20.0, 48e3, xf, 1000000)
    g = dev_window(y.ptr, 0, len(xf), np.float32)
    out_agc_err = float(np.linalg.norm(g - yo) / np.linalg.norm(yo))
    record("cfg5_agc", ms, k, clocks, 8, out_agc_err, 1e-5, "rel_l2",
           {"workload": f"AGC(20, 48 kHz), {2 * n} float samples, run() blocks of 1e6"}, count=2 * n)
    # (ii) ComplexAGC on amplitude-modulated QPSK
    lib.check(L.qdsp_synth_qpsk_cf32(x.ptr, 0, n, 21, 4, 0.01, 0.07, 0.5, 50000, cx.sp))
    cagc = B.ComplexAGC(1.0, 65535.0, 1e-3)
    ms, k, clocks = cx.timed(lambda: cagc.process_device(x.ptr, y.ptr, n, stream=cx.sp))
    c0 = B.ComplexAGC(1.0, 65535.0, 1e-3)
    c0.process_device(x.ptr, y.ptr, n, stream=cx.sp)
    xo = dev_window(x.ptr, 0, pre)
    yo = P.complex_agc(1.0, 65535.0, 1e-3, xo)
    g = dev_window(y.ptr, 0, pre)
    record("cfg5_complex_agc", ms, k, clocks, 16, float(np.linalg.norm(g - yo) / np.linalg.norm(yo)), 1e-4, "rel_l2",
           {"workload": f"ComplexAGC(1.0, 65535, 1e-3), {n} samples of amplitude-modulated QPSK"})
    # FeedForwardAGC on the same stream
    ff = B.FeedForwardAGC()
    ms, k, clocks = cx.timed(lambda: ff.process_device(x.ptr, y.ptr, n, stream=cx.sp))
    f0 = B.FeedForwardAGC()
    mo = f0.process_device(x.ptr, y.ptr, n, stream=cx.sp)
    yo = P.ff_agc(xo)
    g = dev_window(y.ptr, 0, len(yo))
    record("cfg5_ff_agc", ms, k, clocks, 16, float(np.abs(g - yo).max()), 0.0, "max_abs_err",
           {"workload": f"FeedForwardAGC<complex_t>, {n} samples", "bit_exact": bool(np.array_equal(g.view(np.uint32), yo.view(np.uint32))),
            "out_count": int(mo)})
    # (iii) CostasLoop<4>(0.004) on QPSK, 0.01 rad/sample offset, sigma 0.07
    lib.check(L.qdsp_synth_qpsk_cf32(x.ptr, 0, n, 23, 4, 0.01, 0.07, 0.0, 1, cx.sp))
    pl = B.CostasLoop(4, 0.004)
    ms, k, clocks = cx.timed(lambda: pl.process_device(x.ptr, y.ptr, n, stream=cx.sp))
    p0 = B.CostasLoop(4, 0.004)
    p0.process_device(x.ptr, y.ptr, n, stream=cx.sp)
    resid = p0.last_residual()
    xo = dev_window(x.ptr, 0, pre)
    yo, _ = P.costas(4, 0.004, xo)
    g = dev_window(y.ptr, 0, pre)
    record("cfg5_costas4", ms, k, clocks, 16, float(np.abs(g - yo).max()), 1e-4, "max_abs_err",
           {"workload": f"CostasLoop<4>(0.004), {n} QPSK samples (0.01 rad/sample offset, sigma 0.07), chunked scan",
            "boundary_residual": resid})
    x.free()
    y.free()
    return out


def ours(args):
    cx = Ctx(args)
    torch, L = cx.torch, cx.L
    want = set(c for c in args.configs.split(",") if c)
    main = run_cfg2(cx)
    configs = {}
    fp32_peak = None
    if want & {"1", "3", "4"}:
        fp32_peak = float(L.qdsp_measure_fp32_peak(1, 20000))
    if "1" in want and cx.world == 1:
        configs.update(run_cfg1(cx, fp32_peak))
    if "3" in want:
        configs["cfg3"] = run_cfg3(cx, fp32_peak)
    if "4" in want:
        configs.update(run_cfg4(cx, fp32_peak))
    if "5" in want and cx.world == 1:
        configs.update(run_cfg5(cx))
    launches_total = int(L.qdsp_launch_count())
    clocks_all = cx.sampler.stop() if cx.sampler else None
    if cx.rank != 0:
        if cx.world > 1:
            cx.dist.destroy_process_group()
        return
    cpu = None
    if not args.no_cpu:
        ncpu = os.cpu_count() or 1
        v, cores, kind, desc = cpu_reference_run(8 * BLOCK * 1, 1)
        # run again with all cores the reference's threading model can use
        replicas = max(1, min(ncpu // 3, 16))
        v_all, cores_all, _, desc_all = cpu_reference_run(replicas * 8 * BLOCK, replicas)
        cpu = {"value": v_all, "unit": "Msamples/s", "cores": cores_all, "kind": kind, "sample": desc_all,
               "single_chain": {"value": v, "cores": cores, "sample": desc}, "host_cpus": ncpu}
    line = {
        "metric": "Msamples/s cf32 through xlate-resample-demod chain", "value": main["value"], "unit": "Msamples/s",
        "n_gpus": cx.world, "steps": args.steps, "warmup": main["warm"], "ms_per_step": main["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "cfg2: NCO xlator + polyphase resampler 2.4MS/s->48kS/s (401 taps, I=1, D=50) + FM demod, fused",
                   "samples_per_gpu": main["n"], "block": BLOCK, "parallelism": f"independent streams x{cx.world} (no collective)",
                   "l2": "input (2 GiB/GPU) is larger than L2: no flush needed"},
        "e2e": main["e2e"], "gpu_launches": main["launches"], "clocks": main["clocks"], "roofline": main["roofline"],
        "sustained": main["sustained"], "parity": main["parity"], "cpu_baseline": cpu, "configs": configs,
        "fp32_peak_probe_ffma2_tflops": fp32_peak, "fp32_peak_nominal_tflops": FP32_NOMINAL_TFLOPS,
        "gpu_launches_whole_run": launches_total, "clocks_whole_run": clocks_all,
    }
    print(json.dumps(line), flush=True)
    if args.dump_outputs:
        dump_output(args.dump_outputs, "audio", main["last_audio"])
    if cx.world > 1:
        cx.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--samples", type=int, default=N_SAMPLES)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--configs", default="1,3,4,5", help="other BASELINE configs to run after the headline (subset of 1,3,4,5; '' = none)")
    ap.add_argument("--n3", type=int, default=1 << 30, help="config 3 stream length (BASELINE: 2^30)")
    ap.add_argument("--n4", type=int, default=1 << 26, help="config 4 wideband stream length (BASELINE: 2^26)")
    ap.add_argument("--cfg4-world", type=int, default=0, help="development aid: run rank 0's channel share of a W-GPU partition on one GPU")
    ap.add_argument("--n5", type=int, default=1 << 28, help="config 5 stream length (BASELINE: 2^28)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline chain's audio from its last timed step (rank 0) as DIR/audio.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        reference_arm(args)
    else:
        ours(args)


if __name__ == "__main__":
    main()
