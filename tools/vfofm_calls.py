"""tools/vfofm_calls.py — back-to-back calls of the fused VFO -> FM chain (config 2's step) on one handle, timed with one
CUDA event pair around the whole loop, with the per-launch timing ring (qdsp_vfofm_enable_timing_ring, what bench.py turns
on for its headline region) off and on, and overlapped launches allowed (QDSP_PDL=1) or not (QDSP_PDL=0).

    python tools/vfofm_calls.py [--trees . OTHER_TREE] [--pdl 1 0] [--steps 200] [--loops 4] [--reps 2]

Each (tree, QDSP_PDL) runs in a subprocess of its own (the library reads the variable once); the combinations are
alternated `--reps` times, and inside a subprocess ring-off and ring-on loops alternate `--loops` times.
Every call reads the same input and writes the same audio buffer, as bench.py's timed steps do. One JSON line per loop,
then one summary line per arm (median GS/s). `audio_crc` is the CRC-32 of the last call's audio bytes: equal values mean
bit-identical audio across arms and trees."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import zlib

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
N_SAMPLES = 1 << 28
BLOCK = 819_200
FS, FC, FM, DEV = 2_400_000, 250_000, 1_000, 5e3
OUT_SR, BW = 48e3, 48e3


def child(a):
    sys.path.insert(0, os.path.abspath(a.tree))
    import torch
    from qdsp_b200 import blocks as B, lib

    L = lib.load()
    dev = torch.device("cuda:0")
    sp = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    n = a.samples
    x = torch.empty(n, dtype=torch.complex64, device=dev)
    lib.check(L.qdsp_synth_fm_cf32(x.data_ptr(), 0, n, FS, FC, FM, DEV, 0.5, 0.005, 2, sp))
    chain = B.VFOFM(float(FC), float(FS), OUT_SR, BW, DEV)
    n_out = chain.out_count(n, BLOCK)
    audio = torch.empty(n_out + 64, dtype=torch.float32, device=dev)

    def step():
        m = L.qdsp_vfofm_process(chain.h, x.data_ptr(), audio.data_ptr(), None, n, None, 0, BLOCK, None, sp)
        if m != n_out:
            raise SystemExit(f"process returned {m}, expected {n_out}: {lib.last_error()}")

    for _ in range(a.warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for loop in range(a.loops):
        for ring in (0, 1):
            if ring:
                lib.check(L.qdsp_vfofm_enable_timing_ring(chain.h, a.steps), "enable_timing_ring")
            else:
                L.qdsp_vfofm_enable_timing(chain.h, 0)
            e0.record()
            for _ in range(a.steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            rec = {"tree": a.tree, "pdl": os.environ.get("QDSP_PDL", "1"),
                   "ring": ring, "loop": loop, "steps": a.steps, "ms": round(ms, 4),
                   "us_per_call": round(ms * 1e3 / a.steps, 2), "GS_per_s": round(n * a.steps / ms / 1e6, 1)}
            if ring:
                nrec = C.c_int(0)
                k_ms = float(L.qdsp_vfofm_kernel_ms_mean(chain.h, C.byref(nrec)))
                rec.update({"ring_us_mean": round(k_ms * 1e3, 2), "ring_launches": nrec.value})
            print(json.dumps(rec), flush=True)
    L.qdsp_vfofm_enable_timing(chain.h, 0)
    crc = zlib.crc32(audio[:n_out].cpu().numpy().tobytes())
    print(json.dumps({"tree": a.tree, "pdl": os.environ.get("QDSP_PDL", "1"),
                      "calls": a.warmup + 2 * a.loops * a.steps, "audio_crc": f"{crc:08x}"}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trees", nargs="+", default=["."], help="repository trees whose built library to time (alternated)")
    ap.add_argument("--pdl", nargs="+", default=["1", "0"], help="QDSP_PDL values")
    ap.add_argument("--steps", type=int, default=200, help="calls per timed loop")
    ap.add_argument("--loops", type=int, default=4, help="ring-off / ring-on loop pairs per subprocess")
    ap.add_argument("--reps", type=int, default=2, help="subprocesses per arm, alternated")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--samples", type=int, default=N_SAMPLES)
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--tree", default=".", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        child(a)
        return
    rows = []
    for _ in range(a.reps):
        for tree in a.trees:
            for pdl in a.pdl:
                env = dict(os.environ, QDSP_PDL=str(pdl))
                cmd = [sys.executable, os.path.abspath(__file__), "--child", "--tree", tree, "--steps", str(a.steps),
                       "--loops", str(a.loops), "--warmup", str(a.warmup), "--samples", str(a.samples)]
                out = subprocess.run(cmd, env=env, cwd=REPO, check=True, capture_output=True, text=True).stdout
                for line in out.splitlines():
                    print(line, flush=True)
                    rows.append(json.loads(line))
    arms = {}
    for r in rows:
        if "ring" in r:
            arms.setdefault((r["tree"], r["pdl"], r["ring"]), []).append(r)
    for (tree, pdl, ring), rs in arms.items():
        g = [r["GS_per_s"] for r in rs]
        s = {"summary": True, "tree": tree, "pdl": pdl, "ring": ring, "loops": len(g),
             "GS_per_s_median": statistics.median(g), "GS_per_s_min": min(g), "GS_per_s_max": max(g)}
        if ring:
            s["ring_us_mean_median"] = statistics.median(r["ring_us_mean"] for r in rs)
        print(json.dumps(s), flush=True)
    crcs = sorted({r["audio_crc"] for r in rows if "audio_crc" in r})
    print(json.dumps({"summary": True, "audio_crcs": crcs, "all_equal": len(crcs) == 1}), flush=True)


if __name__ == "__main__":
    main()
