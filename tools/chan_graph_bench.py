"""The dsp:: channelizer graph against the C ABI it runs on, and the cost of one retune, on one GPU at config 4's geometry.

256 channels fs / 256 apart (61.44 MS/s -> 48 kS/s, 10 241 taps, D = 1280: the FFT polyphase form), run() blocks of
819 200 samples. Arms, alternated for `--rounds` rounds:

  c_abi        qdsp_channelizer_process on 2^26 device-resident samples, uniform 819 200-sample blocks, audio only
               (bench.py configs.cfg4's call at N = 1), CUDA events over >= 0.7 s of back-to-back calls
  graph        host producer thread -> dsp::Channelizer -> 256 sinks that recycle their buffer as NullSink does (and count
               the blocks): the producer uploads two blocks once, into the two device sides of the input stream, and then
               only publishes them (swapDevice), so the graph is device-resident after that first copy. Wall clock over
               `--graph-blocks` blocks after warm-up, from the first publish to every sink holding the last block and a
               device synchronise
  graph_iq     the same with IQ on: 256 more streams of complex baseband, 256 more sinks
  retune       one qdsp_channelizer_set_offsets on the 256-channel handle (the whole comb moved by 3 bins and back: the FFT
               form is kept), host clock, mean over `--retunes` calls

One JSON line per (round, arm) with gsps (wideband input samples per second / 1e9), the card name, power limit and clocks
(nvidia-smi, read right after the timed region). `--trace DIR` also writes a torch.profiler trace of one graph pass and its
kernel / API summary. The graph is compiled into a temporary directory; nothing is written into the tree.

  python tools/chan_graph_bench.py [--rounds R] [--out FILE.jsonl] [--trace DIR]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from chan_iq_bench import smi, timed  # noqa: E402

N_SAMPLES = 1 << 26
BLOCK = 819_200
NCH, FS, SPACING, D = 256, 61_440_000, 240_000, 1280
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")

GRAPH = r"""
#include <atomic>
#include <chrono>
#include <memory>
#include <thread>
#include <vector>
#include <cuda_runtime.h>
#include <dsp/channelizer.h>

// NullSink's run(), counting the blocks it has recycled
template <class E> class CountSink : public dsp::generic_block<CountSink<E>> {
    using base = dsp::generic_block<CountSink<E>>;
public:
    CountSink(dsp::stream<E>* in) : _in(in) { base::registerInput(_in); }
    ~CountSink() { base::stop(); }
    int run() override {
        const int count = _in->readDevice(base::cuStream);
        if (count < 0) return -1;
        _in->flushDevice(base::cuStream);
        blocks++;
        return count;
    }
    std::atomic<long long> blocks{0};
private:
    dsp::stream<E>* _in;
};

extern "C" double graph_run(int nch, const float* offsets, int block, int warm, int blocks, int iq, const void* two_blocks_host) {
    std::vector<float> offs(offsets, offsets + nch);
    dsp::stream<dsp::complex_t> input;
    dsp::Channelizer chan(&input, offs, 61.44e6f, 48e3f, 48e3f, 5e3f, true, iq != 0);
    if (!chan.error().empty()) return -1.0;
    std::vector<std::unique_ptr<CountSink<float>>> sa;
    std::vector<std::unique_ptr<CountSink<dsp::complex_t>>> sq;
    for (auto* s : chan.out) { sa.emplace_back(new CountSink<float>(s)); sa.back()->start(); }
    for (auto* s : chan.iqOut) { sq.emplace_back(new CountSink<dsp::complex_t>(s)); sq.back()->start(); }
    chan.start();
    qdsp_stream_t ps = qdsp_stream_create();
    auto wait = [&](long long b) {
        for (auto& s : sa) while (s->blocks.load() < b) std::this_thread::yield();
        for (auto& s : sq) while (s->blocks.load() < b) std::this_thread::yield();
        cudaDeviceSynchronize();
    };
    // the first copy: one block into each device side of the input stream; from then on the producer only publishes
    long long fed = 0;
    for (int b = 0; b < 2; b++) {
        qdsp_copy_h2d(input.writeDev(), (const char*)two_blocks_host + (size_t)b * block * 8, (size_t)block * 8, ps);
        input.swapDevice(block, ps);
        fed++;
    }
    for (; fed < warm; fed++) input.swapDevice(block, ps);
    wait(fed);
    const auto t0 = std::chrono::steady_clock::now();
    for (int b = 0; b < blocks; b++, fed++) input.swapDevice(block, ps);
    wait(fed);
    const auto t1 = std::chrono::steady_clock::now();
    chan.stop();
    for (auto& s : sa) s->stop();
    for (auto& s : sq) s->stop();
    qdsp_stream_destroy(ps);
    return std::chrono::duration<double>(t1 - t0).count();
}
"""


def build_graph(tmp):
    src, so = os.path.join(tmp, "graph.cpp"), os.path.join(tmp, "libchangraph.so")
    with open(src, "w") as f:
        f.write(GRAPH)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I" + os.path.join(ROOT, "include"),
                           "-I" + os.path.join(CUDA, "include"), src, "-L" + os.path.join(ROOT, "qdsp_b200"), "-lqdsp_b200",
                           "-L" + os.path.join(CUDA, "lib64"), "-lcudart", "-lpthread",
                           "-Wl,-rpath," + os.path.join(ROOT, "qdsp_b200"), "-Wl,-rpath," + os.path.join(CUDA, "lib64"), "-o", so])
    g = C.CDLL(so)
    g.graph_run.restype = C.c_double
    g.graph_run.argtypes = [C.c_int, C.POINTER(C.c_float), C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    return g


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--graph-blocks", type=int, default=400)
    ap.add_argument("--retunes", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--trace", default=None, help="directory for a torch.profiler trace of one graph pass")
    args = ap.parse_args()
    import numpy as np
    import torch

    from qdsp_b200 import blocks as B, lib, synth

    L = lib.load()
    lib.require_device()
    torch.cuda.init()
    n = N_SAMPLES
    x = B.DevBuf(n * 8)
    lib.check(L.qdsp_synth_comb_cf32(x.ptr, 0, n, FS, NCH, SPACING, 5e3, 1.0 / 64.0, 0.001, 4, None))
    two = np.ascontiguousarray(x.to_numpy(np.complex64, 2 * BLOCK))
    stride = n // D + 64
    audio = B.DevBuf(NCH * stride * 4)
    offs = synth.cfg4_offsets(NCH, SPACING)
    moved = (offs.astype(np.float64) + 3 * SPACING).astype(np.float32)
    ch = B.Channelizer(offs, float(FS), 48e3, 48e3, 5e3)
    ch.seek(0)
    rt = B.Channelizer(offs, float(FS), 48e3, 48e3, 5e3)
    rt.process_device(x.ptr, audio.ptr, 4 * BLOCK, stride, BLOCK)
    out = open(args.out, "a") if args.out else None

    def emit(rec):
        rec.update(smi())
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")

    with tempfile.TemporaryDirectory() as tmp:
        g = build_graph(tmp)
        fp = offs.ctypes.data_as(C.POINTER(C.c_float))
        for r in range(args.rounds):
            ms, k = timed(torch, lambda: ch.process_device(x.ptr, audio.ptr, n, stride, BLOCK))
            emit({"tool": "chan_graph_bench", "round": r, "arm": "c_abi", "samples_per_call": n, "block": BLOCK, "calls": k,
                  "ms_per_call": round(ms, 4), "gsps": round(n / ms / 1e6, 2)})
            for arm, iq in (("graph", 0), ("graph_iq", 1)):
                sec = g.graph_run(NCH, fp, BLOCK, 8, args.graph_blocks, iq, two.ctypes.data)
                assert sec > 0, "graph_run failed"
                emit({"tool": "chan_graph_bench", "round": r, "arm": arm, "block": BLOCK, "blocks": args.graph_blocks,
                      "ms_per_block": round(sec * 1e3 / args.graph_blocks, 4),
                      "gsps": round(args.graph_blocks * BLOCK / sec / 1e9, 2)})
            ts = []
            for i in range(args.retunes):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                rt.set_offsets(moved if i % 2 == 0 else offs)
                ts.append(time.perf_counter() - t0)
                assert rt.fft_form
                rt.process_device(x.ptr, audio.ptr, BLOCK, stride, BLOCK)   # a call between retunes, as in use
            emit({"tool": "chan_graph_bench", "round": r, "arm": "retune", "retunes": args.retunes,
                  "ms_mean": round(1e3 * sum(ts) / len(ts), 4), "ms_max": round(1e3 * max(ts), 4)})
        if args.trace:
            from torch.profiler import ProfilerActivity, profile

            os.makedirs(args.trace, exist_ok=True)
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                g.graph_run(NCH, fp, BLOCK, 8, 100, 0, two.ctypes.data)
            prof.export_chrome_trace(os.path.join(args.trace, "chan_graph.pt.trace.json"))
            with open(os.path.join(args.trace, "chan_graph_summary.txt"), "w") as f:
                f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=40))
                f.write("\n")
                f.write(prof.key_averages().table(sort_by="cpu_time_total", row_limit=40))
    if out:
        out.close()


if __name__ == "__main__":
    main()
