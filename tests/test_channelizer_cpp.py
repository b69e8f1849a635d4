"""dsp::ChannelizerT<T> (include/dsp/channelizer.h), the dsp:: block over one qdsp_channelizer handle: one stream per
channel for audio and for the complex baseband, retunes between run() blocks. CPU: the header compiles alone with -Wall
for every input type, and the example compiles. GPU: a graph compiled here (threaded blocks, the program is the producer
and retunes one channel between two known blocks) and examples/channelizer_chain.cpp are bit-identical to
blocks.Channelizer fed the same blocks with the same retune, also when stop() or setInput() interrupts the block while a
slow sink holds one channel back; the block's device and pinned allocations stay small."""
import json
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INC = os.path.join(ROOT, "include")
LINK = ["-L" + os.path.join(ROOT, "qdsp_b200"), "-lqdsp_b200", "-lpthread", "-Wl,-rpath," + os.path.join(ROOT, "qdsp_b200")]
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
TYPES = ["dsp::complex_t", "dsp::complex_s16_t", "dsp::complex_s8_t", "dsp::complex_u8_t"]
FS4 = 61.44e6
BLK = 163_840
NBLK = 4
RETUNE_BLOCK = 2
OFFGRID6 = [-20.1e6, -7.3e6, 0.5e6, 3.37e6, 11.9e6, 25.05e6]

GRAPH = r"""
// the test's graph: raw file -> stream<T> -> dsp::ChannelizerT<T> (started, its own thread) -> HandlerSink per channel
// stream; the program is the producer and retunes one channel once every sink holds the blocks before `rb`.
// QDSP_TEST_HOLD=kind:c:mode (kind audio | iq, mode stop | rebind): channel c's sink of that kind starts only after block
// 1, so the channelizer blocks on that channel while publishing block 1; the program then interrupts it with stop() and
// start() (or setInput(), which pauses and resumes the worker) before it lets the held sink run
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include <chrono>
#include <memory>
#include <thread>
#include <vector>
#include <cuda_runtime.h>
#include <dsp/channelizer.h>
#include <dsp/sink.h>

template <class E> struct Chan {
    std::vector<E> data;
    std::atomic<int> blocks{0};
    static void handler(E* d, int n, void* ctx) {
        Chan* c = (Chan*)ctx;
        c->data.insert(c->data.end(), d, d + n);
        c->blocks++;
    }
};

template <class T>
static int run(int argc, char** argv) {
    // fmt in out_prefix block iq rb rc roff inSR outSR bw dev offsets...
    FILE* f = fopen(argv[2], "rb");
    const std::string prefix = argv[3];
    const int block = atoi(argv[4]), iq = atoi(argv[5]), rb = atoi(argv[6]), rc = atoi(argv[7]);
    const float roff = (float)atof(argv[8]);
    std::vector<float> offs;
    for (int i = 13; i < argc; i++) offs.push_back((float)atof(argv[i]));
    const int nch = (int)offs.size();
    dsp::stream<T> input;
    dsp::ChannelizerT<T> chan(&input, offs, (float)atof(argv[9]), (float)atof(argv[10]), (float)atof(argv[11]), (float)atof(argv[12]), true, iq != 0);
    if (!chan.error().empty()) { fprintf(stderr, "%s\n", chan.error().c_str()); return 1; }
    char hkind[8] = "", hmode[8] = "";
    int hc = -1;
    if (const char* e = getenv("QDSP_TEST_HOLD")) {
        if (sscanf(e, "%7[a-z]:%d:%7[a-z]", hkind, &hc, hmode) != 3) { fprintf(stderr, "bad QDSP_TEST_HOLD\n"); return 2; }
    }
    const bool holdAudio = hc >= 0 && !strcmp(hkind, "audio"), holdIq = hc >= 0 && !strcmp(hkind, "iq");
    std::vector<Chan<float>> au(nch);
    std::vector<Chan<dsp::complex_t>> qs(iq ? nch : 0);
    std::vector<std::unique_ptr<dsp::HandlerSink<float>>> sa;
    std::vector<std::unique_ptr<dsp::HandlerSink<dsp::complex_t>>> sq;
    for (int c = 0; c < nch; c++) {
        sa.emplace_back(new dsp::HandlerSink<float>(chan.out[c], Chan<float>::handler, &au[c]));
        if (!(holdAudio && c == hc)) sa.back()->start();
        if (iq) {
            sq.emplace_back(new dsp::HandlerSink<dsp::complex_t>(chan.iqOut[c], Chan<dsp::complex_t>::handler, &qs[c]));
            if (!(holdIq && c == hc)) sq.back()->start();
        }
    }
    chan.start();
    auto wait_blocks = [&](int b) {
        for (auto& c : au) while (c.blocks.load() < b) std::this_thread::yield();
        for (auto& c : qs) while (c.blocks.load() < b) std::this_thread::yield();
    };
    int b = 0;
    for (;; b++) {
        const size_t n = fread(input.writeBuf, sizeof(T), block, f);
        if (n == 0) break;
        if (b == rb) {
            wait_blocks(b);   // block b - 1 has left the channelizer: the retune lands between b - 1 and b
            if (!chan.setOffset(rc, roff)) { fprintf(stderr, "setOffset refused\n"); return 1; }
        }
        input.swap((int)n);
        if (b == 1 && hc >= 0) {
            // the channels published before hc (audio goes first, then IQ) have block 1: the worker is stuck publishing it
            // on channel hc
            for (int c = 0; c < (holdAudio ? hc : nch); c++) { while (au[c].blocks.load() < 2) std::this_thread::yield(); }
            for (int c = 0; holdIq && c < hc; c++) { while (qs[c].blocks.load() < 2) std::this_thread::yield(); }
            std::this_thread::sleep_for(std::chrono::milliseconds(20));
            if (!strcmp(hmode, "stop")) { chan.stop(); }
            else { chan.setInput(&input); }
            if (holdAudio) sa[hc]->start(); else sq[hc]->start();
            if (!strcmp(hmode, "stop")) { chan.start(); }
        }
    }
    wait_blocks(b);
    chan.stop();
    for (auto& s : sa) s->stop();
    for (auto& s : sq) s->stop();
    FILE* o = fopen((prefix + ".audio").c_str(), "wb");
    for (auto& c : au) fwrite(c.data.data(), sizeof(float), c.data.size(), o);
    fclose(o);
    if (iq) {
        o = fopen((prefix + ".iq").c_str(), "wb");
        for (auto& c : qs) fwrite(c.data.data(), sizeof(dsp::complex_t), c.data.size(), o);
        fclose(o);
    }
    printf("blocks %d channels %d fft_form %d error %s\n", b, nch, qdsp_channelizer_fft_form(chan.handle()), chan.error().empty() ? "none" : chan.error().c_str());
    return 0;
}

// device memory a 256-channel block with IQ takes at construction (cudaMemGetInfo), and the pinned bytes of its streams
static int mem() {
    std::vector<float> offs(256);
    for (int c = 0; c < 256; c++) offs[c] = (c - 127.5f) * 240e3f;
    dsp::stream<dsp::complex_t> input;
    size_t free0, free1, total;
    cudaDeviceSynchronize();
    cudaMemGetInfo(&free0, &total);
    long long pinned = 0;
    {
        dsp::Channelizer chan(&input, offs, 61.44e6f, 48e3f, 48e3f, 5e3f, true, true);
        cudaDeviceSynchronize();
        cudaMemGetInfo(&free1, &total);
        for (auto* s : chan.out) pinned += 2ll * s->capacity() * (long long)sizeof(float);
        for (auto* s : chan.iqOut) pinned += 2ll * s->capacity() * (long long)sizeof(dsp::complex_t);
        printf("{\"device_bytes\": %lld, \"pinned_bytes\": %lld, \"channel_capacity\": %d, \"fft_form\": %d}\n",
               (long long)free0 - (long long)free1, pinned, chan.channelCapacity(), qdsp_channelizer_fft_form(chan.handle()));
    }
    return 0;
}

int main(int argc, char** argv) {
    if (argc > 1 && !strcmp(argv[1], "mem")) return mem();
    if (argc < 14) { fprintf(stderr, "usage\n"); return 2; }
    if (!strcmp(argv[1], "cf32")) return run<dsp::complex_t>(argc, argv);
    if (!strcmp(argv[1], "cs16")) return run<dsp::complex_s16_t>(argc, argv);
    return 2;
}
"""


def _compile_graph(tmp_path):
    src, exe = tmp_path / "chan_graph.cpp", tmp_path / "chan_graph"
    src.write_text(GRAPH)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I" + INC, "-I" + os.path.join(CUDA, "include"), str(src), *LINK,
                           "-L" + os.path.join(CUDA, "lib64"), "-lcudart", "-Wl,-rpath," + os.path.join(CUDA, "lib64"),
                           "-o", str(exe)])
    return str(exe)


def _compile_example(tmp_path):
    exe = tmp_path / "channelizer_chain"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-I" + INC, os.path.join(ROOT, "examples", "channelizer_chain.cpp"),
                           *LINK, "-o", str(exe)])
    return str(exe)


# ---- CPU ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("t", TYPES)
def test_header_compiles_alone_with_wall(qlib, tmp_path, t):
    src = tmp_path / "one.cpp"
    src.write_text("#include <dsp/channelizer.h>\n"
                   f"template class dsp::ChannelizerT<{t}>;\n"
                   f"int main() {{ dsp::ChannelizerT<{t}>* c = nullptr; return c ? c->channels() : 0; }}\n")
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Werror", "-I" + INC, str(src), *LINK, "-o", str(tmp_path / "one")])


def test_example_compiles(qlib, tmp_path):
    assert os.path.exists(_compile_example(tmp_path))


# ---- GPU ---------------------------------------------------------------------------------------------------------
def _case(name):
    from qdsp_b200 import synth

    if name == "comb256":
        offs = synth.cfg4_offsets(256)
        return offs, 10, float(offs[10]) + 9e3        # the retune takes the comb off the grid: direct form from then on
    return np.asarray(OFFGRID6, np.float32), 3, 3.41e6


def _reference(offs, x, rc, roff, fmt, iq):
    """blocks.Channelizer fed the same run() blocks, one call each, with the same retune before block RETUNE_BLOCK."""
    from qdsp_b200 import blocks as B

    ch = B.Channelizer(offs, FS4, 48e3, 48e3, 5e3)
    if fmt == "cs16":
        ch.set_input_format("cs16")
    per = 2 if fmt == "cs16" else 1
    auds, iqs = [], []
    for b in range(NBLK):
        if b == RETUNE_BLOCK:
            o = offs.copy()
            o[rc] = np.float32(roff)
            ch.set_offsets(o)
        xb = x[b * BLK * per:(b + 1) * BLK * per]
        if iq:
            q, a = ch.process_iq(xb, BLK)
            iqs.append(q)
        else:
            a = ch.process(xb, BLK)
        auds.append(a)
    return np.concatenate(auds, axis=1), (np.concatenate(iqs, axis=1) if iq else None)


def _input(fmt):
    from qdsp_b200 import synth

    x = synth.cfg4_input(0, NBLK * BLK, nch=256)
    return synth.quantize_iq(x, "cs16").reshape(-1) if fmt == "cs16" else x


def _bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("name,fmt,iq,hold", [("comb256", "cf32", 1, None), ("comb256", "cs16", 0, None),
                                              ("offgrid6", "cf32", 0, None), ("offgrid6", "cs16", 1, None),
                                              # stop() / setInput() while one channel's sink holds the block back
                                              ("comb256", "cf32", 1, "audio:200:stop"), ("comb256", "cf32", 1, "iq:7:rebind"),
                                              ("offgrid6", "cs16", 1, "iq:3:stop"), ("offgrid6", "cf32", 0, "audio:2:rebind")])
def test_graph_bit_identical_to_c_abi(qlib, tmp_path, name, fmt, iq, hold):
    exe = _compile_graph(tmp_path)
    offs, rc, roff = _case(name)
    x = _input(fmt)
    fin = tmp_path / "in.raw"
    x.tofile(fin)
    prefix = str(tmp_path / "out")
    args = [exe, fmt, str(fin), prefix, str(BLK), str(iq), str(RETUNE_BLOCK), str(rc), repr(roff), repr(FS4), "48000", "48000",
            "5000"] + [repr(float(o)) for o in offs]
    env = dict(os.environ, QDSP_TEST_HOLD=hold) if hold else None
    r = subprocess.run(args, capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "error none" in r.stdout and f"blocks {NBLK} " in r.stdout, r.stdout
    ya, yq = _reference(offs, x, rc, roff, fmt, iq)
    got = np.fromfile(prefix + ".audio", np.float32).reshape(len(offs), -1)
    assert _bits_equal(got, ya)
    if iq:
        gq = np.fromfile(prefix + ".iq", np.complex64).reshape(len(offs), -1)
        assert _bits_equal(gq.view(np.float32), yq.view(np.float32))


@pytest.mark.gpu
@pytest.mark.parametrize("name,fmt", [("comb256", "cf32"), ("offgrid6", "cs16")])
def test_example_bit_identical_to_c_abi(qlib, tmp_path, name, fmt):
    exe = _compile_example(tmp_path)
    offs, rc, roff = _case(name)
    x = _input(fmt)
    fin = tmp_path / "in.raw"
    x.tofile(fin)
    out = tmp_path / "out"
    out.mkdir()
    # the example's comb is (count, spacing, first): both sets here are evenly spaced or given as such
    n = len(offs)
    spacing = float(offs[1]) - float(offs[0]) if name == "comb256" else None
    if name == "comb256":
        comb = [str(n), repr(spacing), repr(float(offs[0]))]
    else:
        # six channels 4.93 MHz apart from -12.1 MHz: off the fs / 256 grid (direct form)
        offs = np.asarray([-12.1e6 + 4.93e6 * c for c in range(6)], np.float32)
        rc, roff = 3, float(offs[3]) + 2.5e3
        comb = ["6", "4930000", "-12100000"]
    args = [exe, fmt, str(fin), str(out), *comb, "--block", str(BLK), "--iq", "--retune", f"{rc}:{roff!r}@{RETUNE_BLOCK}"]
    r = subprocess.run(args, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    # the example builds its offsets in double and rounds them to float, as here
    ya, yq = _reference(offs, x, rc, np.float32(roff), fmt, True)
    for c in range(n):
        a = np.fromfile(out / f"ch{c:03d}.f32", np.float32)
        q = np.fromfile(out / f"ch{c:03d}.cf32", np.complex64)
        assert _bits_equal(a, ya[c]) and _bits_equal(q.view(np.float32), yq[c].view(np.float32)), c


@pytest.mark.gpu
def test_block_allocation_is_small(qlib, tmp_path):
    exe = _compile_graph(tmp_path)
    r = subprocess.run([exe, "mem"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    m = json.loads(r.stdout.strip().splitlines()[-1])
    print(m)
    assert m["fft_form"] == 1 and m["channel_capacity"] == 1_000_000 // 1280 + 1
    assert m["device_bytes"] < 64 << 20, m
    assert m["pinned_bytes"] < 64 << 20, m
