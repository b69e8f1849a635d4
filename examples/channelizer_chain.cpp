// examples/channelizer_chain.cpp — a many-channel receiver as a main.cpp-style graph: a raw recording (cf32, or cs16 as
// the radio delivered it) -> dsp::ChannelizerT<T> (one handle for N x [VFO -> FloatFMDemod]) -> one FileSink<float> per
// channel, and with --iq one FileSink<complex_t> per channel for its complex baseband. The comb is `count` channels,
// `spacing` Hz apart from `first` Hz; 256 channels 240 kHz apart at 61.44 MS/s (BASELINE config 4) take the FFT polyphase
// form. --retune c:offset@b moves channel c to `offset` Hz from run() block b on (phase continuous).
//
//   g++ -O2 -std=c++17 -Iinclude examples/channelizer_chain.cpp -Lqdsp_b200 -lqdsp_b200 -lpthread -o channelizer_chain
//   ./channelizer_chain cf32|cs16 in.raw outdir count spacing first [--block N] [--iq] [--retune c:offset@b]
//                       [--rates inSR outSR bandWidth deviation]          (outdir/chNNN.f32, outdir/chNNN.cf32)
//
// This program is its own producer and calls the block's run() itself, one input block at a time, so a retune lands
// exactly between blocks b - 1 and b; the sinks run on their own threads as usual.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <memory>
#include <string>
#include <vector>
#include <dsp/channelizer.h>
#include <dsp/sink.h>

struct Options {
    int count = 256, block = 819200, retuneCh = -1, retuneBlock = -1;
    double spacing = 240e3, first = -30.72e6;
    float retuneOffset = 0.0f, inSR = 61.44e6f, outSR = 48e3f, bw = 48e3f, dev = 5e3f;
    bool iq = false;
};

template <class T>
static long long run_graph(FILE* f, const std::string& dir, const Options& o) {
    std::vector<float> offsets(o.count);
    for (int c = 0; c < o.count; c++) { offsets[c] = (float)(o.first + c * o.spacing); }
    dsp::stream<T> input;
    dsp::ChannelizerT<T> chan(&input, offsets, o.inSR, o.outSR, o.bw, o.dev, true, o.iq);
    if (!chan.error().empty()) {
        fprintf(stderr, "channelizer: %s\n", chan.error().c_str());
        return -1;
    }
    std::vector<std::unique_ptr<dsp::FileSink<float>>> audio;
    std::vector<std::unique_ptr<dsp::FileSink<dsp::complex_t>>> iq;
    char name[64];
    for (int c = 0; c < o.count; c++) {
        snprintf(name, sizeof(name), "/ch%03d.f32", c);
        audio.emplace_back(new dsp::FileSink<float>(chan.out[c], dir + name));
        audio.back()->start();
        if (o.iq) {
            snprintf(name, sizeof(name), "/ch%03d.cf32", c);
            iq.emplace_back(new dsp::FileSink<dsp::complex_t>(chan.iqOut[c], dir + name));
            iq.back()->start();
        }
    }
    printf("%d channels, FFT polyphase form: %s\n", o.count, qdsp_channelizer_fft_form(chan.handle()) ? "yes" : "no");

    long long fed = 0;
    for (int b = 0;; b++) {
        const size_t n = fread(input.writeBuf, sizeof(T), o.block, f);
        if (n == 0) { break; }
        if (b == o.retuneBlock && !chan.setOffset(o.retuneCh, o.retuneOffset)) { fprintf(stderr, "bad --retune\n"); }
        input.swap((int)n);
        if (chan.run() < 0) {
            fprintf(stderr, "run: %s\n", chan.error().empty() ? qdsp_last_error() : chan.error().c_str());
            return -1;
        }
        fed += (long long)n;
    }
    // an empty block on every channel stream goes through once its sink has taken the last real one
    for (auto* s : chan.out) { s->swap(0); }
    for (auto* s : chan.iqOut) { s->swap(0); }
    for (auto& s : audio) { s->stop(); }
    for (auto& s : iq) { s->stop(); }
    return fed;
}

int main(int argc, char** argv) {
    if (argc < 7) {
        fprintf(stderr, "usage: %s cf32|cs16 in.raw outdir count spacing first [--block N] [--iq] [--retune c:offset@b] "
                        "[--rates inSR outSR bandWidth deviation]\n", argv[0]);
        return 2;
    }
    Options o;
    const char* fmt = argv[1];
    o.count = atoi(argv[4]);
    o.spacing = atof(argv[5]);
    o.first = atof(argv[6]);
    for (int i = 7; i < argc; i++) {
        if (!strcmp(argv[i], "--block") && i + 1 < argc) { o.block = atoi(argv[++i]); }
        else if (!strcmp(argv[i], "--iq")) { o.iq = true; }
        else if (!strcmp(argv[i], "--retune") && i + 1 < argc) {
            if (sscanf(argv[++i], "%d:%f@%d", &o.retuneCh, &o.retuneOffset, &o.retuneBlock) != 3) { fprintf(stderr, "--retune c:offset@b\n"); return 2; }
        } else if (!strcmp(argv[i], "--rates") && i + 4 < argc) {
            o.inSR = (float)atof(argv[i + 1]);
            o.outSR = (float)atof(argv[i + 2]);
            o.bw = (float)atof(argv[i + 3]);
            o.dev = (float)atof(argv[i + 4]);
            i += 4;
        } else { fprintf(stderr, "unknown argument %s\n", argv[i]); return 2; }
    }
    if (o.count <= 0 || o.block <= 0 || o.block > STREAM_BUFFER_SIZE) { fprintf(stderr, "bad count or block\n"); return 2; }
    FILE* f = fopen(argv[2], "rb");
    if (!f) { perror(argv[2]); return 1; }
    if (qdsp_device_count() <= 0) { fprintf(stderr, "no CUDA device: %s\n", qdsp_last_error()); return 3; }

    long long fed;
    if (!strcmp(fmt, "cf32")) { fed = run_graph<dsp::complex_t>(f, argv[3], o); }
    else if (!strcmp(fmt, "cs16")) { fed = run_graph<dsp::complex_s16_t>(f, argv[3], o); }
    else { fprintf(stderr, "unknown format %s\n", fmt); return 2; }
    fclose(f);
    if (fed < 0) { return 1; }
    printf("fed %lld %s samples to %d channels\n", fed, fmt, o.count);
    return 0;
}
