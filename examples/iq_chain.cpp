// examples/iq_chain.cpp — a main.cpp-style graph fed with a raw recording as the radio delivered it: interleaved
// int16 (cs16: USRP, BladeRF, LimeSDR, ...), int8 (cs8: HackRF) or uint8 (cu8: RTL-SDR) pairs. The samples stay
// integers up to the GPU: the input edge copies 4 or 2 bytes per sample, and FusedVFOFloatFMDemodT<T> takes them
// directly; with `convert`, IQToComplex<T> turns them into complex_t for the block-by-block VFO -> FloatFMDemod graph.
//
//   g++ -O2 -std=c++17 -Iinclude examples/iq_chain.cpp -Lqdsp_b200 -lqdsp_b200 -lpthread -o iq_chain
//   ./iq_chain cs16|cs8|cu8 in.raw out.f32 [block] [convert]      (raw f32 audio out)
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include <thread>
#include <vector>
#include <dsp/convertion.h>
#include <dsp/demodulator.h>
#include <dsp/sink.h>
#include <dsp/vfo.h>

static std::vector<float> audio;
static std::atomic<long long> received{0};
static void audioHandler(float* data, int count, void* ctx) {
    audio.insert(audio.end(), data, data + count);
    received += count;
}

template <class T>
static long long run_graph(FILE* f, int block, bool convert) {
    dsp::stream<T> input;
    dsp::FusedVFOFloatFMDemodT<T> chain;
    dsp::IQToComplex<T> toComplex;
    dsp::VFO vfo;
    dsp::FloatFMDemod demod;
    dsp::HandlerSink<float> sink;
    if (convert) {
        toComplex.init(&input);
        vfo.init(&toComplex.out, 250e3, 2.4e6, 48e3, 48e3);
        demod.init(vfo.out, 48e3, 5e3);
        sink.init(&demod.out, audioHandler, NULL);
        toComplex.start();
        vfo.start();
        demod.start();
    } else {
        chain.init(&input, 250e3, 2.4e6, 48e3, 48e3, 5e3);
        sink.init(&chain.out, audioHandler, NULL);
        chain.start();
    }
    sink.start();

    long long fed = 0, expect = 0;
    for (;;) {
        const size_t n = fread(input.writeBuf, sizeof(T), block, f);
        if (n == 0) { break; }
        if (!input.swap((int)n)) { break; }
        fed += (long long)n;
        expect += (long long)n / 50;  // I = 1, D = 50: every run() block yields count / 50 outputs
    }
    while (received.load() < expect) { std::this_thread::yield(); }
    sink.stop();
    if (convert) { demod.stop(); vfo.stop(); toComplex.stop(); } else { chain.stop(); }
    return fed;
}

int main(int argc, char** argv) {
    if (argc < 4) { fprintf(stderr, "usage: %s cs16|cs8|cu8 in.raw out.f32 [block] [convert]\n", argv[0]); return 2; }
    const char* fmt = argv[1];
    const int block = argc > 4 ? atoi(argv[4]) : 819200;
    const bool convert = argc > 5 && !strcmp(argv[5], "convert");
    FILE* f = fopen(argv[2], "rb");
    if (!f) { perror(argv[2]); return 1; }
    if (qdsp_device_count() <= 0) { fprintf(stderr, "no CUDA device: %s\n", qdsp_last_error()); return 3; }

    long long fed;
    if (!strcmp(fmt, "cs16")) { fed = run_graph<dsp::complex_s16_t>(f, block, convert); }
    else if (!strcmp(fmt, "cs8")) { fed = run_graph<dsp::complex_s8_t>(f, block, convert); }
    else if (!strcmp(fmt, "cu8")) { fed = run_graph<dsp::complex_u8_t>(f, block, convert); }
    else { fprintf(stderr, "unknown format %s\n", fmt); return 2; }
    fclose(f);

    FILE* o = fopen(argv[3], "wb");
    if (!o) { perror(argv[3]); return 1; }
    fwrite(audio.data(), sizeof(float), audio.size(), o);
    fclose(o);
    printf("fed %lld %s samples, wrote %zu audio samples (%s)\n", fed, fmt, audio.size(), convert ? "IQToComplex -> VFO -> FloatFMDemod" : "fused");
    return 0;
}
