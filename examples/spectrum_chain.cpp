// examples/spectrum_chain.cpp — a raw cf32 recording -> Spectrum -> FileSink<float>: the rows of a waterfall display,
// computed on the GPU. The IQ crosses to the device once, at the input edge; only the rows come back.
//
//   g++ -O2 -std=c++17 -Iinclude examples/spectrum_chain.cpp -Lqdsp_b200 -lqdsp_b200 -lpthread -o spectrum_chain
//   ./spectrum_chain in.cf32 out.f32 fftSize hop average [block] [window.f32]
//     (out.f32: rows of fftSize float32 powers, bin 0 = -fs / 2; window.f32: fftSize float32 values, default rectangular)
#include <stdio.h>
#include <stdlib.h>
#include <vector>
#include <dsp/sink.h>
#include <dsp/spectrum.h>

int main(int argc, char** argv) {
    if (argc < 6) { fprintf(stderr, "usage: %s in.cf32 out.f32 fftSize hop average [block] [window.f32]\n", argv[0]); return 2; }
    const int fftSize = atoi(argv[3]), hop = atoi(argv[4]), average = atoi(argv[5]);
    const int block = argc > 6 ? atoi(argv[6]) : STREAM_BUFFER_SIZE;
    if (block <= 0 || block > STREAM_BUFFER_SIZE) { fprintf(stderr, "block must be in [1, %d]\n", STREAM_BUFFER_SIZE); return 2; }
    std::vector<float> window;
    if (argc > 7) {
        FILE* w = fopen(argv[7], "rb");
        if (!w) { perror(argv[7]); return 1; }
        window.resize(fftSize > 0 ? fftSize : 0);
        const size_t got = fread(window.data(), sizeof(float), window.size(), w);
        fclose(w);
        if ((int)got != fftSize) { fprintf(stderr, "%s holds fewer than %d floats\n", argv[7], fftSize); return 1; }
    }
    FILE* f = fopen(argv[1], "rb");
    if (!f) { perror(argv[1]); return 1; }
    if (qdsp_device_count() <= 0) { fprintf(stderr, "no CUDA device: %s\n", qdsp_last_error()); return 3; }

    dsp::stream<dsp::complex_t> input;
    dsp::Spectrum spectrum(&input, fftSize, window.empty() ? nullptr : window.data(), hop, average);
    if (spectrum.error()) { fprintf(stderr, "%s\n", spectrum.error()); return 2; }
    dsp::FileSink<float> sink(&spectrum.out, argv[2]);
    if (!sink.isOpen()) { fprintf(stderr, "cannot open %s\n", argv[2]); return 1; }
    spectrum.start();
    sink.start();

    long long fed = 0;
    for (;;) {
        const size_t n = fread(input.writeBuf, sizeof(dsp::complex_t), block, f);
        if (n == 0) { break; }
        if (!input.swap((int)n)) { break; }
        fed += (long long)n;
    }
    fclose(f);
    // drain: swap() returns once Spectrum's run() on the previous buffer has finished, rows swapped out included. So the
    // first empty swap returns when the last block's rows are out, the second when Spectrum has swapped out the empty
    // block's zero rows, which waited for FileSink to write the last block's rows.
    for (int i = 0; i < 2; i++) { input.swap(0); }
    spectrum.stop();
    sink.stop();
    printf("fed %lld samples through Spectrum(%d, hop %d, average %d) -> FileSink\n", fed, fftSize, hop, average);
    return 0;
}
