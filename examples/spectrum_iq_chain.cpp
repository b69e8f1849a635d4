// examples/spectrum_iq_chain.cpp — a raw recording as the radio delivered it (interleaved int16 cs16: USRP, BladeRF, ...;
// int8 cs8: HackRF; uint8 cu8: RTL-SDR) -> SpectrumT<T> -> FileSink<float>: the rows of a waterfall display, computed on
// the GPU. The samples stay integers up to the frames kernel: the input edge copies 4 or 2 bytes per sample, and no
// complex_t copy of the stream is made (except at fftSize 16384 with hop <= fftSize, include/qdsp_b200.h).
//
//   g++ -O2 -std=c++17 -Iinclude examples/spectrum_iq_chain.cpp -Lqdsp_b200 -lqdsp_b200 -lpthread -o spectrum_iq_chain
//   ./spectrum_iq_chain cs16|cs8|cu8 in.raw out.f32 fftSize hop average [block]
//     (out.f32: rows of fftSize float32 powers, bin 0 = -fs / 2; Hann window; the usual conversion of the format)
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include <dsp/sink.h>
#include <dsp/spectrum.h>

template <class T>
static int run_graph(FILE* f, const char* outPath, int fftSize, int hop, int average, int block, long long& fed) {
    std::vector<float> window(fftSize);
    for (int i = 0; i < fftSize; i++) { window[i] = (float)(0.5 - 0.5 * cos(2.0 * M_PI * i / fftSize)); }
    dsp::stream<T> input;
    dsp::SpectrumT<T> spectrum(&input, fftSize, window.data(), hop, average);
    if (spectrum.error()) { fprintf(stderr, "%s\n", spectrum.error()); return 2; }
    dsp::FileSink<float> sink(&spectrum.out, outPath);
    if (!sink.isOpen()) { fprintf(stderr, "cannot open %s\n", outPath); return 1; }
    spectrum.start();
    sink.start();
    for (;;) {
        const size_t n = fread(input.writeBuf, sizeof(T), block, f);
        if (n == 0) { break; }
        if (!input.swap((int)n)) { break; }
        fed += (long long)n;
    }
    // drain as examples/spectrum_chain.cpp does: the second empty swap returns once the last block's rows are written
    for (int i = 0; i < 2; i++) { input.swap(0); }
    spectrum.stop();
    sink.stop();
    return 0;
}

int main(int argc, char** argv) {
    if (argc < 7) { fprintf(stderr, "usage: %s cs16|cs8|cu8 in.raw out.f32 fftSize hop average [block]\n", argv[0]); return 2; }
    const char* fmt = argv[1];
    const int fftSize = atoi(argv[4]), hop = atoi(argv[5]), average = atoi(argv[6]);
    const int block = argc > 7 ? atoi(argv[7]) : STREAM_BUFFER_SIZE;
    if (block <= 0 || block > STREAM_BUFFER_SIZE) { fprintf(stderr, "block must be in [1, %d]\n", STREAM_BUFFER_SIZE); return 2; }
    if (fftSize <= 0) { fprintf(stderr, "fftSize must be positive\n"); return 2; }
    FILE* f = fopen(argv[2], "rb");
    if (!f) { perror(argv[2]); return 1; }
    if (qdsp_device_count() <= 0) { fprintf(stderr, "no CUDA device: %s\n", qdsp_last_error()); return 3; }

    long long fed = 0;
    int rc;
    if (!strcmp(fmt, "cs16")) { rc = run_graph<dsp::complex_s16_t>(f, argv[3], fftSize, hop, average, block, fed); }
    else if (!strcmp(fmt, "cs8")) { rc = run_graph<dsp::complex_s8_t>(f, argv[3], fftSize, hop, average, block, fed); }
    else if (!strcmp(fmt, "cu8")) { rc = run_graph<dsp::complex_u8_t>(f, argv[3], fftSize, hop, average, block, fed); }
    else { fprintf(stderr, "unknown format %s\n", fmt); rc = 2; }
    fclose(f);
    if (rc != 0) { return rc; }
    printf("fed %lld %s samples through SpectrumT(%d, hop %d, average %d) -> FileSink\n", fed, fmt, fftSize, hop, average);
    return 0;
}
