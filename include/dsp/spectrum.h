// include/dsp/spectrum.h — Spectrum: Welch-averaged power spectrum rows of a complex_t stream (qdsp_spectrum_*), the
// data of a spectrum or waterfall display. An addition: the reference computes no spectrum.
#pragma once
#include <string>
#include <dsp/block.h>

namespace dsp {
    // Each output row is fftSize floats: the mean of `average` consecutive |FFT(window * frame)|^2, frames `hop` samples
    // apart, FFT-shifted (bin 0 is -fs / 2), linear power. A row is a pure function of the stream, so the run() sizes of
    // the input do not change it. Requires average * hop >= fftSize: rows then never hold more floats than the samples
    // that completed them (plus one row), and one stream buffer always has room; otherwise (or with a bad fftSize, hop,
    // average or window, include/qdsp_b200.h) init() leaves the block without a handle, run() returns -1 and error()
    // says why.
    class Spectrum : public generic_block<Spectrum> {
        using base = generic_block<Spectrum>;

    public:
        Spectrum() {}
        Spectrum(stream<complex_t>* in, int fftSize, const float* window, int hop, int average) { init(in, fftSize, window, hop, average); }
        ~Spectrum() {
            base::stop();
            if (h) { qdsp_spectrum_destroy(h); }
        }
        void init(stream<complex_t>* in, int fftSize, const float* window, int hop, int average) {
            _in = in;
            _fftSize = fftSize;
            if (h) { qdsp_spectrum_destroy(h); }
            h = nullptr;
            _error.clear();
            if ((long long)average * hop < fftSize) {
                _error = "dsp::Spectrum: average * hop must be at least fftSize";
            } else {
                h = qdsp_spectrum_create(fftSize, window, hop, average);
                if (!h) { _error = qdsp_last_error(); }
            }
            base::registerInput(_in);
            base::registerOutput(&out);
        }
        void setInput(stream<complex_t>* in) { base::rebindInput(_in, in); }
        // why init() left the block without a handle (NULL when it has one)
        const char* error() const { return h ? nullptr : _error.c_str(); }
        int run() override {
            const int count = _in->readDevice(base::cuStream);
            if (count < 0 || !h) { return -1; }
            // a piece of c samples completes at most c / (average * hop) + 1 rows, i.e. at most c + fftSize floats: a full
            // input buffer goes through in two pieces, each swapped out on its own
            const int piece = STREAM_BUFFER_SIZE - _fftSize;
            int done = 0;
            do {
                const int c = count - done < piece ? count - done : piece;
                out.acquireWriteDev(base::cuStream);
                const long long rows = qdsp_spectrum_process(h, _in->readDev() + done, out.writeDev(), c, base::cuStream);
                if (rows < 0) { _in->flushDevice(base::cuStream); return -1; }
                if (!out.swapDevice((int)(rows * _fftSize), base::cuStream)) { _in->flushDevice(base::cuStream); return -1; }
                done += c;
            } while (done < count);
            _in->flushDevice(base::cuStream);
            return count;
        }

        stream<float> out;

    private:
        stream<complex_t>* _in = nullptr;
        qdsp_spectrum* h = nullptr;
        int _fftSize = 0;
        std::string _error;   // a copy: qdsp_last_error() is overwritten by the thread's next failing call
    };
}
