// include/dsp/spectrum.h — SpectrumT<T>: Welch-averaged power spectrum rows of an IQ stream (qdsp_spectrum_*), the
// data of a spectrum or waterfall display. An addition: the reference computes no spectrum.
#pragma once
#include <mutex>
#include <string>
#include <dsp/block.h>

namespace dsp {
    // Each output row is fftSize floats: the mean of `average` consecutive |FFT(window * frame)|^2, frames `hop` samples
    // apart, FFT-shifted (bin 0 is -fs / 2), linear power. A row is a pure function of the stream, so the run() sizes of
    // the input do not change it. Requires average * hop >= fftSize: rows then never hold more floats than the samples
    // that completed them (plus one row), and one stream buffer always has room; otherwise (or with a bad fftSize, hop,
    // average or window, include/qdsp_b200.h) init() leaves the block without a handle, run() returns -1 and error()
    // says why.
    // T is the input sample type: complex_t, or integer IQ (complex_s16_t, complex_s8_t, complex_u8_t) with the usual
    // conversion of iq_format<T> until setInputScale. The frames kernel reads the integers itself: the input edge copies
    // 4 or 2 bytes per sample and no complex_t copy of the stream is made (except at fftSize 16384 with hop <= fftSize,
    // include/qdsp_b200.h). Spectrum is the complex_t block.
    template <class T>
    class SpectrumT : public generic_block<SpectrumT<T>> {
        using base = generic_block<SpectrumT<T>>;

    public:
        SpectrumT() {}
        SpectrumT(stream<T>* in, int fftSize, const float* window, int hop, int average) { init(in, fftSize, window, hop, average); }
        ~SpectrumT() {
            base::stop();
            if (h) { qdsp_spectrum_destroy(h); }
        }
        void init(stream<T>* in, int fftSize, const float* window, int hop, int average) {
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
            if (h && iq_format<T>::code != QDSP_CF32) {
                qdsp_spectrum_set_input_format(h, iq_format<T>::code, iq_format<T>::scale, iq_format<T>::offset);
            }
            base::registerInput(_in);
            base::registerOutput(&out);
        }
        void setInput(stream<T>* in) { base::rebindInput(_in, in); }
        // integer input: y = (float(x) + offset) * scale per component (e.g. 1 / 2048 for BladeRF sc16q11), from the next
        // run() block on (a finite, non-zero scale and a finite offset; anything else is ignored)
        void setInputScale(float scale, float offset) {
            std::lock_guard<std::mutex> lck(scaleMtx);
            pendScale = true;
            _scale = scale;
            _scaleOffset = offset;
        }
        // why init() left the block without a handle (NULL when it has one)
        const char* error() const { return h ? nullptr : _error.c_str(); }
        int run() override {
            const int count = _in->readDevice(base::cuStream);
            if (count < 0 || !h) { return -1; }
            {
                std::lock_guard<std::mutex> lck(scaleMtx);
                if (pendScale && iq_format<T>::code != QDSP_CF32) { qdsp_spectrum_set_input_format(h, iq_format<T>::code, _scale, _scaleOffset); }
                pendScale = false;
            }
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
        stream<T>* _in = nullptr;
        qdsp_spectrum* h = nullptr;
        int _fftSize = 0;
        std::string _error;   // a copy: qdsp_last_error() is overwritten by the thread's next failing call
        std::mutex scaleMtx;  // setInputScale -> the next run() block
        bool pendScale = false;
        float _scale = 1.0f, _scaleOffset = 0.0f;
    };
    using Spectrum = SpectrumT<complex_t>;
}
