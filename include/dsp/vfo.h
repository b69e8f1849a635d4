// include/dsp/vfo.h — dsp::VFO (reference src/dsp/vfo.h:9-111): FrequencyXlator(-offset) feeding a
// PolyphaseResampler whose window is designed from (bandwidth, rates); `out` points at the resampler output.
// FusedVFOFloatFMDemod is this library's single-pass equivalent of VFO -> FloatFMDemod (one kernel, the
// translated and resampled IQ never leave the chip); it is numerically the composition of the three blocks.
#pragma once
#include <algorithm>
#include <dsp/block.h>
#include <dsp/processing.h>
#include <dsp/resampling.h>
#include <dsp/window.h>

namespace dsp {
    class VFO {
    public:
        VFO() {}
        ~VFO() { stop(); }
        VFO(stream<complex_t>* in, float offset, float inSampleRate, float outSampleRate, float bandWidth) {
            init(in, offset, inSampleRate, outSampleRate, bandWidth);
        }

        void init(stream<complex_t>* in, float offset, float inSampleRate, float outSampleRate, float bandWidth) {
            _in = in;
            _offset = offset;
            _inSampleRate = inSampleRate;
            _outSampleRate = outSampleRate;
            _bandWidth = bandWidth;
            const float cutoff = realCutoff();
            xlator.init(_in, _inSampleRate, -_offset);
            win.init(cutoff, cutoff, inSampleRate);
            resamp.init(&xlator.out, &win, _inSampleRate, _outSampleRate);
            win.setSampleRate(_inSampleRate * resamp.getInterpolation());
            resamp.updateWindow(&win);
            out = &resamp.out;
        }
        // the reference never sets `running` (vfo.h:38-48), which makes its stop() a no-op; here the flag is kept
        void start() {
            if (running) { return; }
            xlator.start();
            resamp.start();
            running = true;
        }
        void stop() {
            if (!running) { return; }
            xlator.stop();
            resamp.stop();
            running = false;
        }
        void setInSampleRate(float inSampleRate) {
            _inSampleRate = inSampleRate;
            const bool was = running;
            if (was) { stop(); }
            xlator.setSampleRate(_inSampleRate);
            resamp.setInSampleRate(_inSampleRate);
            redesign();
            if (was) { start(); }
        }
        void setOutSampleRate(float outSampleRate) {
            _outSampleRate = outSampleRate;
            const bool was = running;
            if (was) { stop(); }
            resamp.setOutSampleRate(_outSampleRate);
            redesign();
            if (was) { start(); }
        }
        void setOutSampleRate(float outSampleRate, float bandWidth) {
            _bandWidth = bandWidth;
            setOutSampleRate(outSampleRate);
        }
        void setOffset(float offset) {
            _offset = offset;
            xlator.setFrequency(-_offset);
        }
        void setBandwidth(float bandWidth) {
            _bandWidth = bandWidth;
            redesign();
        }

        stream<complex_t>* out = nullptr;

    private:
        float realCutoff() const { return std::min<float>(_bandWidth, std::min<float>(_inSampleRate, _outSampleRate)) / 2.0f; }
        void redesign() {
            const float cutoff = realCutoff();
            win.setSampleRate(_inSampleRate * resamp.getInterpolation());
            win.setCutoff(cutoff);
            win.setTransWidth(cutoff);
            resamp.updateWindow(&win);
        }
        bool running = false;
        float _offset = 0, _inSampleRate = 1, _outSampleRate = 1, _bandWidth = 1;
        filter_window::BlackmanWindow win;
        stream<complex_t>* _in = nullptr;
        FrequencyXlator<complex_t> xlator;
        PolyphaseResampler<complex_t> resamp;
    };

    // VFO -> FloatFMDemod in one kernel launch per run() call. T is the input sample type: complex_t, or integer IQ
    // (complex_s16_t, complex_s8_t, complex_u8_t), converted to complex_t on the GPU by one more kernel; the input edge
    // then copies 4 or 2 bytes per sample. FusedVFOFloatFMDemod is the complex_t chain.
    template <class T>
    class FusedVFOFloatFMDemodT : public generic_block<FusedVFOFloatFMDemodT<T>> {
        using base = generic_block<FusedVFOFloatFMDemodT<T>>;

    public:
        FusedVFOFloatFMDemodT() {}
        FusedVFOFloatFMDemodT(stream<T>* in, float offset, float inSampleRate, float outSampleRate, float bandWidth, float deviation) {
            init(in, offset, inSampleRate, outSampleRate, bandWidth, deviation);
        }
        ~FusedVFOFloatFMDemodT() {
            base::stop();
            if (h) { qdsp_vfofm_destroy(h); }
        }
        void init(stream<T>* in, float offset, float inSampleRate, float outSampleRate, float bandWidth, float deviation) {
            _in = in;
            if (h) { qdsp_vfofm_destroy(h); }
            h = qdsp_vfofm_create(offset, inSampleRate, outSampleRate, bandWidth, deviation);
            if (h && iq_format<T>::code != QDSP_CF32) { setInputScale(iq_format<T>::scale, iq_format<T>::offset); }
            base::registerInput(_in);
            base::registerOutput(&out);
        }
        void setOffset(float offset) { qdsp_vfofm_set_offset(h, offset); }
        // integer input: y = (float(x) + offset) * scale per component (e.g. 1 / 2048 for BladeRF sc16q11)
        void setInputScale(float scale, float offset) { qdsp_vfofm_set_input_format(h, iq_format<T>::code, scale, offset); }
        int run() override {
            const int count = _in->readDevice(base::cuStream);
            if (count < 0) { return -1; }
            out.acquireWriteDev(base::cuStream);
            const int one = count;
            const long long n = qdsp_vfofm_process(h, _in->readDev(), out.writeDev(), nullptr, count, &one, 1, 0, nullptr, base::cuStream);
            _in->flushDevice(base::cuStream);
            if (n < 0) { return -1; }
            if (!out.swapDevice((int)n, base::cuStream)) { return -1; }
            return count;
        }

        stream<float> out;

    private:
        stream<T>* _in = nullptr;
        qdsp_vfofm* h = nullptr;
    };
    using FusedVFOFloatFMDemod = FusedVFOFloatFMDemodT<complex_t>;
}
