// include/dsp/convertion.h (sic) — ComplexToStereo, ComplexToReal, ComplexToImag, RealToComplex (reference
// src/dsp/convertion.h:5-170), and IQToComplex<T>: integer IQ from a radio front end to complex_t.
#pragma once
#include <dsp/audio.h>

namespace dsp {
    class ComplexToStereo : public detail::layout_block<ComplexToStereo, complex_t, stereo_t, QDSP_LAYOUT_COMPLEX_TO_STEREO> {
    public:
        ComplexToStereo() {}
        ComplexToStereo(stream<complex_t>* in) { init(in); }
        static_assert(sizeof(complex_t) == sizeof(stereo_t), "Can't convert complex to stereo: different sizes");  // convertion.h:11
    };
    class ComplexToReal : public detail::layout_block<ComplexToReal, complex_t, float, QDSP_LAYOUT_COMPLEX_TO_REAL> {
    public:
        ComplexToReal() {}
        ComplexToReal(stream<complex_t>* in) { init(in); }
    };
    class ComplexToImag : public detail::layout_block<ComplexToImag, complex_t, float, QDSP_LAYOUT_COMPLEX_TO_IMAG> {
    public:
        ComplexToImag() {}
        ComplexToImag(stream<complex_t>* in) { init(in); }
    };
    class RealToComplex : public detail::layout_block<RealToComplex, float, complex_t, QDSP_LAYOUT_REAL_TO_COMPLEX> {
    public:
        RealToComplex() {}
        RealToComplex(stream<float>* in) { init(in); }
    };

    // stream<complex_s16_t | complex_s8_t | complex_u8_t> -> stream<complex_t>, so any graph (VFO, PSKDemod, ...) can start
    // from radio samples; the graph's input edge then copies 4 or 2 bytes per sample (qdsp_iq_convert_process)
    template <class T>
    class IQToComplex : public generic_block<IQToComplex<T>> {
        using base = generic_block<IQToComplex<T>>;

    public:
        IQToComplex() {}
        IQToComplex(stream<T>* in, float scale = iq_format<T>::scale, float offset = iq_format<T>::offset) { init(in, scale, offset); }
        ~IQToComplex() { base::stop(); }
        void init(stream<T>* in, float scale = iq_format<T>::scale, float offset = iq_format<T>::offset) {
            _in = in;
            _scale = scale;
            _offset = offset;
            base::registerInput(_in);
            base::registerOutput(&out);
        }
        void setInput(stream<T>* in) { base::rebindInput(_in, in); }
        int run() override {
            const int count = _in->readDevice(base::cuStream);
            if (count < 0) { return -1; }
            out.acquireWriteDev(base::cuStream);
            const long long n = qdsp_iq_convert_process(iq_format<T>::code, _scale, _offset, _in->readDev(), out.writeDev(), count,
                                                        base::cuStream);
            _in->flushDevice(base::cuStream);
            if (n < 0) { return -1; }
            if (!out.swapDevice(count, base::cuStream)) { return -1; }
            return count;
        }

        stream<complex_t> out;

    private:
        stream<T>* _in = nullptr;
        float _scale = 1.0f, _offset = 0.0f;
    };
}
