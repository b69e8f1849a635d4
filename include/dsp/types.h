// include/dsp/types.h — POD sample types of the dsp:: mirror.
// Same names, layout (sizeof == 8, interleaved) and operators as the reference's src/dsp/types.h:7-84,
// so host code that fills stream buffers or inspects results compiles unchanged. Device kernels see
// these as float2.
#pragma once
#include <math.h>
#include <stdint.h>
#include <qdsp_b200.h>

#define FL_M_PI 3.1415926535f  // the reference's float "pi" (src/dsp/types.h:4)

namespace dsp {
    struct complex_t {
        float re;
        float im;

        complex_t operator*(const float b) const { return complex_t{re * b, im * b}; }
        complex_t operator/(const float b) const { return complex_t{re / b, im / b}; }
        complex_t operator*(const complex_t& b) const { return complex_t{(re * b.re) - (im * b.im), (im * b.re) + (re * b.im)}; }
        complex_t operator+(const complex_t& b) const { return complex_t{re + b.re, im + b.im}; }
        complex_t operator-(const complex_t& b) const { return complex_t{re - b.re, im - b.im}; }
        inline complex_t conj() const { return complex_t{re, -im}; }
        inline float phase() const { return atan2f(im, re); }
        // linear-approximation arctangent, the formula the FM demodulators use (types.h:36-54)
        inline float fastPhase() const {
            const float mag_im = fabsf(im);
            if (re == 0.0f && im == 0.0f) { return 0.0f; }
            float ang;
            if (re >= 0.0f) { ang = (FL_M_PI / 4.0f) - (FL_M_PI / 4.0f) * ((re - mag_im) / (re + mag_im)); }
            else { ang = (3.0f * (FL_M_PI / 4.0f)) - (FL_M_PI / 4.0f) * ((re + mag_im) / (mag_im - re)); }
            return (im < 0.0f) ? -ang : ang;
        }
        inline float amplitude() const { return sqrtf((re * re) + (im * im)); }
        // NOTE: the reference computes |re| twice here (types.h:58-64); FeedForwardAGC parity depends on it
        inline float fastAmplitude() const {
            const float a = fabsf(re);
            return a + 0.4f * a;
        }
    };

    struct stereo_t {
        float l;
        float r;
        stereo_t operator*(const float b) const { return stereo_t{l * b, r * b}; }
        stereo_t operator+(const stereo_t& b) const { return stereo_t{l + b.l, r + b.r}; }
        stereo_t operator-(const stereo_t& b) const { return stereo_t{l - b.l, r - b.r}; }
    };

    static_assert(sizeof(complex_t) == 8 && sizeof(stereo_t) == 8, "samples must be 8-byte interleaved pairs");

    // integer IQ as radio front ends deliver it (interleaved re, im): USRP / BladeRF / LimeSDR / SDRplay / Airspy HF+
    // (int16), HackRF (int8), RTL-SDR (uint8). Read as complex_t by IQToComplex<T> (convertion.h) and directly by
    // FusedVFOFloatFMDemodT<T> (vfo.h), both converting on the GPU: y = (float(x) + offset) * scale per component.
    struct complex_s16_t { int16_t re; int16_t im; };
    struct complex_s8_t { int8_t re; int8_t im; };
    struct complex_u8_t { uint8_t re; uint8_t im; };
    static_assert(sizeof(complex_s16_t) == 4 && sizeof(complex_s8_t) == 2 && sizeof(complex_u8_t) == 2, "packed pairs");

    // the C ABI format code of a sample type and its usual conversion (include/qdsp_b200.h)
    template <class T> struct iq_format;
    template <> struct iq_format<complex_t> {
        static constexpr int code = QDSP_CF32;
        static constexpr float scale = 1.0f, offset = 0.0f;
    };
    template <> struct iq_format<complex_s16_t> {
        static constexpr int code = QDSP_CS16;
        static constexpr float scale = 1.0f / 32768.0f, offset = 0.0f;
    };
    template <> struct iq_format<complex_s8_t> {
        static constexpr int code = QDSP_CS8;
        static constexpr float scale = 1.0f / 128.0f, offset = 0.0f;
    };
    template <> struct iq_format<complex_u8_t> {
        static constexpr int code = QDSP_CU8;
        static constexpr float scale = 1.0f / 128.0f, offset = -127.5f;
    };
}
