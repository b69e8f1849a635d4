// include/dsp/channelizer.h — ChannelizerT<T>: the single-handle equivalent of the reference's Splitter<T> feeding N x VFO
// (vfo.h:9-111) and N x FloatFMDemod (demodulator.h:81-99), on one qdsp_channelizer. A uniform comb of 256 channels fs / 256
// apart at decimation 1280 takes the FFT polyphase form; any other set of offsets the direct form. Either way the wideband
// stream is read once per run() block instead of once per channel, and no per-channel copy of it is made.
#pragma once
#include <cmath>
#include <mutex>
#include <string>
#include <vector>
#include <dsp/block.h>

namespace dsp {
    // T is the input sample type: complex_t, or integer IQ (complex_s16_t, complex_s8_t, complex_u8_t), converted to
    // complex_t on the GPU (qdsp_channelizer_set_input_format). Stream c of `out` carries channel c's FM audio, the stream
    // a reference graph's FloatFMDemod::out of channel c would carry; stream c of `iqOut` (with iq = true) its complex
    // baseband, VFO::out of channel c. Each channel stream holds floor(C * I / D) + 1 elements, what one input block yields
    // (C: the input stream's capacity, STREAM_BUFFER_SIZE for a default stream), not STREAM_BUFFER_SIZE: 256 channels with
    // IQ then pin 4.8 MB, not 4 GB. A larger input block (an input rebound with setInput) is refused: run() returns -1.
    //
    // run() makes one process (or process_iq) call per input block: the kernels write every channel into one planar
    // buffer, and one scatter launch per output kind copies each row into its channel's stream buffer, through a device
    // table of those buffers built once per stream side. Retunes (setOffset / setOffsets) and setInputScale apply from the
    // next run() block, never in the middle of one; a retune synchronises the device (qdsp_channelizer_set_offsets).
    // stop() or setInput() may interrupt run() while it publishes a block channel by channel (a slow sink): the next run()
    // first publishes the block on the channels it had not reached, so every channel stream carries every block, in order.
    template <class T>
    class ChannelizerT : public generic_block<ChannelizerT<T>> {
        using base = generic_block<ChannelizerT<T>>;

    public:
        using base::init;
        ChannelizerT() {}
        ChannelizerT(stream<T>* in, const std::vector<float>& offsets, float inSampleRate, float outSampleRate, float bandWidth,
                     float deviation, bool audio = true, bool iq = false) {
            init(in, offsets, inSampleRate, outSampleRate, bandWidth, deviation, audio, iq);
        }
        ~ChannelizerT() {
            base::stop();
            release();
        }
        void init(stream<T>* in, const std::vector<float>& offsets, float inSampleRate, float outSampleRate, float bandWidth,
                  float deviation, bool audio = true, bool iq = false) {
            release();
            _in = in;
            _offsets = offsets;
            _error.clear();
            delivering = false;
            if (!audio && !iq) {
                _error = "dsp::Channelizer: neither audio nor iq output requested";
            } else {
                h = qdsp_channelizer_create((int)offsets.size(), offsets.data(), inSampleRate, outSampleRate, bandWidth, deviation);
                if (!h) { _error = qdsp_last_error(); }
            }
            if (h) {
                int interp = 1, decim = 1;
                qdsp_channelizer_design(h, nullptr, &interp, &decim);
                _interp = interp;
                _decim = decim;
                const long long inCap = _in ? _in->capacity() : STREAM_BUFFER_SIZE;
                _cap = (int)((inCap * interp) / decim) + 1;
                const int nch = (int)offsets.size();
                if (iq_format<T>::code != QDSP_CF32) { qdsp_channelizer_set_input_format(h, iq_format<T>::code, iq_format<T>::scale, iq_format<T>::offset); }
                if (audio) {
                    audioPlanar = (float*)qdsp_malloc_device((size_t)nch * _cap * sizeof(float));
                    for (int c = 0; c < nch; c++) {
                        out.push_back(new stream<float>(_cap));
                        base::registerOutput(out.back());
                    }
                }
                if (iq) {
                    iqPlanar = (complex_t*)qdsp_malloc_device((size_t)nch * _cap * sizeof(complex_t));
                    for (int c = 0; c < nch; c++) {
                        iqOut.push_back(new stream<complex_t>(_cap));
                        base::registerOutput(iqOut.back());
                    }
                }
            }
            base::registerInput(_in);
        }
        void setInput(stream<T>* in) { base::rebindInput(_in, in); }

        // VFO::setOffset of channel c (vfo.h:69-72): its NCO phase is continuous, every other channel is untouched.
        // false (nothing changes) for a channel out of range or a non-finite offset.
        bool setOffset(int c, float offset) {
            std::lock_guard<std::mutex> lck(base::ctrlMtx);
            if (c < 0 || c >= (int)_offsets.size() || !std::isfinite(offset)) { return false; }
            _offsets[c] = offset;
            post();
            return true;
        }
        // every channel at once: false (nothing changes) unless there is one finite offset per channel
        bool setOffsets(const std::vector<float>& offsets) {
            std::lock_guard<std::mutex> lck(base::ctrlMtx);
            if (offsets.size() != _offsets.size()) { return false; }
            for (float o : offsets) {
                if (!std::isfinite(o)) { return false; }
            }
            _offsets = offsets;
            post();
            return true;
        }
        // integer input: y = (float(x) + offset) * scale per component (e.g. 1 / 2048 for BladeRF sc16q11)
        void setInputScale(float scale, float offset) {
            std::lock_guard<std::mutex> lck(base::ctrlMtx);
            std::lock_guard<std::mutex> p(pendMtx);
            pendScale = true;
            _scale = scale;
            _scaleOffset = offset;
        }
        int channels() const { return (int)_offsets.size(); }
        // elements each channel stream holds
        int channelCapacity() const { return _cap; }
        // the handle (NULL when init() failed): qdsp_channelizer_fft_form and the other C calls
        qdsp_channelizer* handle() { return h; }
        // why init() left the block without a handle, why the last retune was refused or why run() refused a block
        // (empty when none of these happened); a copy, since the worker thread may set it again
        std::string error() const {
            std::lock_guard<std::mutex> p(pendMtx);
            return _error;
        }

        int run() override {
            const qdsp_stream_t s = base::cuStream;
            if (!publish()) { return -1; }      // the rest of a block that stop() / setInput() interrupted
            const int count = _in->readDevice(s);
            if (count < 0 || !h) { return -1; }
            if (((long long)count * _interp) / _decim + 1 > _cap) {
                // the planar buffers and the channel streams hold _cap outputs per channel: never write past them
                setError("dsp::Channelizer: input block larger than the channel streams were sized for");
                _in->flushDevice(s);
                return -1;
            }
            applyPending();
            // one uniform block of `count` samples: the same partition as blocks = {count}, and the FFT form can take it
            const long long n = iqPlanar
                ? qdsp_channelizer_process_iq(h, _in->readDev(), iqPlanar, audioPlanar, _cap, count, nullptr, 0, count, s)
                : qdsp_channelizer_process(h, _in->readDev(), audioPlanar, _cap, count, nullptr, 0, count, s);
            _in->flushDevice(s);
            if (n < 0) { return -1; }
            if (!scatter(out, audioPlanar, audioTab, audioNext, (int)n) || !scatter(iqOut, iqPlanar, iqTab, iqNext, (int)n)) { return -1; }
            pendN = (int)n;
            nextAudio = nextIq = 0;
            delivering = true;
            return publish() ? count : -1;
        }

        std::vector<stream<float>*> out;
        std::vector<stream<complex_t>*> iqOut;

    private:
        struct Table {
            void** dev = nullptr;             // [nch] device pointers
            std::vector<void*> host;          // the same, on the host
        };

        void post() {
            std::lock_guard<std::mutex> p(pendMtx);
            pendOffsets = _offsets;
            pendRetune = true;
        }
        void setError(const char* e) {
            std::lock_guard<std::mutex> p(pendMtx);
            _error = e;
        }
        void applyPending() {
            std::lock_guard<std::mutex> p(pendMtx);
            if (pendScale && iq_format<T>::code != QDSP_CF32) { qdsp_channelizer_set_input_format(h, iq_format<T>::code, _scale, _scaleOffset); }
            pendScale = false;
            if (pendRetune && qdsp_channelizer_set_offsets(h, pendOffsets.data()) != 0) { _error = qdsp_last_error(); }
            pendRetune = false;
        }
        // the device table of the buffers that take this block: the channel streams swap together, so the two tables (one
        // per side) are built once; every entry is checked against the streams before a table is used, and a table that
        // does not match is built again
        template <class E>
        void** table(std::vector<stream<E>*>& v, Table (&tab)[2], int& next) {
            for (Table& t : tab) {
                bool same = t.dev != nullptr;
                for (size_t c = 0; same && c < v.size(); c++) { same = t.host[c] == (void*)v[c]->writeDev(); }
                if (same) { return t.dev; }
            }
            Table& t = tab[next];
            next ^= 1;
            if (t.dev) { qdsp_stream_sync(base::cuStream); }   // the scatter that last read this table has finished
            else { t.dev = (void**)qdsp_malloc_device(v.size() * sizeof(void*)); }
            t.host.resize(v.size());
            for (size_t c = 0; c < v.size(); c++) { t.host[c] = v[c]->writeDev(); }
            qdsp_copy_h2d(t.dev, t.host.data(), v.size() * sizeof(void*), base::cuStream);
            return t.dev;
        }
        // row c of the planar buffer -> channel c's write buffer, once the channel's previous reader has let go of it
        template <class E>
        bool scatter(std::vector<stream<E>*>& v, E* planar, Table (&tab)[2], int& next, int n) {
            if (v.empty()) { return true; }
            for (stream<E>* st : v) { st->acquireWriteDev(base::cuStream); }
            return qdsp_scatter_rows(planar, _cap, table(v, tab, next), (int)v.size(), n, (int)sizeof(E), base::cuStream) >= 0;
        }
        // publish the scattered block channel by channel; a stop while a slow sink holds channel c back leaves channels
        // c.. for the next run() (their write buffers keep the block: nothing else writes them)
        bool publish() {
            if (!delivering) { return true; }
            for (; nextAudio < out.size(); nextAudio++) {
                if (!out[nextAudio]->swapDevice(pendN, base::cuStream)) { return false; }
            }
            for (; nextIq < iqOut.size(); nextIq++) {
                if (!iqOut[nextIq]->swapDevice(pendN, base::cuStream)) { return false; }
            }
            delivering = false;
            return true;
        }
        void release() {
            for (stream<float>* s : out) { base::unregisterOutput(s); delete s; }
            for (stream<complex_t>* s : iqOut) { base::unregisterOutput(s); delete s; }
            out.clear();
            iqOut.clear();
            if (_in) { base::unregisterInput(_in); }
            for (Table* tab : {audioTab, iqTab}) {
                for (int i = 0; i < 2; i++) {
                    if (tab[i].dev) { qdsp_free_device(tab[i].dev); }
                    tab[i] = Table();
                }
            }
            audioNext = iqNext = 0;
            delivering = false;
            if (audioPlanar) { qdsp_free_device(audioPlanar); }
            if (iqPlanar) { qdsp_free_device(iqPlanar); }
            audioPlanar = nullptr;
            iqPlanar = nullptr;
            if (h) { qdsp_channelizer_destroy(h); }
            h = nullptr;
        }

        stream<T>* _in = nullptr;
        qdsp_channelizer* h = nullptr;
        std::vector<float> _offsets;
        int _cap = 0, _interp = 1, _decim = 1;
        float* audioPlanar = nullptr;           // [nch][_cap]: what the kernels write
        complex_t* iqPlanar = nullptr;
        Table audioTab[2], iqTab[2];
        int audioNext = 0, iqNext = 0;          // per kind, the table a rebuild replaces (the older one)
        bool delivering = false;                // a scattered block not yet published on every channel stream
        int pendN = 0;
        size_t nextAudio = 0, nextIq = 0;       // the first channel stream of each kind it has not been published on
        mutable std::mutex pendMtx;                   // setters -> the next run() block (run() never takes ctrlMtx: stop() holds it)
        std::vector<float> pendOffsets;
        bool pendRetune = false, pendScale = false;
        float _scale = 1.0f, _scaleOffset = 0.0f;
        std::string _error;
    };
    using Channelizer = ChannelizerT<complex_t>;
}
