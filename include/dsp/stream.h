// include/dsp/stream.h — dsp::stream<T>, the double-buffered hand-off between blocks, device-resident.
//
// Source-compatible with the reference (src/dsp/stream.h:10-125): public `writeBuf` / `readBuf` raw
// pointers that host code may dereference, `swap(n)`, `read()`, `flush()`, `stopWriter()/stopReader()`
// and the clear calls, -1 / false on stop. What changed underneath (SURVEY.md §8b.3):
//   * each of the two buffers has a PINNED host side (what writeBuf/readBuf point at) and a DEVICE side;
//   * a producer that computed on the GPU calls `swapDevice(n, cudaStream)`, a consumer that computes on the
//     GPU calls `readDevice(cudaStream)`: block -> block hops never touch the host, ordering between the two
//     blocks' CUDA streams is carried by events (no host synchronisation);
//   * `read()` by a host consumer after a device producer performs the one D2H copy, `readDevice()` after a
//     host producer performs the one H2D copy -- the copies happen exactly at the graph's edges.
#pragma once
#include <condition_variable>
#include <mutex>
#include <qdsp_b200.h>

#define STREAM_BUFFER_SIZE 1000000  // elements per buffer, as in the reference (src/dsp/stream.h:7)

namespace dsp {
    class untyped_steam {  // (sic) the reference's spelling, kept for source compatibility
    public:
        virtual ~untyped_steam() {}
        virtual bool swap(int size) { return false; }
        virtual int read() { return -1; }
        virtual void flush() {}
        virtual void stopWriter() {}
        virtual void clearWriteStop() {}
        virtual void stopReader() {}
        virtual void clearReadStop() {}
    };

    template <class T>
    class stream : public untyped_steam {
        enum Residency { ON_HOST, ON_DEVICE };
        struct Side {
            T* host = nullptr;
            T* dev = nullptr;
            Residency where = ON_HOST;
            void* produced = nullptr;  // recorded by a device producer after its last kernel
            void* consumed = nullptr;  // recorded by a device consumer when it lets go of the buffer
            bool consumedValid = false;
        };

    public:
        stream() { allocate(STREAM_BUFFER_SIZE); }
        // an addition: buffers of `capacity` elements instead of STREAM_BUFFER_SIZE, for streams that never carry more
        // (a decimating block's outputs: dsp::ChannelizerT owns one per channel)
        explicit stream(int capacity) { allocate(capacity > 0 ? capacity : 1); }
        ~stream() {
            for (Side& s : side) {
                qdsp_free_pinned(s.host);
                qdsp_free_device(s.dev);
                qdsp_event_destroy(s.produced);
                qdsp_event_destroy(s.consumed);
            }
        }
        stream(const stream&) = delete;
        stream& operator=(const stream&) = delete;

        // ---- host-side protocol (unchanged semantics) -------------------------------------------
        bool swap(int size) override { return publish(size, ON_HOST, nullptr); }
        int read() override {
            const int n = awaitData();
            if (n < 0) { return -1; }
            Side& s = side[rd];
            if (s.where == ON_DEVICE) {  // device producer, host consumer: the graph's output edge
                qdsp_event_sync(s.produced);
                qdsp_copy_d2h(s.host, s.dev, (size_t)n * sizeof(T), nullptr);
                qdsp_stream_sync(nullptr);
            }
            return n;
        }
        void flush() override { release(nullptr); }

        // ---- device-side protocol (used by the blocks of this library) ---------------------------
        T* writeDev() { return side[wr].dev; }
        T* readDev() { return side[rd].dev; }
        // producer finished enqueueing kernels that fill writeDev() on `cuStream`
        bool swapDevice(int size, qdsp_stream_t cuStream) { return publish(size, ON_DEVICE, cuStream); }
        // consumer: returns the element count, makes `cuStream` wait for the producer's kernels (or uploads
        // host-written data); the data is at readDev()
        int readDevice(qdsp_stream_t cuStream) {
            const int n = awaitData();
            if (n < 0) { return -1; }
            Side& s = side[rd];
            if (s.where == ON_DEVICE) { qdsp_stream_wait_event(cuStream, s.produced); }
            else { qdsp_copy_h2d(s.dev, s.host, (size_t)n * sizeof(T), cuStream); }  // the graph's input edge
            return n;
        }
        // consumer enqueued everything that reads readDev() on `cuStream`
        void flushDevice(qdsp_stream_t cuStream) { release(cuStream); }
        // call before the first kernel that writes writeDev(): waits (on the GPU) for the previous reader
        void acquireWriteDev(qdsp_stream_t cuStream) {
            Side& s = side[wr];
            if (s.consumedValid) { qdsp_stream_wait_event(cuStream, s.consumed); }
        }

        void stopWriter() override { setFlag(writerStop, true); }
        void clearWriteStop() override { setFlag(writerStop, false); }
        void stopReader() override { setFlag(readerStop, true); }
        void clearReadStop() override { setFlag(readerStop, false); }

        T* writeBuf;
        T* readBuf;

        // elements each of the two buffers holds
        int capacity() const { return cap; }

    private:
        void allocate(int n) {
            cap = n;
            for (Side& s : side) {
                s.host = (T*)qdsp_malloc_pinned((size_t)n * sizeof(T));
                s.dev = (T*)qdsp_malloc_device((size_t)n * sizeof(T));
                s.produced = qdsp_event_create();
                s.consumed = qdsp_event_create();
            }
            wr = 0;
            rd = 1;
            writeBuf = side[wr].host;
            readBuf = side[rd].host;
        }
        bool publish(int size, Residency where, qdsp_stream_t cuStream) {
            std::unique_lock<std::mutex> lk(mtx);
            cv.wait(lk, [this] { return !full || writerStop; });
            if (writerStop) { return false; }
            Side& filled = side[wr];
            filled.where = where;
            if (where == ON_DEVICE) { qdsp_event_record(filled.produced, cuStream); }
            count = size;
            const int t = wr; wr = rd; rd = t;
            writeBuf = side[wr].host;
            readBuf = side[rd].host;
            // a host producer must not scribble over pinned memory a device reader may still be copying from
            if (side[wr].consumedValid && where == ON_HOST) { qdsp_event_sync(side[wr].consumed); }
            full = true;
            lk.unlock();
            cv.notify_all();
            return true;
        }
        int awaitData() {
            std::unique_lock<std::mutex> lk(mtx);
            cv.wait(lk, [this] { return full || readerStop; });
            return readerStop ? -1 : count;
        }
        void release(qdsp_stream_t cuStream) {
            {
                std::lock_guard<std::mutex> lk(mtx);
                Side& s = side[rd];
                if (cuStream != nullptr || s.where == ON_DEVICE) {
                    qdsp_event_record(s.consumed, cuStream);
                    s.consumedValid = true;
                } else {
                    s.consumedValid = false;
                }
                full = false;
            }
            cv.notify_all();
        }
        void setFlag(bool& flag, bool v) {
            { std::lock_guard<std::mutex> lk(mtx); flag = v; }
            cv.notify_all();
        }

        Side side[2];
        int wr, rd;
        std::mutex mtx;
        std::condition_variable cv;
        bool full = false;
        bool readerStop = false, writerStop = false;
        int count = 0;
        int cap = 0;
    };
}
