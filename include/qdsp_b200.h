/* include/qdsp_b200.h — C ABI of libqdsp_b200.so (B200 / sm_100a).
 *
 * This is the drop-in boundary underneath the reference's header-only `dsp::` block API
 * (AlexandreRouma/qdsp, src/dsp/*.h). The reference has no FFI seam of its own: every block is a
 * C++ class whose `run()` does the arithmetic on the CPU (mostly through VOLK). Each entry point
 * below replaces the body of one `run()` (cited per function) and is what the new
 * `include/dsp/*.h` mirror headers, the ctypes binding (`qdsp_b200/lib.py`) and `bench.py` call.
 *
 * Conventions
 *   - plain C types only; all `*_dev` pointers are CUDA device pointers owned by the caller;
 *     `qdsp_stream_t` is a `cudaStream_t` passed as `void*` (NULL = the legacy default stream);
 *   - every `*_process` call is asynchronous on that stream and allocation-free on the hot path;
 *   - return value mirrors `run()`: number of elements produced (>= 0) or -1 on error, with the
 *     text available from `qdsp_last_error()`;
 *   - per-block state (history tail, NCO phase, demod phase, IIR/AGC/PLL scalars) lives on the
 *     device inside the opaque handle and can be read/written with `*_get_state/_set_state`
 *     (used for checkpointing, parity injection and multi-GPU time-sharding);
 *   - where the reference's result depends on how the stream was cut into `run()` calls
 *     (resampler schedule restart, AGC decay) the batch entry points take the block partition:
 *     `blocks[nblocks]` (sizes, sum == count) or, with `blocks == NULL`, a uniform `nblocks`-way
 *     partition described by `block_size` (last block short).
 *   - there is NO CPU fallback: if no CUDA device is usable every compute entry point fails.
 */
#ifndef QDSP_B200_H
#define QDSP_B200_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

#define QDSP_ABI_VERSION 1
typedef void* qdsp_stream_t;
enum { QDSP_F32 = 0, QDSP_CF32 = 1 }; /* element type of a stream: float or {float re,im} (== stereo_t) */
/* integer IQ as radio front ends deliver it: interleaved (re, im) pairs of int16 (USRP, BladeRF sc16q11, LimeSDR,
 * SDRplay, Airspy HF+), int8 (HackRF) or uint8 (RTL-SDR). Accepted by qdsp_iq_convert_process and, after
 * *_set_input_format, by the fused VFO -> FM chain and the channelizer; every `dtype` argument rejects them. */
enum { QDSP_CS16 = 2, QDSP_CS8 = 3, QDSP_CU8 = 4 };

/* ---- runtime plumbing (replaces volk_malloc/volk_free in src/dsp/stream.h:25-31) ------------- */
int qdsp_abi_version(void);
const char* qdsp_last_error(void);
int qdsp_device_count(void);
int qdsp_set_device(int device);
int qdsp_get_device(void);
void* qdsp_malloc_device(size_t bytes);
void qdsp_free_device(void* p);
void* qdsp_malloc_pinned(size_t bytes);
void qdsp_free_pinned(void* p);
int qdsp_memset_device(void* dst_dev, int value, size_t bytes, qdsp_stream_t s);
int qdsp_copy_h2d(void* dst_dev, const void* src_host, size_t bytes, qdsp_stream_t s);
int qdsp_copy_d2h(void* dst_host, const void* src_dev, size_t bytes, qdsp_stream_t s);
int qdsp_copy_d2d(void* dst_dev, const void* src_dev, size_t bytes, qdsp_stream_t s);
int qdsp_copy_peer(void* dst_dev, int dst_device, const void* src_dev, int src_device, size_t bytes, qdsp_stream_t s);
int qdsp_enable_peer_access(int device, int peer);
/* cross-process peer memory (one process per GPU): export a qdsp_malloc_device allocation as a 64-byte handle, map a
 * peer process's handle into this process (reads / writes then travel over NVLink P2P), unmap it */
#define QDSP_IPC_HANDLE_BYTES 64
int qdsp_ipc_export(const void* dev_ptr, void* handle_out);
void* qdsp_ipc_open(const void* handle);
int qdsp_ipc_close(void* mapped);
qdsp_stream_t qdsp_stream_create(void);
void qdsp_stream_destroy(qdsp_stream_t s);
int qdsp_stream_sync(qdsp_stream_t s);
/* events order work between the per-block CUDA streams of the dsp:: mirror (include/dsp/stream.h) */
void* qdsp_event_create(void);
void qdsp_event_destroy(void* ev);
int qdsp_event_record(void* ev, qdsp_stream_t s);
int qdsp_stream_wait_event(qdsp_stream_t s, void* ev);
int qdsp_event_sync(void* ev);
/* number of kernels this library has launched in this process (bench.py "gpu_launches") */
long long qdsp_launch_count(void);

/* ---- integer IQ -> cf32 --------------------------------------------------------------------- *
 * One conversion rule wherever this library reads integer IQ: y = (float(x) + offset) * scale, each step rounded to  *
 * float32 (for cu8, x is the byte value 0..255). Usual parameters, all exact: cs16 1/32768, 0; cs8 1/128, 0; cu8     *
 * 1/128, -127.5; sc16q11 is cs16 with 1/2048. `scale` must be finite and non-zero, `offset` finite. in_dev holds      *
 * `count` pairs, aligned to its pair (4 bytes for cs16, 2 for the 8-bit formats); out_dev gets `count` cf32 samples.  */
long long qdsp_iq_convert_process(int fmt, float scale, float offset, const void* in_dev, void* out_dev, long long count,
                                  qdsp_stream_t s);

/* ---- tap design, host side, bit-exact with the reference (src/dsp/window.h) ------------------ */
int qdsp_blackman_tap_count(float cutoff, float transWidth, float sampleRate);                 /* window.h:36-50 */
void qdsp_blackman_taps(float cutoff, float transWidth, float sampleRate, float* taps, int tapCount,
                        float factor);                                                        /* window.h:52-70 */
void qdsp_blackman_bandpass_taps(float cutoff, float transWidth, float offset, float sampleRate, float* taps,
                                 int tapCount, float factor);                                 /* window.h:120-141 */
void qdsp_rrc_taps(int tapCount, float sampleRate, float baudRate, float alpha, float* taps);  /* window.h:184-229 */
void qdsp_rates_to_ratio(float inSampleRate, float outSampleRate, int* interp, int* decim);    /* resampling.h:28-30 */
/* VFO::init tap design (vfo.h:26-33): returns tap count; fills taps (if maxTaps suffices), I and D */
int qdsp_vfo_design(float inSampleRate, float outSampleRate, float bandWidth, float* taps, int maxTaps, int* interp,
                    int* decim);
/* resampler schedule of one block (resampling.h:121-125): phase[k] = (k*D)%I, index[k] = (k*D)/I */
int qdsp_resamp_schedule(int interp, int decim, int count, int* phase, int* index);

/* ---- FIR<float> / FIR<complex_t>::run, src/dsp/filter.h:51-74 ------------------------------- */
typedef struct qdsp_fir qdsp_fir;
qdsp_fir* qdsp_fir_create(int dtype, const float* taps, int tapCount);
void qdsp_fir_destroy(qdsp_fir* h);
int qdsp_fir_set_taps(qdsp_fir* h, const float* taps, int tapCount);      /* FIR::updateWindow, filter.h:43-49 */
long long qdsp_fir_process(qdsp_fir* h, const void* in_dev, void* out_dev, long long count, qdsp_stream_t s);
int qdsp_fir_history_len(qdsp_fir* h);                                     /* tapCount - 1 elements */
int qdsp_fir_get_history(qdsp_fir* h, void* hist_host);
int qdsp_fir_set_history(qdsp_fir* h, const void* hist_host);
/* time-sharding halo: adopt the previous shard's last (tapCount-1) elements, read from a device
 * pointer that may live on a peer GPU (NVLink P2P); replaces the memmove at filter.h:71 */
int qdsp_fir_import_tail(qdsp_fir* h, const void* tail_dev, int src_device, qdsp_stream_t s);
/* the same without the copy: this ONE call reads its (tapCount-1)-element history straight from `halo_dev` -- any
 * device-accessible pointer, e.g. the previous time shard's tail on a peer GPU mapped with qdsp_ipc_open (the kernel
 * loads go over NVLink); NULL = zeros. The handle's own history then continues from this call's input (filter.h:71). */
long long qdsp_fir_process_halo(qdsp_fir* h, const void* halo_dev, const void* in_dev, void* out_dev, long long count,
                                qdsp_stream_t s);
int qdsp_fir_reset(qdsp_fir* h);
/* force a kernel variant: 0 = auto, 1 = generic, 2 = register-blocked sm_100a kernel */
int qdsp_fir_set_variant(qdsp_fir* h, int variant);

/* ---- PolyphaseResampler<T>::run, src/dsp/resampling.h:99-132 (+buildTapPhases :137-166) ----- */
typedef struct qdsp_resamp qdsp_resamp;
qdsp_resamp* qdsp_resamp_create(int dtype, const float* taps, int tapCount, int interp, int decim);
void qdsp_resamp_destroy(qdsp_resamp* h);
int qdsp_resamp_set_taps(qdsp_resamp* h, const float* taps, int tapCount);
int qdsp_resamp_taps_per_phase(qdsp_resamp* h);
long long qdsp_resamp_out_count(qdsp_resamp* h, long long count);          /* calcOutSize, resampling.h:95-97 */
/* batch of run() calls over one contiguous input; out_counts (host, optional) gets per-block counts */
long long qdsp_resamp_process(qdsp_resamp* h, const void* in_dev, void* out_dev, long long count, const int* blocks,
                              int nblocks, int block_size, int* out_counts, qdsp_stream_t s);
/* device-evaluated schedule of the same batch (parity of indices): phase/index per output */
long long qdsp_resamp_schedule_device(qdsp_resamp* h, long long count, const int* blocks, int nblocks, int block_size,
                                      int* phase_dev, long long* index_dev, qdsp_stream_t s);
int qdsp_resamp_history_len(qdsp_resamp* h);                               /* tapsPerPhase elements */
int qdsp_resamp_get_history(qdsp_resamp* h, void* hist_host);
int qdsp_resamp_set_history(qdsp_resamp* h, const void* hist_host);
int qdsp_resamp_reset(qdsp_resamp* h);
int qdsp_resamp_set_variant(qdsp_resamp* h, int variant);

/* ---- PowerDecimator::run, src/dsp/resampling.h:220-249 ---------------------------------------- */
long long qdsp_power_decim_process(unsigned int power, const void* in_dev, void* out_dev, long long count,
                                   qdsp_stream_t s);

/* ---- FrequencyXlator<complex_t>::run + VOLK rotator, src/dsp/processing.h:55-70 ------------- */
typedef struct qdsp_xlator qdsp_xlator;
qdsp_xlator* qdsp_xlator_create(float sampleRate, float freq);             /* init, processing.h:16-24 */
void qdsp_xlator_destroy(qdsp_xlator* h);
int qdsp_xlator_set_frequency(qdsp_xlator* h, float sampleRate, float freq); /* processing.h:36-49 */
void qdsp_xlator_get_phase_delta(qdsp_xlator* h, float* re, float* im);
void qdsp_xlator_get_phase(qdsp_xlator* h, float* re, float* im);          /* VOLK `lv_32fc_t* phase` */
void qdsp_xlator_set_phase(qdsp_xlator* h, float re, float im);
long long qdsp_xlator_process(qdsp_xlator* h, const void* in_dev, void* out_dev, long long count, qdsp_stream_t s);

/* ---- FloatFMDemod / FMDemod::run, src/dsp/demodulator.h:81-99 / 158-178 ---------------------- */
typedef struct qdsp_fmdemod qdsp_fmdemod;
qdsp_fmdemod* qdsp_fmdemod_create(float sampleRate, float deviation, int stereo_out);
void qdsp_fmdemod_destroy(qdsp_fmdemod* h);
float qdsp_fmdemod_get_phase(qdsp_fmdemod* h);
int qdsp_fmdemod_set_phase(qdsp_fmdemod* h, float phase);
long long qdsp_fmdemod_process(qdsp_fmdemod* h, const void* in_dev, void* out_dev, long long count, qdsp_stream_t s);

/* ---- StereoFMDemod::run, src/dsp/demodulator.h:189-330 ("next" row of the scope table) ------------------------ *
 * FloatFMDemod -> pilot FIR<float>(BlackmanBandpassWindow(1000, 1000, 19000, fs)) -> AGC(20, fs) -> L/R matrix;   *
 * out_dev is stereo_t[count]; the run() partition matters through the AGC.                                          */
typedef struct qdsp_stereofm qdsp_stereofm;
qdsp_stereofm* qdsp_stereofm_create(float sampleRate, float deviation);
void qdsp_stereofm_destroy(qdsp_stereofm* h);
long long qdsp_stereofm_process(qdsp_stereofm* h, const void* in_dev, void* out_dev, long long count, const int* blocks,
                                int nblocks, int block_size, qdsp_stream_t s);
/* the matrix step alone: out[i] = {mpx + mpx*pilot^2, mpx - mpx*pilot^2} */
long long qdsp_stereo_matrix_process(const float* mpx_dev, const float* pilot_dev, void* out_dev, long long count,
                                     qdsp_stream_t s);

/* ---- fused VFO (vfo.h:19-36: Xlator(-offset) -> PolyphaseResampler) -> FloatFMDemod ---------- *
 * One pass: the translated and the resampled IQ never reach HBM unless iq_out_dev != NULL.        */
typedef struct qdsp_vfofm qdsp_vfofm;
qdsp_vfofm* qdsp_vfofm_create(float offset, float inSampleRate, float outSampleRate, float bandWidth,
                              float deviation);
void qdsp_vfofm_destroy(qdsp_vfofm* h);
int qdsp_vfofm_design(qdsp_vfofm* h, int* tapCount, int* interp, int* decim);
int qdsp_vfofm_set_offset(qdsp_vfofm* h, float offset);                    /* VFO::setOffset, vfo.h:87-90 */
/* NCO phase at the current stream position, as VOLK's `lv_32fc_t* phase` (processing.h:64,78): lets a caller
 * (or a parity test) re-synchronise the closed-form oscillator with a recursive float32 reference phasor */
void qdsp_vfofm_get_phase(qdsp_vfofm* h, float* re, float* im);
int qdsp_vfofm_set_phase(qdsp_vfofm* h, float re, float im);
long long qdsp_vfofm_out_count(qdsp_vfofm* h, long long count, const int* blocks, int nblocks, int block_size);
long long qdsp_vfofm_process(qdsp_vfofm* h, const void* in_dev, float* audio_out_dev, void* iq_out_dev,
                             long long count, const int* blocks, int nblocks, int block_size, int* out_counts,
                             qdsp_stream_t s);
/* same call with HOST buffers: chunked, double-buffered H2D / D2H inside (the end-to-end path) */
long long qdsp_vfofm_process_host(qdsp_vfofm* h, const void* in_host, float* audio_out_host, long long count,
                                  int block_size, qdsp_stream_t s);
int qdsp_vfofm_reset(qdsp_vfofm* h);
int qdsp_vfofm_set_variant(qdsp_vfofm* h, int variant);
/* element type of in_dev (process) and in_host (process_host) from the next call on: QDSP_CF32 (the default; scale and
 * offset ignored) or QDSP_CS16 / QDSP_CS8 / QDSP_CU8 with the conversion of qdsp_iq_convert_process. The state carried
 * from call to call (history tail, import_tail, history_len) stays cf32, so formats may change from call to call. */
int qdsp_vfofm_set_input_format(qdsp_vfofm* h, int fmt, float scale, float offset);
/* time-sharding: start this shard at absolute stream sample `start` (NCO phase in closed form),
 * history/demod state imported from the previous shard */
/* DEBUG replay of the reference's recursive float32 NCO (attribution of its drift, DESIGN.md "NCO"): the translator is
 * evaluated run by run of 512 samples from `ckpt_host` -- the phase state volk_32fc_s32fc_x2_rotator_32fc holds at the start
 * of every 512-sample run of every run() call (processing.h:64; n_ckpt = sum over blocks of ceil(count_b / 512), computed
 * by the caller, e.g. with the oracle's rotator) -- with the reference's float recursion inside a run: the mixed samples are
 * bit-identical to the reference's. Unfused (translator, resampler, demodulator as three kernels); state (history of the
 * MIXED stream, demodulator phase) is separate from the fused path's: do not interleave the two on one handle. cf32 input
 * only: fails after qdsp_vfofm_set_input_format with an integer format. */
long long qdsp_vfofm_process_replay(qdsp_vfofm* h, const void* in_dev, float* audio_out_dev, void* iq_out_dev,
                                    long long count, const int* blocks, int nblocks, int block_size,
                                    const float* ckpt_host, long long n_ckpt, qdsp_stream_t s);
int qdsp_vfofm_seek(qdsp_vfofm* h, long long start);
int qdsp_vfofm_import_tail(qdsp_vfofm* h, const void* tail_dev, int src_device, qdsp_stream_t s);
int qdsp_vfofm_history_len(qdsp_vfofm* h);
/* bench hook: bracket the dominant kernel of each process call with CUDA events on the caller's
 * stream; kernel_ms() synchronises and returns the last launch's device time */
int qdsp_vfofm_enable_timing(qdsp_vfofm* h, int on);
double qdsp_vfofm_kernel_ms(qdsp_vfofm* h);
/* per-launch timing of a whole timed region without a synchronisation, or any stream operation, between launches: the
 * row-per-lane kernel writes %globaltimer stamps (first CTA start, last CTA end) into one of `pairs` slots per launch, for
 * the first `pairs` launches since enable; kernel_ms_mean() synchronises and returns the mean completion-to-completion time
 * of those launches (the first one: start to end), which for launches that do not overlap equals an event pair around
 * each. Calls that take another kernel are not recorded. enable_timing() turns the ring off. */
int qdsp_vfofm_enable_timing_ring(qdsp_vfofm* h, int pairs);
double qdsp_vfofm_kernel_ms_mean(qdsp_vfofm* h, int* launches);

/* ---- channelizer: nch x [VFO -> FloatFMDemod] off one Splitter (routing.h:47-57) ------------ */
typedef struct qdsp_channelizer qdsp_channelizer;
qdsp_channelizer* qdsp_channelizer_create(int nch, const float* offsets, float inSampleRate, float outSampleRate,
                                          float bandWidth, float deviation);
void qdsp_channelizer_destroy(qdsp_channelizer* h);
int qdsp_channelizer_design(qdsp_channelizer* h, int* tapCount, int* interp, int* decim);
/* audio_out_dev is [nch][out_stride] floats; returns outputs per channel */
long long qdsp_channelizer_process(qdsp_channelizer* h, const void* in_dev, float* audio_out_dev,
                                   long long out_stride, long long count, const int* blocks, int nblocks,
                                   int block_size, qdsp_stream_t s);
int qdsp_channelizer_reset(qdsp_channelizer* h);
/* as qdsp_vfofm_set_input_format */
int qdsp_channelizer_set_input_format(qdsp_channelizer* h, int fmt, float scale, float offset);
/* variant 0: the fastest path the geometry allows (a uniform comb of 256 channels fs / 256 apart with decimation 1280 --
 * BASELINE config 4 -- takes the FFT polyphase kernels, k_chanfft.cu); 2: direct form (every channel its own VFO) always;
 * 1: the generic kernels. */
int qdsp_channelizer_set_variant(qdsp_channelizer* h, int variant);
/* Time-sharding: the next call's first sample is sample `start` of the stream (the NCOs are closed-form in the position).
 * A shard that starts mid-stream is fed max(history, decimation) extra samples ahead of its first wanted output and drops
 * the outputs those produce (bench.py config 4 at N > 1). Extension: the reference's state is implicit in its run() order. */
int qdsp_channelizer_seek(qdsp_channelizer* h, long long start);

/* ---- power spectrum: Welch-averaged FFT rows of a cf32 stream (an addition: the reference computes no spectrum) ---- *
 * Frame f covers stream samples [f hop, f hop + N) (sample 0 = the first after create or reset; samples in a gap between *
 * frames are never read); P_f[k] = |sum_n w[n] x[f hop + n] e^{-2 pi i k n / N}|^2. Row r is the mean of P over frames   *
 * r A .. r A + A - 1, FFT-shifted (out[j] = mean P[(j + N / 2) mod N]: bin 0 of a row is -fs / 2), linear power, float32. *
 * A row is a pure function of the stream: any split into calls gives the same bits. N a power of two in [64, 16384],     *
 * window N floats (NULL = rectangular), hop >= 1, average >= 1; create returns NULL on anything else. process writes the  *
 * rows it completes contiguously (N floats each) and returns their number, -1 for a negative count or in_dev not 8-byte  *
 * aligned; samples of rows not yet complete stay in the handle. out_rows: rows the next call of `count` samples returns.*/
typedef struct qdsp_spectrum qdsp_spectrum;
qdsp_spectrum* qdsp_spectrum_create(int fftSize, const float* window, int hop, int average);
void qdsp_spectrum_destroy(qdsp_spectrum* h);
long long qdsp_spectrum_out_rows(qdsp_spectrum* h, long long count);
long long qdsp_spectrum_process(qdsp_spectrum* h, const void* in_dev, float* rows_out_dev, long long count, qdsp_stream_t s);
int qdsp_spectrum_reset(qdsp_spectrum* h);

/* ---- recurrent blocks (chunked block-parallel scans) ----------------------------------------- */
/* BFMDeemp::run, src/dsp/filter.h:129-158 (stereo_t in/out, state lastOutL/R) */
typedef struct qdsp_deemp qdsp_deemp;
qdsp_deemp* qdsp_deemp_create(float sampleRate, float tau);
void qdsp_deemp_destroy(qdsp_deemp* h);
long long qdsp_deemp_process(qdsp_deemp* h, const void* in_dev, void* out_dev, long long count, qdsp_stream_t s);
int qdsp_deemp_set_params(qdsp_deemp* h, float sampleRate, float tau);       /* setSampleRate / setTau, filter.h:117-127: scalars only, state survives */
int qdsp_deemp_get_state(qdsp_deemp* h, float* lastL, float* lastR);
int qdsp_deemp_set_state(qdsp_deemp* h, float lastL, float lastR);

/* AGC::run, src/dsp/processing.h:119-134 (per-block decay, block max, scale) */
typedef struct qdsp_agc qdsp_agc;
qdsp_agc* qdsp_agc_create(float fallRate, float sampleRate);
void qdsp_agc_destroy(qdsp_agc* h);
long long qdsp_agc_process(qdsp_agc* h, const float* in_dev, float* out_dev, long long count, const int* blocks,
                           int nblocks, int block_size, qdsp_stream_t s);
int qdsp_agc_set_params(qdsp_agc* h, float fallRate, float sampleRate);      /* processing.h:101-113 */
int qdsp_agc_get_state(qdsp_agc* h, float* level);
int qdsp_agc_set_state(qdsp_agc* h, float level);

/* ComplexAGC::run, src/dsp/processing.h:271-286 */
typedef struct qdsp_cagc qdsp_cagc;
qdsp_cagc* qdsp_cagc_create(float setPoint, float maxGain, float rate);
void qdsp_cagc_destroy(qdsp_cagc* h);
long long qdsp_cagc_process(qdsp_cagc* h, const void* in_dev, void* out_dev, long long count, qdsp_stream_t s);
int qdsp_cagc_set_params(qdsp_cagc* h, float setPoint, float maxGain, float rate); /* processing.h:258-269 */
int qdsp_cagc_get_state(qdsp_cagc* h, float* gain);
int qdsp_cagc_set_state(qdsp_cagc* h, float gain);

/* FeedForwardAGC<complex_t>::run, src/dsp/processing.h:175-223; returns valid outputs (toProcess) */
typedef struct qdsp_ffagc qdsp_ffagc;
qdsp_ffagc* qdsp_ffagc_create(int dtype);
void qdsp_ffagc_destroy(qdsp_ffagc* h);
long long qdsp_ffagc_process(qdsp_ffagc* h, const void* in_dev, void* out_dev, long long count, qdsp_stream_t s);

/* CostasLoop<ORDER>::run, src/dsp/pll.h:47-102; state = {vcoFrequency, vcoPhase, lastVCO.re, lastVCO.im} */
typedef struct qdsp_costas qdsp_costas;
qdsp_costas* qdsp_costas_create(int order, float loopBandwidth);
void qdsp_costas_destroy(qdsp_costas* h);
long long qdsp_costas_process(qdsp_costas* h, const void* in_dev, void* out_dev, long long count, qdsp_stream_t s);
int qdsp_costas_get_state(qdsp_costas* h, float state[4]);
int qdsp_costas_set_state(qdsp_costas* h, const float state[4]);
/* chunk length / warm-up of the block-parallel scan (0,0 = strictly sequential single thread);
 * after a process call, max boundary phase residual (validity check of the stitched scan) */
int qdsp_costas_set_chunking(qdsp_costas* h, int chunk, int warmup);
float qdsp_costas_last_residual(qdsp_costas* h);

/* ---- element-wise, layout and per-block-statistic blocks ("next" rows of the scope table) ------------------- *
 * Each call replaces one run() body; two-input blocks require equal counts (the reference drops mismatched      *
 * blocks, math.h:26-30).                                                                                        */
enum { QDSP_MATH_ADD = 0, QDSP_MATH_SUB = 1, QDSP_MATH_MUL = 2 };
/* Add<T> / Substract<T> / Multiply<T>::run, src/dsp/math.h:21-43 / 68-90 / 115-137 (dtype QDSP_CF32 = complex_t or
 * stereo_t; Multiply on QDSP_CF32 is the complex product of volk_32fc_x2_multiply_32fc) */
long long qdsp_math_process(int op, int dtype, const void* a_dev, const void* b_dev, void* out_dev, long long count,
                            qdsp_stream_t s);
enum {
    QDSP_LAYOUT_MONO_TO_STEREO = 0,     /* MonoToStereo::run, audio.h:26-35: float -> stereo_t {x, x}                 */
    QDSP_LAYOUT_CHANNELS_TO_STEREO = 1, /* ChannelsToStereo::run, audio.h:70-86: in0 = left, in1 = right            */
    QDSP_LAYOUT_STEREO_TO_MONO = 2,     /* StereoToMono::run, audio.h:125-137: (l + r) * 0.5f                        */
    QDSP_LAYOUT_STEREO_TO_CHANNELS = 3, /* StereoToChannels::run, audio.h:169-179: out0 = left, out1 = right        */
    QDSP_LAYOUT_COMPLEX_TO_STEREO = 4,  /* ComplexToStereo::run, convertion.h:28-37 (a copy)                         */
    QDSP_LAYOUT_COMPLEX_TO_REAL = 5,    /* ComplexToReal::run, convertion.h:67-76                                    */
    QDSP_LAYOUT_COMPLEX_TO_IMAG = 6,    /* ComplexToImag::run, convertion.h:106-115                                  */
    QDSP_LAYOUT_REAL_TO_COMPLEX = 7     /* RealToComplex::run, convertion.h:153-162: {x, 0}                          */
};
long long qdsp_layout_process(int op, const void* in0_dev, const void* in1_dev, void* out0_dev, void* out1_dev,
                              long long count, qdsp_stream_t s);
/* Volume<float|stereo_t>::run, src/dsp/processing.h:388-411; level = qdsp_volume_level(volume) = powf(volume, 2)
 * (setVolume, :371-374 -- note that the reference's init() leaves level at 1.0 until setVolume is called) */
float qdsp_volume_level(float volume);
long long qdsp_volume_process(int dtype, float level, int muted, const void* in_dev, void* out_dev, long long count,
                              qdsp_stream_t s);
/* Threshold::run, src/dsp/processing.h:589-599: out[i] = in[i] > 0 (uint8) */
long long qdsp_threshold_process(const float* in_dev, unsigned char* out_dev, long long count, qdsp_stream_t s);
/* DelayImag::run, src/dsp/processing.h:321-337: out[i] = {in[i].re, in[i-1].im}; state lastIm */
typedef struct qdsp_delayimag qdsp_delayimag;
qdsp_delayimag* qdsp_delayimag_create(void);
void qdsp_delayimag_destroy(qdsp_delayimag* h);
long long qdsp_delayimag_process(qdsp_delayimag* h, const void* in_dev, void* out_dev, long long count, qdsp_stream_t s);
int qdsp_delayimag_get_state(qdsp_delayimag* h, float* lastIm);
int qdsp_delayimag_set_state(qdsp_delayimag* h, float lastIm);
/* AMDemod::run, src/dsp/demodulator.h:355-374: magnitude minus the mean magnitude of the run() block (so the
 * partition matters); the mean is summed in double here, sequentially in float by the reference */
typedef struct qdsp_amdemod qdsp_amdemod;
qdsp_amdemod* qdsp_amdemod_create(void);
void qdsp_amdemod_destroy(qdsp_amdemod* h);
long long qdsp_amdemod_process(qdsp_amdemod* h, const void* in_dev, float* out_dev, long long count, const int* blocks,
                               int nblocks, int block_size, qdsp_stream_t s);
/* Squelch::run, src/dsp/processing.h:460-479: a run() block passes iff 10*log10f(mean |x|) >= level, else zeros */
typedef struct qdsp_squelch qdsp_squelch;
qdsp_squelch* qdsp_squelch_create(float level);
void qdsp_squelch_destroy(qdsp_squelch* h);
void qdsp_squelch_set_level(qdsp_squelch* h, float level);
float qdsp_squelch_get_level(qdsp_squelch* h);
long long qdsp_squelch_process(qdsp_squelch* h, const void* in_dev, void* out_dev, long long count, const int* blocks,
                               int nblocks, int block_size, qdsp_stream_t s);
/* SSBDemod::run, src/dsp/demodulator.h:475-487: VOLK rotator by +-pi*bandWidth/sampleRate per sample (USB / LSB; DSB
 * does not rotate), then the real part; the NCO is the closed form used by the translator */
enum { QDSP_SSB_USB = 0, QDSP_SSB_LSB = 1, QDSP_SSB_DSB = 2 };   /* SSBDemod::MODE_*, demodulator.h:391-395 */
typedef struct qdsp_ssbdemod qdsp_ssbdemod;
qdsp_ssbdemod* qdsp_ssbdemod_create(float sampleRate, float bandWidth, int mode);
void qdsp_ssbdemod_destroy(qdsp_ssbdemod* h);
int qdsp_ssbdemod_configure(qdsp_ssbdemod* h, float sampleRate, float bandWidth, int mode);   /* setSampleRate / setBandWidth / setMode */
void qdsp_ssbdemod_get_phase_delta(qdsp_ssbdemod* h, float* re, float* im);
void qdsp_ssbdemod_get_phase(qdsp_ssbdemod* h, float* re, float* im);
void qdsp_ssbdemod_set_phase(qdsp_ssbdemod* h, float re, float im);
long long qdsp_ssbdemod_process(qdsp_ssbdemod* h, const void* in_dev, float* out_dev, long long count, qdsp_stream_t s);

/* ---- MMClockRecovery<float | complex_t>::run, src/dsp/clock_recovery.h:127-215 ("next" row) ------------------ *
 * Symbol-timing recovery: out_dev receives the recovered symbols (at most qdsp_mm_max_out(count) of them), the     *
 * return value is their number (data dependent, so this call waits for the kernel; out_counts, optional, gets the *
 * per-run()-block counts the reference passes to out.swap()). `interp_taps` is the caller's INTERP_TAPS[129][8]    *
 * (src/dsp/interpolation_taps.h:6-136, a baked MMSE table this library does not reproduce). The reference leaves  *
 * its delay buffer uninitialised for the first block (:218); here that history is zeros.                          */
typedef struct qdsp_mm qdsp_mm;
qdsp_mm* qdsp_mm_create(int dtype, float omega, float gainOmega, float muGain, float omegaRelLimit,
                        const float* interp_taps);
void qdsp_mm_destroy(qdsp_mm* h);
int qdsp_mm_set_omega(qdsp_mm* h, float omega, float omegaRelLimit);           /* setOmega, :90-97 (quirk kept)    */
int qdsp_mm_set_gains(qdsp_mm* h, float gainOmega, float muGain);              /* setGains, :99-104                */
int qdsp_mm_set_omega_rel_limit(qdsp_mm* h, float omegaRelLimit);              /* setOmegaRelLimit, :106-112       */
long long qdsp_mm_max_out(qdsp_mm* h, long long count);
long long qdsp_mm_process(qdsp_mm* h, const void* in_dev, void* out_dev, long long count, const int* blocks, int nblocks,
                          int block_size, int* out_counts, qdsp_stream_t s);
/* state[44]: mu, dynOmega, lastOutput, p_0T p_1T p_2T, c_0T c_1T c_2T, nextOffset, delay[0..6] (re, im pairs) */
int qdsp_mm_get_state(qdsp_mm* h, float state[44]);
int qdsp_mm_set_state(qdsp_mm* h, const float state[44]);

/* SineSource::run, src/dsp/source.h:55-59: the VOLK rotator over a buffer of ones, i.e. the NCO phasor itself
 * (closed form here); one call produces one block of `count` samples */
typedef struct qdsp_sinesource qdsp_sinesource;
qdsp_sinesource* qdsp_sinesource_create(float sampleRate, float freq);
void qdsp_sinesource_destroy(qdsp_sinesource* h);
int qdsp_sinesource_configure(qdsp_sinesource* h, float sampleRate, float freq);   /* setSampleRate / setFrequency */
void qdsp_sinesource_get_phase(qdsp_sinesource* h, float* re, float* im);
void qdsp_sinesource_set_phase(qdsp_sinesource* h, float re, float im);
long long qdsp_sinesource_process(qdsp_sinesource* h, void* out_dev, long long count, qdsp_stream_t s);

/* ---- device-side synthetic IQ (bench inputs; same integer recipe as qdsp_b200/synth.py) ------ */
int qdsp_synth_uniform_cf32(void* out_dev, unsigned long long seed, long long start, long long count, qdsp_stream_t s);
int qdsp_synth_fm_cf32(void* out_dev, long long start, long long count, long long fs, long long fc, long long fm,
                       double dev, double amp, double noise_amp, unsigned long long noise_seed, qdsp_stream_t s);
/* config 4's wideband comb (nch FM carriers `spacing` Hz apart, fm = 300 + 10k Hz) and config 5's QPSK streams; float32
 * evaluation of exact integer phase fractions -- test signals, the oracle consumes the generated samples themselves */
int qdsp_synth_comb_cf32(void* out_dev, long long start, long long count, long long fs, int nch, long long spacing,
                         double dev, double amp, double noise_amp, unsigned long long noise_seed, qdsp_stream_t s);
int qdsp_synth_qpsk_cf32(void* out_dev, long long start, long long count, unsigned long long seed, int sps, double freq_off,
                         double sigma, double am_depth, long long am_period, qdsp_stream_t s);

/* ---- microbenchmarks used by bench.py to measure the FP32 roofline denominator -------------- */
/* runs `iters` dependent-chain FMA iterations on every SM; returns achieved TFLOP/s (2 flop/FMA) */
double qdsp_measure_fp32_peak(int packed /*0: FFMA, 1: FFMA2*/, int iters);

#ifdef __cplusplus
}
#endif
#endif /* QDSP_B200_H */
