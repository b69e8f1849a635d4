// qdsp_b200/csrc/kernels.cuh — host-side launchers of every kernel family (defined in k_*.cu).
#pragma once
#include "internal.cuh"

namespace qdsp {

// Per-channel NCO constants on the device: phase(n_abs) = init + step * n_abs (turns * 2^64).
struct NcoDev {
    uint64_t init;
    uint64_t step;
};

// ---- k_generic.cu -------------------------------------------------------------------------------
template <typename T>
int launch_generic_resamp(const T* hist, int H, const T* in, const float* phases_dev, int TPP, int lead,
                          const Partition& part, T* out, cudaStream_t s);
int launch_schedule(const Partition& part, int* phase_dev, long long* index_dev, cudaStream_t s);
// nch channels (grid.z); audio is [nch][out_stride], iq optional [nch][out_stride];
// demod_state is [2][nch] ping-pong (read slot `st_in`, write the other).
int launch_generic_vfofm(const float2* hist, int H, const float2* in, const float* phases_dev, int TPP,
                         const Partition& part, const NcoDev* nco, long long abs0, int nch, float phasor_speed,
                         const float* demod_in, float* demod_out, float* audio, float2* iq, long long out_stride,
                         cudaStream_t s);

// ---- k_elementwise.cu ---------------------------------------------------------------------------
int launch_xlator(const float2* in, float2* out, long long count, uint64_t phase0, uint64_t step, float2 inc1,
                  float2 inc2, float2 inc3, cudaStream_t s);
int launch_xlator_replay(const float2* in, float2* out, const Partition& part, const long long* run0_dev,
                         const float2* ckpt_dev, float2 inc, long long nruns, cudaStream_t s);
int launch_fmdemod(const float2* in, void* out, long long count, float phasor_speed, const float* state_in,
                   float* state_out, int stereo, cudaStream_t s);
int launch_stereo_matrix(const float* mpx, const float* pilot, float2* out, long long count, cudaStream_t s);
int launch_power_decim(const float2* in, float2* out, long long n_out, int copy_only, cudaStream_t s);
int launch_synth_uniform(float2* out, unsigned long long seed, long long start, long long count, cudaStream_t s);
int launch_synth_fm(float2* out, long long start, long long count, long long fs, long long fc, long long fm,
                    double dev, double amp, double noise_amp, unsigned long long noise_seed, cudaStream_t s);
int launch_synth_comb(float2* out, long long start, long long count, long long fs, int nch, long long spacing, double dev,
                      double amp, double noise_amp, unsigned long long noise_seed, cudaStream_t s);
int launch_synth_qpsk(float2* out, long long start, long long count, unsigned long long seed, int sps, double freq_off,
                      double sigma, double am_depth, long long am_period, cudaStream_t s);
double run_fp32_peak(int packed, int iters);

// ---- k_decim.cu: column-parallel decimating FIR (I = 1, even D), optional NCO + FM demod --------
struct DecimPlan;  // opaque, owned by the handle
DecimPlan* decim_plan_create(const float* taps, int T, int D);
void decim_plan_destroy(DecimPlan* p);
bool decim_plan_supported(int T, int interp, int decim);
// mode: 0 = cf32 resampler output; 1 = fused NCO prologue + FM demod epilogue (audio [+ iq])
int launch_decim(DecimPlan* plan, const float2* hist, int H, const float2* in, const Partition& part, int mode,
                 const NcoDev* nco, long long abs0, int nch, float phasor_speed, const float* demod_in,
                 float* demod_out, float2* out_iq, float* audio, long long out_stride, cudaStream_t s);

// ---- k_rowlane.cu: row-per-lane decimating FIR (narrow rows, one channel), folds the history advance ----
bool rowlane_supported(const DecimPlan* plan);
int rowlane_uniform_pad(const Partition& part, int T);
int launch_decim_rowlane(DecimPlan* plan, const float* taps_host, const float2* hist, float2* hist_next, int H,
                         const float2* in, const Partition& part, int mode, const NcoDev* nco_dev, const NcoDev* nco_host,
                         long long abs0, float phasor_speed, const float* demod_in, float* demod_out, float2* out_iq,
                         float* audio, int pad, cudaStream_t s, bool overlap_prev, unsigned long long* tstamp);

// ---- k_chan.cu: channel-per-lane decimating FIR (wide rows, many channels off one input) --------------------
bool chan_supported(const DecimPlan* plan);
void chan_plan_released(const DecimPlan* plan);
int launch_chan(DecimPlan* plan, const float* taps_host, const float2* hist, int H, const float2* in, const Partition& part,
                int mode, const NcoDev* nco_dev, long long abs0, int nch, float phasor_speed, const float* demod_in,
                float* demod_out, float2* out_iq, float* audio, long long out_stride, int pad, cudaStream_t s);
int launch_decim_finish(const float2* ypart, long long ypart_stride, int nslices, long long total_out, int demod,
                        float phasor_speed, const float* demod_in, float* demod_out, float2* out_iq, float* audio,
                        long long out_stride, int nch, cudaStream_t s);

// ---- k_chanfft.cu: FFT polyphase channelizer (256 channels on a uniform fs/256 comb, decimation 1280) ---------------
struct ChanFftPlan;
// nco_phases: the channels' closed-form phase constants (NULL: all equal); channel k's difference to channel 0's goes into
// its epilogue constant, so the kernels take only channel 0's phase. nullptr when the steps do not form the comb, or when
// a device allocation failed: then *failed (if given) is set, and qdsp_last_error says why
ChanFftPlan* chanfft_plan_create(const float* taps, int T, int interp, int decim, int nch, const uint64_t* nco_steps,
                                 const uint64_t* nco_phases = nullptr, bool* failed = nullptr);
void chanfft_plan_destroy(ChanFftPlan* p);
// hand `from`'s U / V scratch (grown to the largest call) to `to`, which has none yet: a retune keeps it
void chanfft_plan_take_scratch(ChanFftPlan* to, ChanFftPlan* from);
bool chanfft_usable(const ChanFftPlan* p, const Partition& part, const void* in);
int launch_chanfft(ChanFftPlan* plan, const float2* hist, int H, const float2* in, const Partition& part, uint64_t beta_step,
                   uint64_t beta_ph0, long long abs0, float phasor_speed, const float* demod_in, float* demod_out, float* audio,
                   float2* iq, long long out_stride, cudaStream_t s);

// ---- k_spectrum.cu: Welch power spectrum (windowed N-point FFT frames, |X|^2 averaged per row, FFT-shifted) --------------
struct SpectrumPlan;
SpectrumPlan* spectrum_plan_create(int N, const float* window, int hop, int average);   // parameters checked by the caller
void spectrum_plan_destroy(SpectrumPlan* p);
void spectrum_plan_reset(SpectrumPlan* p);
long long spectrum_out_rows(const SpectrumPlan* p, long long count);
// false where integer input is converted to cf32 by launch_iq_convert before launch_spectrum instead of being read by the
// frames kernel (N = 16384 with hop <= N)
bool spectrum_native_integer(const SpectrumPlan* p);
// `in`: cf32 (fmt QDSP_CF32, 8-byte aligned) or integer pairs (QDSP_CS16 / QDSP_CS8 / QDSP_CU8, converted by `conv`,
// aligned to the pair); returns the rows written to rows_out ([rows][N]) or -1
long long launch_spectrum(SpectrumPlan* p, const void* in, int fmt, IqConv conv, float* rows_out, long long count,
                          cudaStream_t s);

// ---- k_fir.cu: register-blocked dense FIR (cf32, D = 1) -----------------------------------------
struct FirPlan;
FirPlan* fir_plan_create(const float* taps, int T);
void fir_plan_destroy(FirPlan* p);
int launch_fir_dense(FirPlan* plan, const float2* hist, int H, const float2* in, long long count, int lead,
                     float2* out, cudaStream_t s, float2* hist_next = nullptr, bool overlap_prev = false,
                     bool* advanced = nullptr);

// small-decimation FIR (interp = 1, 2 <= D <= 8): polyphase sub-streams through the dense inner loop
struct FirDecimPlan;
FirDecimPlan* fir_decim_plan_create(const float* taps, int T, int D);
void fir_decim_plan_destroy(FirDecimPlan* p);
int launch_fir_decim(FirDecimPlan* plan, const float2* hist, int H, const float2* in, long long count,
                     long long n_out, float2* out, cudaStream_t s);

// ---- k_firrow.cu: row-per-lane decimating FIR for small decimations (config 1b: D = 4, 127 taps) ------------------
bool firrow_supported(int T, int D);
int launch_firrow(const float* taps_host, int T, int D, const float2* hist, float2* hist_next, int H, const float2* in,
                  long long count, long long n_out, float2* out, cudaStream_t s, bool overlap_prev);

// ---- k_recurrent.cu -----------------------------------------------------------------------------
int launch_deemp(const float2* in, float2* out, long long count, float alpha, float* state, void* scratch,
                 size_t scratch_bytes, cudaStream_t s);
int agc_fused_chunk_blocks(const Partition& part, const float* in, const float* out);
size_t agc_fused_scratch_bytes(int cb);
int launch_agc_fused(const float* in, float* out, const Partition& part, float corrected_fall_rate, float* level_state, void* scratch,
                     int cb, cudaStream_t s);
int launch_agc(const float* in, float* out, const Partition& part, float corrected_fall_rate, float* level_state,
               float* blockmax_scratch, float* level_scratch, cudaStream_t s);
int launch_cagc(const float2* in, float2* out, long long count, float set_point, float max_gain, float rate,
                float* gain_state, void* scratch, size_t scratch_bytes, cudaStream_t s);
int launch_ffagc(const void* hist, int H, const void* in, void* out, long long n_valid, int is_complex,
                 cudaStream_t s);
int launch_costas(const float2* in, float2* out, long long count, int order, float alpha, float beta, float* state,
                  int chunk, int warmup, void* scratch, size_t scratch_bytes, float* residual_dev, cudaStream_t s);
size_t scan_scratch_bytes(long long count);
size_t costas_scratch_bytes(long long count, int chunk);

// ---- k_pointwise.cu: element-wise / layout / per-block-statistic blocks ---------------------------
int launch_math(int op, int complex_mul, const float* a, const float* b, float* out, long long nfloats, cudaStream_t s);
int launch_layout(int mode, const float* in0, const float* in1, float* out0, float* out1, long long count, cudaStream_t s);
int launch_scale(const float* in, float* out, long long nfloats, float level, cudaStream_t s);
int launch_threshold(const float* in, unsigned char* out, long long n, cudaStream_t s);
int launch_delay_imag(const float2* in, float2* out, long long count, const float* state_in, float* state_out,
                      cudaStream_t s);
size_t mag_scratch_bytes(int nblocks);
int launch_amdemod(const float2* in, float* out, const Partition& part, double* partial, cudaStream_t s);
int launch_squelch(const float2* in, float2* out, const Partition& part, double* partial, float level, cudaStream_t s);
int launch_sine(float2* out, long long count, uint64_t phase0, uint64_t step, float2 inc1, float2 inc2, float2 inc3,
                cudaStream_t s);
int launch_ssb(const float2* in, float* out, long long count, uint64_t phase0, uint64_t step, float2 inc1, float2 inc2,
               float2 inc3, cudaStream_t s);
// integer IQ (fmt QDSP_CS16 / QDSP_CS8 / QDSP_CU8, `in` aligned to its pair) -> cf32 (`out` 8-byte aligned)
int launch_iq_convert(int fmt, IqConv c, const void* in, float2* out, long long count, cudaStream_t s);

// ---- k_route.cu: row r of a planar [nrows][src_stride] buffer -> dst_table[r] (device table), elem_bytes 4 or 8 ----------
int launch_scatter_rows(const void* src, long long src_stride, void* const* dst_table, int nrows, long long count, int elem_bytes,
                        cudaStream_t s);

// ---- k_clock.cu: MMClockRecovery (sequential-exact, one warp per stream) --------------------------
int launch_mm(int cplx, const void* in, const Partition& part, const float* taps_dev, float omega, float gainOmega,
              float muGain, float omegaMin, float omegaMax, float* state, void* out, int* out_counts_dev,
              long long* total_dev, cudaStream_t s);

}  // namespace qdsp
