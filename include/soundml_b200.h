/* soundml_b200.h — C ABI of libsoundml_b200.so
 *
 * The B200-native replacement for the arithmetic under SoundML's spectral hot
 * path: framing -> window -> batched rFFT -> |X|^p -> mel projection, plus the
 * polyphase resampler / FIR.  Plain C: opaque plan handles, raw pointers and
 * sizes, int status codes.  This is exactly what the reference's OCaml layer
 * would bind through dune `foreign_stubs` (see INTEGRATION.md and ocaml/).
 *
 * Reference seams each entry point replaces (paths inside gabyfle/SoundML):
 *   smb_stft_*            Stft.Config.create / frames / transform /
 *                         power_spectrum    soundml/lib/stft.ml:61-111,217-223,
 *                                           632-666,670-691  (Nx.stft, Nx.magnitude)
 *   smb_mel_*             Mel.Config.create / filterbank / apply
 *                                           soundml/lib/mel.ml:119-164,198-231 (Nx.matmul)
 *   smb_mel_spectrogram   Soundml.mel_spectrogram   soundml/lib/soundml.ml:12-24
 *   smb_window_make       Window.make               soundml/lib/window.ml:374-401
 *   smb_resample_*        Resample.Config.create / output_frames / apply
 *                                           soundml/lib/resample.ml:872-1051,1913-1936
 *                         and the C executor it calls,
 *                         soundml_resample_step     soundml/lib/resample_stubs.c:232-297
 *   smb_fir_apply         the resampler's direct stage at L = M = 1
 *                         (SURVEY.md 8a "FIR note"; resample_stubs.c:127-143)
 *
 * Conventions
 *   - Tensors are C-contiguous, time axis last, leading axes flattened to
 *     `batch` (the reference flattens the same way: stft.ml:637, resample.ml:1921).
 *   - Spectral outputs are [batch, bins | n_mels, frames], frames contiguous.
 *   - `mem` says where x/out live: SMB_MEM_DEVICE pointers are used in place and
 *     the call only enqueues work on the plan's stream; SMB_MEM_HOST pointers
 *     (pageable or pinned) are staged through device buffers owned by the plan
 *     and the call returns after the result has landed in `out`.
 *   - Every function returns SMB_OK or an error code; smb_last_error() gives
 *     the message (thread-local).  SMB_EINVAL carries the reference's
 *     Invalid_argument wording; SMB_ECUDA is a runtime failure (OCaml Failure).
 *   - Plans are single-owner, like the reference's kernels ("not domain-safe",
 *     stft.mli:436-437): do not share one plan across threads.
 *   - There is no CPU fallback: compute entry points fail with SMB_ECUDA when
 *     no sm_100 device is usable.
 */
#ifndef SOUNDML_B200_H
#define SOUNDML_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { SMB_OK = 0, SMB_EINVAL = 1, SMB_ECUDA = 2, SMB_ENOMEM = 3 };
enum { SMB_MEM_DEVICE = 0, SMB_MEM_HOST = 1 };
enum { SMB_F32 = 0, SMB_F64 = 1 };

/* The stream a plan creates for itself (see smb_*_plan_set_stream). */
#define SMB_STREAM_OWN ((void*)(intptr_t)-1)

/* Omitted optional integer argument (OCaml ?hop, ?win_length). */
#define SMB_DEFAULT INT32_MIN

/* Window.t (window.ml:22-33); `param` is beta / std / taper where it applies. */
enum {
  SMB_WINDOW_HANN = 0, SMB_WINDOW_HAMMING, SMB_WINDOW_BLACKMAN,
  SMB_WINDOW_BLACKMAN_HARRIS, SMB_WINDOW_NUTTALL, SMB_WINDOW_BARTLETT,
  SMB_WINDOW_KAISER, SMB_WINDOW_GAUSSIAN, SMB_WINDOW_TUKEY, SMB_WINDOW_FLAT_TOP,
  SMB_WINDOW_RECTANGULAR
};
enum { SMB_ALIGN_CENTERED = 0, SMB_ALIGN_LEFT = 1, SMB_ALIGN_RIGHT = 2 };
enum { SMB_PAD_REFLECT = 0, SMB_PAD_CONSTANT = 1, SMB_PAD_EDGE = 2 };
enum { SMB_SCALE_NONE = 0, SMB_SCALE_MAGNITUDE = 1, SMB_SCALE_PSD = 2 };
enum { SMB_MEL_SLANEY = 0, SMB_MEL_HTK = 1 };
enum { SMB_NORM_SLANEY = 0, SMB_NORM_NONE = 1 };
enum { SMB_QUALITY_FAST = 0, SMB_QUALITY_HIGH = 1, SMB_QUALITY_BEST = 2, SMB_QUALITY_CUSTOM = 3 };
enum { SMB_EXEC_DIRECT = 0, SMB_EXEC_OLS = 1, SMB_EXEC_GEMM = 2, SMB_EXEC_PLANNED = 3 };
/* Kernel selection for the STFT family (testing / benchmarking): AUTO picks the
 * fused fft-2048 kernel when the geometry allows it, else the double-interior
 * generic kernel; FAST forces the fused CUDA-core kernel (register FFT), TENSOR the
 * fused tcgen05 kernel (both 32-point FFT passes as split-fp16 products in TMEM),
 * PAIR the frame-pair kernel (two frames per warp in float32x2 lanes; mel output of
 * fft 2048, what AUTO picks for smb_mel_spectrogram when it applies);
 * a forced kernel that does not cover the call is SMB_EINVAL.
 *
 * NUMERICAL CONTRACT.  The reference computes every float32 call in a double interior
 * and rounds once (stft.ml:61-142, mel.ml:202-231; its gate is per element, rtol 1e-6 /
 * atol 1e-7).  SMB_PATH_GENERIC does exactly that, at any size.  The fused kernels
 * (FAST, PAIR, TENSOR: what AUTO picks for float32 audio and fft_size in 128 .. 2048)
 * keep a FLOAT32 interior -- window, twiddles, mel weights and the transform itself
 * rounded to float32 -- and hold a weaker, peak-relative contract: every output is within
 * 1e-6 of its clip's largest output (measured 5e-7; tests gate 1e-4, the bar
 * BASELINE.json states for this path), so values more than ~120 dB below the clip's
 * peak are noise.  In decibels with the reference's default 80 dB floor that is within
 * 0.01 dB (tests/test_gpu_pair_kernel.py::test_high_dynamic_range_elementwise; log-mel
 * and MFCC through the fused path are gated on the reference's goldens and the oracle in
 * tests/test_gpu_db_mfcc.py).  smb_stft_invert's fused kernel likewise runs its
 * transforms in float32 but divides by the overlap envelope in double, including the
 * partially covered head and tail.  Float64 audio always takes the double interior.
 * A caller that needs the per-element contract forces SMB_PATH_GENERIC. */
enum { SMB_PATH_AUTO = 0, SMB_PATH_GENERIC = 1, SMB_PATH_FAST = 2, SMB_PATH_TENSOR = 3,
       SMB_PATH_PAIR = 4 };

typedef struct smb_stft_plan smb_stft_plan;
typedef struct smb_mel_plan smb_mel_plan;
typedef struct smb_resample_plan smb_resample_plan;
typedef struct smb_fir_plan smb_fir_plan;

const char* smb_last_error(void);
const char* smb_version(void);

/* ---- device and buffers ------------------------------------------------- */
int smb_device_count(int* count);
int smb_set_device(int device);
int smb_device_alloc(void** ptr, size_t bytes);
int smb_device_free(void* ptr);
int smb_host_alloc_pinned(void** ptr, size_t bytes);
int smb_host_free_pinned(void* ptr);
int smb_memcpy_h2d(void* dst_device, const void* src_host, size_t bytes);
int smb_memcpy_d2h(void* dst_host, const void* src_device, size_t bytes);
int smb_device_synchronize(void);
/* Number of kernels this library has launched in the calling process. */
int64_t smb_kernel_launch_count(void);

/* ---- host-side design (no GPU needed) ------------------------------------ */
/* Window.make Nx.float64 ~periodic kind n -> out[n]. */
int smb_window_make(int kind, double param, int periodic, int64_t n, double* out);

/* ---- STFT ---------------------------------------------------------------- */
/* Stft.Config.create ?window ?win_length ?hop ?alignment ?pad ?scale ~fft_size. */
int smb_stft_plan_create(smb_stft_plan** plan, int64_t fft_size, int64_t hop,
                         int64_t win_length, int window_kind, double window_param,
                         int alignment, int pad_kind, double pad_value, int scale);
/* Same, with the analysis window (fft_size doubles, already centred and
 * scaled) supplied by the caller — what an OCaml Stft.Config.t already holds. */
int smb_stft_plan_create_with_window(smb_stft_plan** plan, int64_t fft_size,
                                     int64_t hop, int alignment, int pad_kind,
                                     double pad_value, const double* analysis_window);
int smb_stft_plan_destroy(smb_stft_plan* plan);
/* Run this plan's kernels on an existing CUDA stream (cudaStream_t; NULL is the
 * CUDA default stream); SMB_STREAM_OWN restores the plan's own stream. */
int smb_stft_plan_set_stream(smb_stft_plan* plan, void* cuda_stream);
int smb_stft_plan_set_path(smb_stft_plan* plan, int path);
int smb_stft_plan_sync(smb_stft_plan* plan);
int64_t smb_stft_fft_size(const smb_stft_plan* plan);
int64_t smb_stft_hop(const smb_stft_plan* plan);
int64_t smb_stft_bins(const smb_stft_plan* plan);
/* Stft.frames c ~n; -1 and SMB_EINVAL message on n < 0. */
int64_t smb_stft_frames(const smb_stft_plan* plan, int64_t n);
int smb_stft_analysis_window(const smb_stft_plan* plan, double* out);
/* Source index each padded position reads (-1 = constant fill): the framing
 * contract of Stft.pad_signal, exposed so index parity can be checked bit for
 * bit.  out has n + left_width + right_width entries. */
int smb_stft_source_indices(const smb_stft_plan* plan, int64_t n, int64_t* out,
                            int64_t* padded_len);

/* Stft.transform: x [batch, n] (dtype) -> out [batch, bins, frames] complex
 * (interleaved re, im; complex64 for SMB_F32, complex128 for SMB_F64). */
int smb_stft_transform(smb_stft_plan* plan, const void* x, int64_t batch, int64_t n,
                       int dtype, void* out, int mem);
/* Stft.transform_range ~p0 ~p1 (stft.ml:652-666): frames [p0, p1) of the full
 * transform without evaluating the others; out [batch, bins, p1 - p0] complex.
 * Adjacent ranges reassemble the full transform exactly. */
int smb_stft_transform_range(smb_stft_plan* plan, const void* x, int64_t batch, int64_t n,
                             int dtype, int64_t p0, int64_t p1, void* out, int mem);
/* Stft.power_spectrum ?power: out [batch, bins, frames] real. */
int smb_stft_power_spectrum(smb_stft_plan* plan, const void* x, int64_t batch,
                            int64_t n, int dtype, double power, void* out, int mem);

/* Least-squares synthesis, Stft.invert dtype c ?length z (stft.ml:693-939).
 * smb_stft_nola: 1 when the overlap-added squared window stays above 1e-10 of
 * its maximum (stft.ml:731-742), else 0.  smb_stft_output_length: the length
 * synthesis returns for `frames` frames when none is named (stft.ml:790-794),
 * -1 on error.  smb_stft_invert: z [batch, bins, frames] complex (in_dtype
 * SMB_F32 = complex64, SMB_F64 = complex128) -> out [batch, length] real
 * (out_dtype); has_length = 0 takes the natural length.  Interior in double,
 * one rounding into out_dtype.  Fails with the reference's messages for a
 * non-invertible configuration or a negative length. */
int smb_stft_nola(const smb_stft_plan* plan);
int64_t smb_stft_output_length(const smb_stft_plan* plan, int64_t frames);
int smb_stft_invert(smb_stft_plan* plan, const void* z, int64_t batch, int64_t frames,
                    int in_dtype, int has_length, int64_t length, int out_dtype, void* out,
                    int mem);

/* Stft.griffin_lim ?n_iter ?momentum ?init ?length c s (stft.ml:964-1025): fast
 * Griffin-Lim phase reconstruction.  s [batch, bins, frames] magnitudes (dtype);
 * init_phase NULL (`Zero_phase) or phases of the same shape and dtype; the loop
 * runs in complex128 at the natural synthesis length on the device, the result
 * out [batch, length] is rounded into dtype. */
int smb_stft_griffin_lim(smb_stft_plan* plan, const void* s, int64_t batch, int64_t frames,
                         int dtype, int64_t n_iter, double momentum, const void* init_phase,
                         int has_length, int64_t length, void* out, int mem);

/* ---- mel ----------------------------------------------------------------- */
/* Mel.Config.create; f_max = NaN means "Nyquist" (the OCaml default). */
int smb_mel_plan_create(smb_mel_plan** plan, int64_t n_mels, int64_t sample_rate,
                        int64_t fft_size, double f_min, double f_max, int scale,
                        int norm);
/* Same, with the [n_mels, bins] float64 weights supplied by the caller. */
int smb_mel_plan_create_with_weights(smb_mel_plan** plan, int64_t n_mels,
                                     int64_t fft_size, const double* weights);
int smb_mel_plan_destroy(smb_mel_plan* plan);
int smb_mel_plan_set_stream(smb_mel_plan* plan, void* cuda_stream);
int64_t smb_mel_n_mels(const smb_mel_plan* plan);
int64_t smb_mel_bins(const smb_mel_plan* plan);
int64_t smb_mel_fft_size(const smb_mel_plan* plan);   /* as given at creation (odd sizes too) */
/* Mel.filterbank Nx.float64: out [n_mels, bins]. */
int smb_mel_filterbank(const smb_mel_plan* plan, double* out);
/* Mel.apply: s [batch, bins, frames] -> out [batch, n_mels, frames]. */
int smb_mel_apply(smb_mel_plan* plan, const void* s, int64_t batch, int64_t frames,
                  int dtype, void* out, int mem);
/* Soundml.mel_spectrogram stft mel ?power x: x [batch, n] ->
 * out [batch, n_mels, frames].  The power spectrogram never reaches HBM on the
 * fused path. */
int smb_mel_spectrogram(smb_stft_plan* stft, smb_mel_plan* mel, const void* x,
                        int64_t batch, int64_t n, int dtype, double power, void* out,
                        int mem);
/* Measurement hook, not part of the drop-in surface: the transform alone on the
 * frame-pair kernel's skeleton (staging, window, both FFT passes, transposition; no
 * split, no |X|^2, no mel).  bench.py reports its time as roofline.compute_floor_ms.
 * x: device float32 [batch, n]; scratch: device, ..._scratch_bytes() bytes. */
int64_t smb_stft_fft_ceiling_scratch_bytes(const smb_stft_plan* plan, int64_t batch, int64_t n);
int smb_stft_fft_ceiling(smb_stft_plan* stft, const void* x, int64_t batch, int64_t n, void* scratch);

/* ---- dB conversion and MFCC (SURVEY.md 8f, rank 1) ------------------------- */
/* Convert.power_to_db / amplitude_to_db ?reference ?amin ?top_db (convert.ml:20-56):
 * elementwise over `count` values in the input's dtype; top_db = NaN means "no
 * clamp", otherwise the clamp sits top_db below the maximum of the whole tensor.
 * Runs on `cuda_stream` (NULL or SMB_STREAM_OWN = the default stream): a host-memory
 * call returns when the result is in `out`, a device-memory call is asynchronous on the
 * stream like every other device-memory entry (no hidden synchronisation). */
int smb_power_to_db(const void* x, int64_t count, int dtype, double reference, double amin,
                    double top_db, void* out, int mem, void* cuda_stream);
int smb_amplitude_to_db(const void* x, int64_t count, int dtype, double reference, double amin,
                        double top_db, void* out, int mem, void* cuda_stream);
/* Soundml.mfcc stft mel ?n_mfcc ?lifter x (soundml.ml:50-95): x [batch, n] ->
 * out [batch, n_mfcc, frames]; lifter = NaN or 0 means none.  Log-mel with the
 * 80 dB clamp below the whole-tensor maximum, orthonormal DCT-II, in double. */
int smb_mfcc(smb_stft_plan* stft, smb_mel_plan* mel, const void* x, int64_t batch, int64_t n,
             int dtype, int64_t n_mfcc, double lifter, void* out, int mem);
/* Convert.power_to_db ?reference ?amin ?top_db (Soundml.mel_spectrogram ?power stft mel x)
 * (convert.ml:20-56 over soundml.ml:12-24) -- the log-mel spectrogram, in the input's
 * dtype, out [batch, n_mels, frames].  top_db = NaN means "no clamp".  For fft 2048
 * float32 the mel kernel leaves the whole-tensor maximum behind as it writes, so the
 * decibel map and its clamp are one pass in place: two launches.  Errors: the mel
 * spectrogram's, then power_to_db's, in the reference's wording. */
int smb_mel_spectrogram_db(smb_stft_plan* stft, smb_mel_plan* mel, const void* x, int64_t batch,
                           int64_t n, int dtype, double power, double reference, double amin,
                           double top_db, void* out, int mem);

/* ---- resampler ------------------------------------------------------------ */
/* Resample.Config.create ?quality ~sample_rate ~target; attenuation/passband
 * are read only for SMB_QUALITY_CUSTOM. */
int smb_resample_plan_create(smb_resample_plan** plan, int64_t sample_rate,
                             int64_t target, int quality, double attenuation,
                             double passband);
int smb_resample_plan_destroy(smb_resample_plan* plan);
int smb_resample_plan_set_stream(smb_resample_plan* plan, void* cuda_stream);
int smb_resample_plan_sync(smb_resample_plan* plan);
/* Which kernel runs the stages: SMB_EXEC_PLANNED (default) follows the planner's
 * tags -- overlap-save FFT blocks for "ols" stages (power-of-two lengths), the
 * tcgen05 banded product for "gemm" stages (L <= 1024; stages wider than 160
 * phases run as column groups of <= 160, one launch each), the direct polyphase
 * kernel for everything else; SMB_EXEC_DIRECT forces the direct kernel
 * everywhere.  Same designed filter either way. */
int smb_resample_plan_set_executor(smb_resample_plan* plan, int exec);
/* Which kernel smb_resample_apply runs for one stage (float32 audio), and how its
 * device tables are laid out.  Read-only; the device tables are built first if no
 * apply has built them yet, so the SMB_ROWS_* and SMB_GEMM_WINDOWS environment
 * switches set at that moment take effect, as they would for a first apply. */
enum { SMB_FORM_DIRECT = 0, SMB_FORM_OLS = 1, SMB_FORM_WINDOW = 2, SMB_FORM_ROW = 3 };
typedef struct smb_resample_layout {
  int form;          /* SMB_FORM_*: direct kernel, overlap-save, tcgen05 window or row form */
  int groups;        /* column groups (launches) of the stage's form; 1 for direct and OLS */
  int columns;       /* phases (output columns) of group `group` */
  int col_begin;     /* its first phase */
  /* row form only (0 otherwise; chunks is also set for the window form): */
  int two_issuers;   /* the main shift's small terms split off, two MMA-issuing threads */
  int a_tmem;        /* A tiles in tensor memory (else shared memory) */
  int a_stages, b_stages;
  int shifts;        /* input-row shifts, one accumulator each */
  int chunks;        /* K-chunks of 32 inputs per tile */
  int slices;        /* products per tile (runs of accumulator columns, times two for split runs) */
} smb_resample_layout;
int smb_resample_stage_layout(smb_resample_plan* plan, int stage, int group,
                              smb_resample_layout* out);
/* Config.pp one-liner, e.g. "resample(44100 -> 16000 Hz, quality=high, ...)". */
int smb_resample_describe(const smb_resample_plan* plan, char* buf, size_t cap);
int64_t smb_resample_l(const smb_resample_plan* plan);
int64_t smb_resample_m(const smb_resample_plan* plan);
int64_t smb_resample_latency(const smb_resample_plan* plan);
int smb_resample_num_stages(const smb_resample_plan* plan);
/* Stage i: factors, group delay K, executor tag, OLS geometry (0 if none). */
int smb_resample_stage_info(const smb_resample_plan* plan, int stage, int64_t* l,
                            int64_t* m, int64_t* k, int* exec, int64_t* ols_n,
                            int64_t* ols_b, int64_t* ols_delta);
/* Stage i design parameters: cutoff (Nyquist units of the interpolated rate)
 * and Kaiser beta handed to design_prototype (resample.ml:145-163). */
int smb_resample_stage_design(const smb_resample_plan* plan, int stage, double* fc,
                              double* beta);
/* Stage prototype (2*K*L + 1 doubles); returns the length through *len when
 * out is NULL. */
int smb_resample_stage_prototype(const smb_resample_plan* plan, int stage,
                                 double* out, int64_t* len);
/* Config.output_frames c ~n = ceil(n*L/M); -1 on error. */
int64_t smb_resample_output_frames(const smb_resample_plan* plan, int64_t n);
/* Resample.apply: x [batch, n] f32 -> out [batch, output_frames(n)] f32. */
int smb_resample_apply(smb_resample_plan* plan, const float* x, int64_t batch,
                       int64_t n, float* out, int mem);

/* Same for float64 audio (the reference carries both, resample.ml:72-84); runs
 * the direct polyphase kernel in double. */
int smb_resample_apply_f64(smb_resample_plan* plan, const double* x, int64_t batch,
                           int64_t n, double* out, int mem);

/* Resample.Kernel.prepare / step / flush / reset (resample.ml:1343-1424, 1844-1909): the
 * chunked form of apply, what soundml-io's decode loop (soundml_io.ml:639, 768, 798) and
 * cqt.ml:797-879 bind.  The carry (the input some future output still needs) lives in
 * device memory.  A chunk is [channels, n] C-contiguous, dtype SMB_F32 or SMB_F64 as given
 * at creation; step writes the samples that became computable, [channels, frames]
 * C-contiguous with frames = smb_resample_kernel_step_frames(kernel, n) asked BEFORE the
 * step (exact integer bookkeeping, may be 0); flush writes the delayed tail,
 * smb_resample_kernel_flush_frames frames; everything written concatenates to
 * smb_resample_apply's result on the concatenated input, ceil(n L / M) samples in all --
 * bit for bit with the direct executor, to rounding (<= 1e-5 of peak) with the block
 * executors.  Not thread-safe, single owner (resample.mli:271-273).  Errors carry the
 * reference's wording (SMB_EINVAL: channels / max_block < 1, chunk longer than max_block,
 * step after flush). */
typedef struct smb_resample_kernel smb_resample_kernel;
int smb_resample_kernel_create(smb_resample_kernel** kernel, smb_resample_plan* plan, int dtype,
                               int64_t channels, int64_t max_block);
int smb_resample_kernel_destroy(smb_resample_kernel* kernel);
int smb_resample_kernel_reset(smb_resample_kernel* kernel);
int64_t smb_resample_kernel_step_frames(const smb_resample_kernel* kernel, int64_t n);
int64_t smb_resample_kernel_flush_frames(const smb_resample_kernel* kernel);
int smb_resample_kernel_step(smb_resample_kernel* kernel, const void* chunk, int64_t n, void* out,
                             int mem);
int smb_resample_kernel_flush(smb_resample_kernel* kernel, void* out, int mem);

/* ---- FIR ------------------------------------------------------------------ */
/* y[c,i] = sum_t h[t] * x[c, i + (taps-1)/2 - t], zeros outside, taps odd.
 * method: SMB_EXEC_DIRECT, SMB_EXEC_OLS (overlap-save on the FFT kernels) or
 * SMB_EXEC_PLANNED (overlap-save from 17 taps up when the filter fits a block,
 * else direct -- the measured crossover on B200). */
int smb_fir_plan_create(smb_fir_plan** plan, const double* h, int64_t taps);
int smb_fir_plan_destroy(smb_fir_plan* plan);
int smb_fir_plan_set_stream(smb_fir_plan* plan, void* cuda_stream);
int smb_fir_apply(smb_fir_plan* plan, const float* x, int64_t batch, int64_t n,
                  float* out, int method, int mem);
/* Kaiser-windowed sinc lowpass, the resampler's design_prototype at L = 1
 * (resample.ml:145-163): taps = 2K+1, cutoff in Nyquist units. */
int smb_fir_design_lowpass(int64_t k, double cutoff, double attenuation, double* out);

/* ---- soundml-io device ingest (SURVEY.md 8f rank 3) -------------------------- */
/* The layout pass of soundml-io's decode path on the device: a decoded block,
 * interleaved [frames][channels] as sf_readf_float / sf_readf_double fill the
 * reference's staging block (soundml-io/lib/soundml_io_stubs.c:832-872,
 * soundml_io_read_planar_*), becomes planar -- channel c at out + c * out_total +
 * out_off -- or, with SMB_INGEST_DOWNMIX, one mono line at out + out_off (channels
 * added in order, one multiply by 1 / channels: the reference's arithmetic, bit for
 * bit).  mem_in / mem_out say where the block and the destination live
 * (SMB_MEM_HOST in + SMB_MEM_DEVICE out is the ingest direction: the block goes up
 * asynchronously on `cuda_stream` (NULL = default stream) and the call returns when
 * it has been consumed).  The result feeds Resample.Kernel.step on arrival, as
 * decode_step does (soundml-io/lib/soundml_io.ml:742-782). */
enum { SMB_INGEST_PLANAR = 1, SMB_INGEST_DOWNMIX = 2 };
int smb_ingest_layout(const void* interleaved, int64_t frames, int64_t channels, int mode,
                      int dtype, void* out, int64_t out_total, int64_t out_off,
                      int mem_in, int mem_out, void* cuda_stream);
/* decode_block_frames ~channels ~elt ~advertised (soundml_io.ml:532-536): frames
 * per decode block of the fused read. */
int64_t smb_ingest_block_frames(int64_t channels, int64_t elt, int64_t advertised);

/* The fused read's decode loop on the device (soundml_io.ml:742-807 decode_step /
 * resolve_eof; the staging block of soundml_io_stubs.c:1175-1239): two PINNED interleaved
 * staging blocks of max_block frames.  The decoder (sf_readf_* on the CPU) fills the block
 * smb_ingest_staging hands out; smb_ingest_submit(frames) only ENQUEUES -- the upload on a
 * copy stream, then, behind an event, the layout pass and the streaming resampler's step on
 * the compute stream, writing [width, released] C-contiguous straight into `out_device`
 * (width = channels, or 1 with SMB_INGEST_DOWNMIX) -- and flips to the other block, so block
 * i + 1 is being decoded while block i is uploaded and resampled.  `released` is integer
 * bookkeeping known beforehand: smb_ingest_submit_frames(frames), asked BEFORE the submit;
 * smb_ingest_finish writes the resampler's tail (smb_ingest_finish_frames) at decoder EOF.
 * target = 0 (or = sample_rate) delivers the native rate: submit is the layout pass alone.
 * smb_ingest_staging blocks only until the upload that last read that block (two submits
 * ago) has left the host.  max_block = 0 takes decode_block_frames' rule.  Everything
 * written concatenates to smb_resample_apply of the whole laid-out signal (bit for bit with
 * the direct executor, <= 1e-5 of peak with the block executors).  Single owner. */
typedef struct smb_ingest smb_ingest;
int smb_ingest_create(smb_ingest** reader, int64_t channels, int64_t sample_rate, int64_t target,
                      int mode, int quality, int64_t max_block, int dtype);
int smb_ingest_destroy(smb_ingest* reader);
int64_t smb_ingest_max_block(const smb_ingest* reader);
int smb_ingest_staging(smb_ingest* reader, void** block);
int64_t smb_ingest_submit_frames(const smb_ingest* reader, int64_t frames);
int smb_ingest_submit(smb_ingest* reader, int64_t frames, void* out_device);
int64_t smb_ingest_finish_frames(const smb_ingest* reader);
int smb_ingest_finish(smb_ingest* reader, void* out_device);
int smb_ingest_sync(smb_ingest* reader);
/* the compute stream (a cudaStream_t): what a consumer of out_device must order itself behind */
void* smb_ingest_stream(smb_ingest* reader);

#ifdef __cplusplus
}
#endif
#endif /* SOUNDML_B200_H */
