// Launch wrappers of the CUDA kernels (internal to the library).
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstdint>

namespace smb {

// How a frame reads the signal: padded position q <-> source index q - left,
// out-of-range indices resolved by `pad` (stft.ml:300-338).
struct FrameGeom {
  long long n;        // samples per signal
  long long frames;   // frames per signal
  int fft, hop, left, pad;
  double pad_value;
};

enum SpecMode { kModeComplex = 0, kModePower = 1 };

extern std::atomic<long long> g_launch_count;   // kernels launched by this library (plans may run on several host threads)

// ---- generic path: any fft size, float64 interior ---------------------------
// x [batch, n] (f32 or f64) -> out [batch, bins, frames]; complex mode writes
// interleaved (re, im) in the input's precision, power mode writes |X|^power.
// window: fft doubles on the device; twiddle: fft double2 (cos, -sin)(2 pi j / fft).
cudaError_t launch_stft_generic(const void* x, int dtype, long long batch, FrameGeom g,
                                const double* window, const double2* twiddle,
                                int mode, double power, void* out, cudaStream_t st);

// Mel.apply: s [batch, bins, frames] -> out [batch, n_mels, frames], float64
// accumulation over each filter's nonzero band [band_lo[m], band_hi[m]).
cudaError_t launch_mel_apply(const void* s, int dtype, long long batch, int bins,
                             long long frames, int n_mels, const double* weights,
                             const int* band_lo, const int* band_hi, void* out,
                             cudaStream_t st);

// ---- synthesis (istft_kernels.cu) ----------------------------------------------
struct IstftArgs {
  const void* z;            // [batch, bins, frames] complex (float2 or double2)
  void* out;                // [batch, out_len] real
  long long frames;         // frame axis of z
  long long count;          // frames that reach the output (<= frames)
  long long out_len;
  int fft, hop, left;
  const double* window;     // [fft] analysis window
  const double2* twiddle;   // exp(-2 pi i j / fft), j < fft
  const double* folded;     // [hop] overlap-added squared window per residue class
  int in_f64, out_f64;
};
cudaError_t launch_istft(const IstftArgs& a, long long batch, cudaStream_t st);
// Griffin-Lim: spec = mags * unit(rebuilt - beta * previous), or the initial spectrum
cudaError_t launch_gl_project(const void* mags, const void* phase, int dtype,
                              const double2* rebuilt, const double2* previous, double beta,
                              int first, long long count, double2* spec, cudaStream_t st);
// fft 2048, complex64 -> float32 on the register FFT (istft2048.cu)
bool istft2048_supports(const IstftArgs& a);
cudaError_t launch_istft2048(const IstftArgs& a, const float* window_scaled, const float2* tw_pass,
                             const float2* tw_base, long long batch, int sm_count,
                             cudaStream_t st);

// ---- phase vocoder (effects_kernels.cu) ------------------------------------------
// z [rows, frames] complex -> out [rows, out_frames] complex of the same width; output
// frame t reads source position t * rate (librosa 0.11 phase_vocoder, DESIGN.md 4.8).
struct PhaseVocoderArgs {
  const void* z;            // float2 or double2
  void* out;
  long long rows;           // batch * bins
  long long frames, out_frames;
  double rate;
  int f64;
};
cudaError_t launch_phase_vocoder(const PhaseVocoderArgs& a, cudaStream_t st);

// ---- harmonic-percussive separation (hpss_kernels.cu) ------------------------------
// s [batch, bins, frames] real or complex -> the masked spectra or the masks of librosa
// 0.11 decompose.hpss (DESIGN.md 4.9).  `what` is SMB_HPSS_*; out is [batch, 2 | 1, bins,
// frames], complex for complex input unless the masks are asked for.
struct HpssArgs {
  const void* s;
  void* out;
  long long batch, bins, frames;
  long long win_harm, win_perc;
  double power;             // > 0, +inf for the hard mask
  double margin_harm, margin_perc;
  int what;
  int f64, complex_in;
};
// The fused tile kernel keeps each window sorted in registers: it takes windows of up to
// kHpssFastWindow; the exact counting kernel takes the rest.
constexpr long long kHpssFastWindow = 32;
bool hpss_fast_supports(long long win_harm, long long win_perc);
cudaError_t launch_hpss(const HpssArgs& a, cudaStream_t st);

// ---- spectral descriptors (spectral_kernels.cu) ---------------------------------
// s [batch, bins, frames] real -> out [batch, popcount(what), frames] of s's type: the
// SMB_SPECTRAL_* rows of `what` in flag order (librosa 0.11; DESIGN.md 4.10).
struct SpectralArgs {
  const void* s;
  void* out;
  long long batch, bins, frames;
  double bin_hz;            // f_k = k * bin_hz
  int what;
  double p;                 // bandwidth: > 0, finite
  int norm;
  double roll_percent;      // in (0, 1)
  double amin, power;       // flatness: > 0
  int f64;
};
cudaError_t launch_spectral(const SpectralArgs& a, cudaStream_t st);

// ---- fast path: fft 2048, float32, fused frame+window+rFFT+|X|^p(+mel) -------
// Tile shape of the fused CUDA-core kernel: a group of kFastTile warps transforms
// kFastTile consecutive frames, one per warp.
constexpr int kFastTile = 8;
// One lane of a mel round of the fused kernels: a piece (a few float4 steps) of one
// filter's band, carried for all the frames of the tile.
struct MelPiece {
  int off;                 // weights: float offset of [step 0][lane] (low 24 bits), steps of the round (high 8)
  short lo;                // first bin read (multiple of 4)
  unsigned short pid;      // partial-sum slot j * mel_mpad + m (4 * mel_mpad = scratch)
};
constexpr int kFastPieceSteps = 3;     // float4 steps per piece, CUDA-core kernel (8 frames per lane)
constexpr int kTcPieceSteps = 4;       // tensor-core kernel (4 frames per lane)
enum FastOut { kFastComplex = 0, kFastPower = 1, kFastMel = 2 };
struct Stft2048Args {
  const float* x;          // [batch, n]
  float* out;              // [batch, bins | n_mels, frames] (float2 for complex)
  long long batch;
  FrameGeom g;
  const float* window;     // [2048]
  const float2* tw_pass;   // [32][32]  W_1024^(k1*n2), index k1*32 + n2
  const float2* tw_post;   // [16][32]  W_2048^(l + 32 j), index j*32 + l
  // piece-wise mel schedule (kFastMel only; one per kernel, see kernel_tables.cpp piece_schedule)
  int n_mels, nnz;
  const float* vals;               // [nnz] weights, [round][step][lane] x float4
  const MelPiece* mel_pieces;      // [warps of a group][mel_rounds][32 lanes]
  const unsigned char* mel_pcnt;   // [n_mels] partial sums of each filter (1..4)
  int mel_rounds, mel_mpad;        // partial-sum slot of (piece j, filter m) = j * mel_mpad + m
  float power;
  int bin_step;                // 2048 / fft_size: 1, or 2/4/8/16 for zero-padded shorter frames
  // tensor-core variant (stft2048tc.cu) only: [hi, lo] fp16 images of the real 64 x 64
  // form of the 32-point DFT, K-major SWIZZLE_128B
  const void* dft_images;
};
// True when the fused kernel can take this geometry (hop small enough for the
// shared-memory sample tile, mel tables small enough to be resident).
bool stft2048_supports(const FrameGeom& g, int out_kind, int n_mels, int nnz, int mel_rounds,
                       int mpad);
cudaError_t launch_stft2048(const Stft2048Args& a, int out_kind, int sm_count, cudaStream_t st);
// ---- frame-pair kernel (stft2048p.cu): two frames per warp in float32x2 lanes -----
#ifndef SMB_PAIR_TILE
#define SMB_PAIR_TILE 8
#endif
constexpr int kPairTile = SMB_PAIR_TILE;   // frames per group tile, two per warp (8: two groups of four warps; 4: four of two)
constexpr int kPairFilters = 32 / (kPairTile / 2);   // filters per mel round: lane = (filter, frame pair)
// One filter of a mel round of the frame-pair kernel: lane (filter i, frame pair j)
// walks `steps` 4-bin steps from bin b0 (even) of warp j's power rows.
struct PairMelItem {
  int w4_steps;            // weights: float4 index of [step 0][filter i] (low 24 bits), half the
                           // (even) step count of the round (high 8)
  unsigned short h0;       // first bin read / 2 (the band starts on an even bin)
  short m;                 // filter the sum belongs to, -1 for an idle lane
};
struct Stft2048PairArgs {
  const float* x;          // [batch, n]
  float* out;              // [batch, n_mels, frames]
  long long batch;
  FrameGeom g;
  const float* window;     // [2048]
  const float2* tw_pass;   // [32][32]  W_1024^(k1*n2), index k1*32 + n2
  const float2* tw_post;   // [32]      W_2048^l
  int n_mels;
  const float* mel_w;               // [round][step][8 filters] x float4 band weights
  int mel_w_floats;                 // multiple of 4
  const PairMelItem* mel_items;     // [4 warps][mel_rounds][8 filters]
  int mel_rounds;
  float power;
  // optional: the maximum of everything written goes here (atomicMax on the
  // order-preserving key of db_kernels.cu), so that power_to_db's whole-tensor clamp
  // and the MFCC epilogue need no reduction pass of their own
  unsigned long long* max_slot;
};
bool stft2048p_supports(const FrameGeom& g, int n_mels, int mel_w_floats, int mel_rounds);
// ceiling = true: the measurement floor of the transform alone (stage + window + both
// register FFT passes + transposition, one store per value; no split, no |X|^2, no
// mel); `out` then takes total_tiles * 128 floats of scratch.
cudaError_t launch_stft2048p(const Stft2048PairArgs& a, bool ceiling, int sm_count, cudaStream_t st);
// Tensor-core variant: both 32-point passes as split-fp16 products on tcgen05, a
// tile = kTcTile frames = 128 MMA rows per group of kTcTile warps.
constexpr int kTcTile = 4;
bool stft2048tc_supports(const FrameGeom& g, int out_kind, int n_mels, int nnz, int mel_rounds,
                         int mpad);
cudaError_t launch_stft2048tc(const Stft2048Args& a, int out_kind, int sm_count, cudaStream_t st);

// ---- resampler / FIR ----------------------------------------------------------
// One polyphase stage, direct form (resample_stubs.c:127-143):
// out[c][i] = sum_s xz[c][(i*m)/l - k + s] * bank[(i*m) % l][s], zeros outside [0, n).
cudaError_t launch_polyphase_direct(const float* x, long long batch, long long n,
                                    const float* bank, int l, int m, int k,
                                    long long n_out, float* out, cudaStream_t st);
// float64 audio: the same kernel in double (the reference's executor carries
// float32 and float64, resample.ml:72-84).
cudaError_t launch_polyphase_direct_f64(const double* x, long long batch, long long n,
                                        const double* bank, int l, int m, int k,
                                        long long n_out, double* out, cudaStream_t st);

// Decibel conversion (convert.ml:20-56) and the MFCC epilogue (soundml.ml:50-95).
cudaError_t launch_to_db(const void* x, long long count, int dtype, int magnitude, double amin,
                         double scale, double offset, bool clamp, double range,
                         unsigned long long* max_slot, void* out, cudaStream_t st);
// max_known: the slot already holds the maximum of `mel` (left by the fused mel kernel)
cudaError_t launch_mfcc(const void* mel, int dtype, long long batch, int n_mels, long long frames,
                        int n_mfcc, const double* dct, unsigned long long* max_slot, bool max_known,
                        double amin, double scale, double offset, double range, void* out,
                        cudaStream_t st);
// power_to_db in place over values whose whole-tensor maximum is in the slot
cudaError_t launch_db_known_max(void* x, long long count, int dtype, double amin, double scale,
                                double offset, bool clamp, double range,
                                const unsigned long long* max_slot, cudaStream_t st);

// soundml-io's layout pass (soundml_io_stubs.c:832-872): interleaved [frames][channels]
// -> planar (channel c at out + c * out_total) or the mono downmix.
cudaError_t launch_ingest_layout(const void* in, int dtype, long long frames, int channels,
                                 int downmix, void* out, long long out_total, cudaStream_t st);

// Overlap-save stage (FIR, xL, /M) on half-length complex FFTs.
struct OlsArgs {
  const float* x;        // [batch, n]
  float* out;            // [batch, n_out]
  long long n, n_out, blocks;
  int L, M, K, N, B, delta, W;
  const float2* H;       // plan spectrum: W/2+1 bins (xL) or N/2+1 (otherwise), scales folded in;
                         // polyphase plans: L spectra of N/2+1 bins, one per branch
  int polyphase;         // xL stage laid out as L input-rate branches (ols2048_kernel)
  const float2* tw;      // exp(-2 pi i j / max(N, W)), j < max(N, W)/2
};
size_t ols_smem_bytes(int N, int W);
cudaError_t launch_ols(const OlsArgs& a, long long batch, cudaStream_t st);
// Warp-per-block register-FFT variant for N = 2048, L = 1 (ols2048.cu).
bool ols2048_supports(const OlsArgs& a);
cudaError_t launch_ols2048(const OlsArgs& a, const float2* tw_pass, const float2* tw_base,
                           long long batch, int sm_count, cudaStream_t st);

// Phase-rich polyphase stage as a banded tf32x3 product on tcgen05 (resample_gemm.cu).
struct GemmResampleArgs {
  const float* x;          // [batch, n]
  float* out;              // [batch, n_out]
  long long n, n_out;
  int l, m, k;             // columns of this launch, stage M, group delay less the skipped K-chunks
  int l_total, col_begin;  // stage L (outputs per block-row) and this launch's first column
  int n_pad;               // l rounded up to a multiple of 16 (UMMA N)
  int chunks;              // ceil(P / 32) K-chunks
  int tmem_cols;           // power of two >= 3 * n_pad
  const float* b_images;   // per chunk: [hi, lo][ncols][32] pre-swizzled K-major tiles of G
  const int4* chunk_meta;  // per chunk: {byte offset into b_images, first column, columns, 0}
};
size_t resample_gemm_smem_bytes(int n_pad);

// The same stage in row form (resample_gemm.cu, resample_rows_kernel): the input is read
// as non-overlapping rows X[i][j'] = xz[i M + j' - K], j' < M, and block-row rho of the
// output is sum_q X[rho + q] G_q with G_q = rows [q M, (q + 1) M) of G -- one accumulator
// per shift q, added with the row shift in the epilogue.  Every input sample is gathered
// and split once per tile instead of P / M times.
struct GemmRowsArgs {
  const float* x;          // [batch, n]
  float* out;              // [batch, n_out]
  long long n, n_out;
  int l, m, k;             // columns of this launch (at most 160), stage M, group delay less the whole input rows skipped
  int l_total, col_begin;  // stage L (outputs per block-row) and this launch's first column
  int n_pad;               // l rounded up to a multiple of 16
  int shifts;              // accumulators: ceil(P / M), at most 4
  int chunks;              // ceil(M / 32) K-chunks (at most 32)
  int slices;              // entries of slice_meta (at most 64)
  int tmem_cols;           // power of two >= sum of acc_w
  int b_stage_bytes;       // largest chunk image (multiple of 1024)
  int a_stages, b_stages;  // pipeline depth of the A tiles and of the B images (2 .. 4)
  int a_tmem, a_tmem_col;  // A tiles in tensor memory (64 columns per stage from a_tmem_col) instead of shared memory
  // accumulators: one per shift q (index q), and optionally one more that takes the two small
  // split terms of the shift holding the filters' main lobes (so that accumulator is a short
  // chain of exact hi x hi products only: what keeps a 14-chunk stage at -132 dB THD+N)
  int n_acc;               // shifts, or shifts + 1
  int acc_shift[5];        // the row shift the accumulator's rows carry
  int acc_col[5];          // its TMEM column (the shifts laid out in descending q)
  int acc_lo[5];           // first G column it holds (multiple of 16)
  int acc_w[5];            // its width (multiple of 16)
  const float* b_images;   // per chunk, per slice: [hi, lo][columns][32] pre-swizzled K-major tiles; a slice is a
                           // contiguous run of TMEM columns (the end of D_q followed by the start of D_(q-1))
  const int4* chunk_meta;  // per chunk: {byte offset into b_images, bytes, first slice, slices}
  const int4* slice_meta;  // per slice: {byte offset of its hi rows inside the chunk image, TMEM column, columns,
                           //  kind | owner << 2 | byte distance from the hi rows to the lo rows << 3}; kind 0: all
                           //  three products, 1: hi x hi only, 2: the two small terms only; owner: which of the
                           //  two issuing threads takes the slice
  int two_issuers;         // slices are dealt to two MMA-issuing threads (every accumulator to one of them)
};
size_t resample_rows_smem_bytes(int a_stages, int b_stages, int b_stage_bytes);
cudaError_t launch_resample_rows(const GemmRowsArgs& a, long long batch, int sm_count, cudaStream_t st);
cudaError_t launch_resample_gemm(const GemmResampleArgs& a, long long batch, cudaStream_t st);

}  // namespace smb
