// Host code that decides the format of every table a kernel reads and fills it in host
// memory: the fft-2048 constants, the fused STFT kernels' mel schedules and the tcgen05
// resampler's stage layouts.  No CUDA runtime call: the C ABI (api.cu) uploads and owns.
#pragma once
#include <cuda_fp16.h>

#include <cmath>
#include <vector>

#include "host_design.h"
#include "kernels.h"

namespace smb {

constexpr double kTwoPi = 6.283185307179586476925286766559;
// (cos, -sin)(2 pi j / n) for j < count, as float2 or double2.
template <typename V>
std::vector<V> unit_roots(int64_t count, int64_t n) {
  std::vector<V> roots((size_t)count);
  for (int64_t j = 0; j < count; ++j) {
    const double a = kTwoPi * double(j) / double(n);
    roots[(size_t)j] = V{(decltype(V::x))std::cos(a), (decltype(V::x))-std::sin(a)};
  }
  return roots;
}
// The inter-pass twiddles of the warp FFT 1024 (32 x 32): W_1024^(k1 n2) at [k1][n2].
std::vector<float2> fft1024_pass_twiddles();
// The tensor-core STFT's 32-point DFT as two split-fp16 operand images.
std::vector<__half> dft32_split_images();

// Mel schedule of a fused kernel (stft2048.cu, stft2048tc.cu).
struct PieceSchedule {
  std::vector<float> vals;               // [round][step][lane] float4 weights
  std::vector<MelPiece> pieces;          // [warps][rounds][32]
  std::vector<unsigned char> pcnt;       // [n_mels]: pieces (= partial sums) of each filter, 1..4
  int rounds = 0, mpad = 0;              // partial-sum slot of (piece j, filter m) = j * mpad + m
};
// Mel schedule of the frame-pair kernel (stft2048p.cu).
struct PairSchedule {
  std::vector<float> w;                  // [round][step][8 filters] x float4
  std::vector<PairMelItem> items;        // [4 warps][rounds][8]
  int rounds = 0;
};
// The schedules of filterbank weights [n_mels][bins], filter m nonzero only in bins
// [band_lo[m], band_hi[m]); empty when the filterbank does not fit the kernel.
PairSchedule pair_schedule(const std::vector<double>& weights, const std::vector<int>& band_lo,
                           const std::vector<int>& band_hi, int64_t n_mels, int64_t bins);
PieceSchedule piece_schedule(const std::vector<double>& weights, const std::vector<int>& band_lo,
                             const std::vector<int>& band_hi, int64_t n_mels, int64_t bins, int warps,
                             int ps, int window);

// The tcgen05 resampler's tables for one stage tagged "gemm" (L <= 1024), in column groups
// of <= 160 (one launch each: a group's accumulators must fit the 512 TMEM columns).
struct GemmLayout {
  template <typename Args>
  struct Group {                                // one launch
    Args a{};                                   // signal and table pointers unset
    std::vector<float> images;
    std::vector<int4> chunk_meta, slice_meta;   // slice_meta: row form only
  };
  std::vector<Group<GemmRowsArgs>> rows;        // resample_rows_kernel; empty when no row layout fits
  std::vector<Group<GemmResampleArgs>> windows; // resample_gemm_kernel, the fall-back; empty: no tcgen05 tables
};
// SMB_ROWS_SPLIT, SMB_ROWS_SMEM_A and SMB_ROWS_TMEM_A force a row layout; they are read here.
GemmLayout gemm_layout(const ResampleStage& s);

}  // namespace smb
