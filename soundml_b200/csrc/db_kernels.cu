// Decibel conversion and MFCC epilogue kernels (SURVEY.md 8f rank 1: what ML
// consumers ingest downstream of the mel spectrogram).
//
//   to_db   convert.ml:20-56   floor at amin, log / scale / offset in the input's
//           own dtype, optional whole-tensor top_db clamp (one max reduction)
//   mfcc    soundml.ml:50-95   log-mel with the 80 dB clamp, raw type-II DCT along
//           the mel axis, orthonormal scales, lifter -- double interior, one
//           rounding
#include "kernels.h"
#include "max_key.cuh"

namespace smb {

namespace {

__device__ __forceinline__ void block_max_to(double v, unsigned long long* slot) { warp_max_to(v, slot); }

template <typename T> __device__ __forceinline__ T log_t(T v);
template <> __device__ __forceinline__ float log_t<float>(float v) { return logf(v); }
template <> __device__ __forceinline__ double log_t<double>(double v) { return log(v); }

// db = log(max(|x| or x, amin)) * scale - offset, every operation in T; the
// running maximum of db goes to *max_slot when the clamp is requested.
template <typename T>
__global__ void to_db_kernel(const T* __restrict__ x, long long count, int magnitude, T amin,
                             T scale, T offset, unsigned long long* max_slot,
                             T* __restrict__ out) {
  double local = -1.0e308;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count;
       i += (long long)gridDim.x * blockDim.x) {
    T v = x[i];
    if (magnitude) v = v < T(0) ? -v : v;
    v = v > amin ? v : amin;
    const T db = log_t<T>(v) * scale - offset;
    out[i] = db;
    local = fmax(local, (double)db);
  }
  if (max_slot) block_max_to(local, max_slot);
}

template <typename T>
__global__ void clamp_db_kernel(T* __restrict__ out, long long count,
                                const unsigned long long* max_slot, double range) {
  const T floor_db = (T)(value_of(*max_slot) - range);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count;
       i += (long long)gridDim.x * blockDim.x) {
    const T v = out[i];
    out[i] = v > floor_db ? v : floor_db;
  }
}

template <typename T>
__global__ void max_value_kernel(const T* __restrict__ x, long long count,
                                 unsigned long long* max_slot) {
  double local = -1.0e308;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count;
       i += (long long)gridDim.x * blockDim.x)
    local = fmax(local, (double)x[i]);
  block_max_to(local, max_slot);
}

constexpr int kMfccFrames = 32;     // frame columns per CTA
constexpr int kMfccThreads = 256;
constexpr int kMfccPer = 3;         // coefficients per thread (the log-mel value is loaded once for them)
constexpr int kMfccGroups = kMfccThreads / kMfccFrames;  // coefficient c = c0 + g + kMfccGroups * j
constexpr int kMfccCoefs = kMfccGroups * kMfccPer;       // coefficients per CTA
constexpr int kMfccChunk = 128;     // mel bands staged at once: shared memory stays under 56 KB

// mel [batch, n_mels, frames] (T) -> out [batch, n_mfcc, frames] (T).  One CTA per
// (32-frame tile, signal, group of kMfccCoefs coefficients).  The mel axis is walked
// in chunks of kMfccChunk bands: each chunk's log-mel tile is built in shared memory in
// double (with the 80 dB clamp below the whole-tensor maximum) next to that chunk's DCT
// rows, then thread (coefficient group, frame) continues its fma chains over the chunk:
// one log-mel load feeds up to three coefficients.  Every coefficient is the same
// ascending-m fma chain whatever the chunking, so the chunk size does not change a bit.
template <typename T>
__global__ void __launch_bounds__(kMfccThreads)
mfcc_kernel(const T* __restrict__ mel, int n_mels, long long frames, int n_mfcc,
            const double* __restrict__ dct, const unsigned long long* max_mel_slot, double amin,
            double scale, double offset, double range, T* __restrict__ out) {
  extern __shared__ __align__(8) double sDb[];           // [chunk][kMfccFrames], then the DCT rows
  const long long b = blockIdx.y;
  const long long p0 = (long long)blockIdx.x * kMfccFrames;
  const int c0 = blockIdx.z * kMfccCoefs;
  const int rows = min(kMfccCoefs, n_mfcc - c0);          // this CTA's coefficients
  const int nf = (int)min((long long)kMfccFrames, frames - p0);
  // the maximum of db is db of the maximum (the map is monotone)
  const double vmax = fmax(value_of(*max_mel_slot), amin);
  const double floor_db = (log(vmax) * scale - offset) - range;
  const T* src = mel + b * n_mels * frames + p0;
  const int f = threadIdx.x & (kMfccFrames - 1);
  const int g = threadIdx.x / kMfccFrames;
  double acc[kMfccPer];
#pragma unroll
  for (int j = 0; j < kMfccPer; ++j) acc[j] = 0.0;
  for (int m0 = 0; m0 < n_mels; m0 += kMfccChunk) {
    const int len = min(kMfccChunk, n_mels - m0);
    double* sDct = sDb + len * kMfccFrames;               // [rows][len]
    if (m0 > 0) __syncthreads();                          // the previous chunk is consumed
    for (int i = threadIdx.x; i < rows * kMfccChunk; i += blockDim.x) {   // (row, band): shifts, no division
      const int r = i / kMfccChunk, m = i % kMfccChunk;
      if (m < len) sDct[r * len + m] = __ldg(dct + (long long)(c0 + r) * n_mels + m0 + m);
    }
    for (int i = threadIdx.x; i < len * kMfccFrames; i += blockDim.x) {
      const int m = i / kMfccFrames, ff = i - m * kMfccFrames;
      double db = 0.0;
      if (ff < nf) {
        const double v = fmax((double)src[(long long)(m0 + m) * frames + ff], amin);
        db = fmax(log(v) * scale - offset, floor_db);
      }
      sDb[i] = db;
    }
    __syncthreads();
    const double* row[kMfccPer];
#pragma unroll
    for (int j = 0; j < kMfccPer; ++j) row[j] = sDct + min(g + kMfccGroups * j, rows - 1) * len;
    for (int m = 0; m < len; ++m) {
      const double v = sDb[m * kMfccFrames + f];
#pragma unroll
      for (int j = 0; j < kMfccPer; ++j) acc[j] = fma(row[j][m], v, acc[j]);
    }
  }
  T* dst = out + b * n_mfcc * frames + p0 + f;
#pragma unroll
  for (int j = 0; j < kMfccPer; ++j)
    if (f < nf && g + kMfccGroups * j < rows) dst[(long long)(c0 + g + kMfccGroups * j) * frames] = (T)acc[j];
}

// db in place over values whose maximum is already in the slot (the fused mel kernel
// left it there): the reference's arithmetic in T, clamp included, one pass
template <typename T>
__global__ void db_with_known_max_kernel(T* __restrict__ x, long long count, T amin, T scale, T offset,
                                         const unsigned long long* max_slot, bool clamp, T range) {
  T vmax = (T)value_of(*max_slot);
  vmax = vmax > amin ? vmax : amin;
  const T floor_db = (log_t<T>(vmax) * scale - offset) - range;     // max of db = db of the max
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count;
       i += (long long)gridDim.x * blockDim.x) {
    T v = x[i];
    v = v > amin ? v : amin;
    const T db = log_t<T>(v) * scale - offset;
    x[i] = clamp && db < floor_db ? floor_db : db;
  }
}

int grid_for(long long count) {
  long long g = (count + 255) / 256;
  return (int)(g < 148 * 8 ? (g < 1 ? 1 : g) : 148 * 8);
}

}  // namespace

cudaError_t launch_to_db(const void* x, long long count, int dtype, int magnitude, double amin,
                         double scale, double offset, bool clamp, double range,
                         unsigned long long* max_slot, void* out, cudaStream_t st) {
  if (count == 0) return cudaSuccess;
  if (clamp) {
    cudaError_t e = cudaMemsetAsync(max_slot, 0, sizeof(unsigned long long), st);
    if (e != cudaSuccess) return e;
  }
  const int grid = grid_for(count);
  if (dtype == 0)
    to_db_kernel<float><<<grid, 256, 0, st>>>((const float*)x, count, magnitude, (float)amin,
                                              (float)scale, (float)offset,
                                              clamp ? max_slot : nullptr, (float*)out);
  else
    to_db_kernel<double><<<grid, 256, 0, st>>>((const double*)x, count, magnitude, amin, scale,
                                               offset, clamp ? max_slot : nullptr, (double*)out);
  ++g_launch_count;
  if (clamp) {
    if (dtype == 0) clamp_db_kernel<float><<<grid, 256, 0, st>>>((float*)out, count, max_slot, range);
    else clamp_db_kernel<double><<<grid, 256, 0, st>>>((double*)out, count, max_slot, range);
    ++g_launch_count;
  }
  return cudaGetLastError();
}

cudaError_t launch_db_known_max(void* x, long long count, int dtype, double amin, double scale,
                                double offset, bool clamp, double range,
                                const unsigned long long* max_slot, cudaStream_t st) {
  if (count == 0) return cudaSuccess;
  if (dtype == 0)
    db_with_known_max_kernel<float><<<grid_for(count), 256, 0, st>>>(
        (float*)x, count, (float)amin, (float)scale, (float)offset, max_slot, clamp, (float)range);
  else
    db_with_known_max_kernel<double><<<grid_for(count), 256, 0, st>>>(
        (double*)x, count, amin, scale, offset, max_slot, clamp, range);
  ++g_launch_count;
  return cudaGetLastError();
}

cudaError_t launch_mfcc(const void* mel, int dtype, long long batch, int n_mels, long long frames,
                        int n_mfcc, const double* dct, unsigned long long* max_slot, bool max_known,
                        double amin, double scale, double offset, double range, void* out,
                        cudaStream_t st) {
  if (batch == 0 || frames == 0) return cudaSuccess;
  cudaError_t e;
  if (!max_known) {                      // else the kernel that wrote `mel` left its maximum in the slot
    e = cudaMemsetAsync(max_slot, 0, sizeof(unsigned long long), st);
    if (e != cudaSuccess) return e;
    const long long count = batch * n_mels * frames;
    if (dtype == 0) max_value_kernel<float><<<grid_for(count), 256, 0, st>>>((const float*)mel, count, max_slot);
    else max_value_kernel<double><<<grid_for(count), 256, 0, st>>>((const double*)mel, count, max_slot);
    ++g_launch_count;
  }
  // one chunk of the log-mel tile and its DCT rows
  const int chunk = n_mels < kMfccChunk ? n_mels : kMfccChunk;
  const int rows = n_mfcc < kMfccCoefs ? n_mfcc : kMfccCoefs;
  const size_t smem = (size_t)chunk * (kMfccFrames + rows) * sizeof(double);
  const long long tiles = (frames + kMfccFrames - 1) / kMfccFrames;
  const unsigned groups = (unsigned)((n_mfcc + kMfccCoefs - 1) / kMfccCoefs);
  if (groups > 65535u) return cudaErrorInvalidConfiguration;
  for (long long b0 = 0; b0 < batch; b0 += 65535) {
    const long long nb = batch - b0 < 65535 ? batch - b0 : 65535;
    dim3 grid((unsigned)tiles, (unsigned)nb, groups);
    if (dtype == 0) {
      e = cudaFuncSetAttribute(mfcc_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return e;
      mfcc_kernel<float><<<grid, kMfccThreads, smem, st>>>(
          (const float*)mel + b0 * n_mels * frames, n_mels, frames, n_mfcc, dct, max_slot, amin,
          scale, offset, range, (float*)out + b0 * n_mfcc * frames);
    } else {
      e = cudaFuncSetAttribute(mfcc_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return e;
      mfcc_kernel<double><<<grid, kMfccThreads, smem, st>>>(
          (const double*)mel + b0 * n_mels * frames, n_mels, frames, n_mfcc, dct, max_slot, amin,
          scale, offset, range, (double*)out + b0 * n_mfcc * frames);
    }
    ++g_launch_count;
  }
  return cudaGetLastError();
}

}  // namespace smb
