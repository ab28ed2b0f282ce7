// Polyphase resampler / FIR kernels (sm_100a).
//
// One stage of the reference's resampler is, whichever executor the planner
// tags it with, the same filter (resample.ml:22-52): output i of a stage with
// factors l/m and group delay k is
//
//     out[i] = sum_{s=0}^{2k} xz[floor(i*m/l) - k + s] * bank[(i*m) mod l][s]
//
// with xz = x extended by zeros on both sides (resample_stubs.c:127-143;
// independent evaluator soundml/test/resample/resample_kernel.ml:144-163).
// Phase and window start are exact integers -- no float time accumulator.

#include "kernels.h"

namespace smb {

namespace {

constexpr int kOutPerCta = 256;

// Direct form: a CTA produces kOutPerCta consecutive outputs of one signal from
// an input span staged once in shared memory; each thread owns one output and
// walks its phase's bank row.
template <typename T>
__global__ void __launch_bounds__(kOutPerCta)
polyphase_direct_kernel(const T* __restrict__ x, long long n,
                        const T* __restrict__ bank, int l, int m, int k,
                        long long n_out, T* __restrict__ out, int span_cap) {
  extern __shared__ __align__(8) unsigned char sRaw[];
  T* sIn = reinterpret_cast<T*>(sRaw);
  const long long c = blockIdx.y;
  const long long i0 = (long long)blockIdx.x * kOutPerCta;
  const int cnt = (int)min((long long)kOutPerCta, n_out - i0);
  const T* xs = x + c * n;
  const int taps = 2 * k + 1;
  const long long lo = (i0 * m) / l - k;                    // first input read
  const long long hi = ((i0 + cnt - 1) * m) / l + k;        // last input read
  const int span = (int)(hi - lo + 1);
  for (int j = threadIdx.x; j < span; j += blockDim.x) {
    const long long s = lo + j;
    sIn[j] = (s >= 0 && s < n) ? __ldg(xs + s) : T(0);
  }
  __syncthreads();
  if ((int)threadIdx.x < cnt) {
    const long long i = i0 + threadIdx.x;
    const long long t = i * m;
    const int phase = (int)(t % l);
    const int off = (int)(t / l - k - lo);
    const T* h = bank + (long long)phase * taps;
    const T* v = sIn + off;
    T a0 = 0, a1 = 0, a2 = 0, a3 = 0;
    int s = 0;
    for (; s + 4 <= taps; s += 4) {
      a0 = fma(v[s], __ldg(h + s), a0);
      a1 = fma(v[s + 1], __ldg(h + s + 1), a1);
      a2 = fma(v[s + 2], __ldg(h + s + 2), a2);
      a3 = fma(v[s + 3], __ldg(h + s + 3), a3);
    }
    for (; s < taps; ++s) a0 = fma(v[s], __ldg(h + s), a0);
    out[c * n_out + i] = (a0 + a1) + (a2 + a3);
  }
}


// ---- register-blocked direct form for small ratios ----------------------------------
//
// A stage with factors L / M advances in cycles of L outputs per M inputs:
//
//     out[L j + p] = sum_s xz[M j + o_p - K + s] * bank[r_p][s],   o_p = (p M) div L,  r_p = (p M) mod L
//
// so for L, M <= 4 (compile-time) everything but j is static.  A thread owns kCycles
// consecutive cycles -- kCycles * L consecutive outputs -- and walks the taps in chunks
// of one 16-byte vector: the inputs a chunk needs are a contiguous window of
// M (kCycles - 1) + max o_p + VEC samples held in registers, which slides by one vector
// per chunk (one 16-byte shared-memory load), and the chunk's taps are one broadcast
// 16-byte load per phase: kCycles * L * VEC FMAs for 1 + L loads.  Every output is one
// accumulator chain over ascending s, whatever tile or call it falls in.  The staged
// inputs carry 16 bytes of padding per 128 so that the 32 lanes, whose windows start
// kCycles * M samples apart, load from distinct bank groups.
#ifndef SMB_BLOCK_CYCLES
#define SMB_BLOCK_CYCLES 8
#endif
#ifndef SMB_BLOCK_THREADS
#define SMB_BLOCK_THREADS 128
#endif
constexpr int kCycles = SMB_BLOCK_CYCLES;
constexpr int kBlockThreads = SMB_BLOCK_THREADS;

template <typename T>
struct alignas(16) Vec16 { T v[16 / sizeof(T)]; };

template <typename T, int L, int M>
struct BlockShape {
  static constexpr int VEC = 16 / (int)sizeof(T);            // elements per 16-byte vector
  static constexpr int BLK = 128 / (int)sizeof(T);           // elements per 128 bytes (then one vector of padding)
  static constexpr int OMAX = ((L - 1) * M) / L;
  static constexpr int WLEN = M * (kCycles - 1) + OMAX + VEC; // window elements a chunk touches
  static constexpr int NV = (WLEN + VEC - 1) / VEC;          // ... in vectors (the ring)
  static int row_vecs(int k) { return (2 * k + 1 + VEC - 1) / VEC; }
  // staged input elements of a tile: the last thread's window at the last chunk, plus the ring's look-ahead
  static int span(int k) { return kBlockThreads * kCycles * M + (row_vecs(k) + NV + 1) * VEC; }
  static size_t smem(int k) {
    const int in_elems = span(k) + (span(k) / BLK + 1) * VEC;
    return (size_t)(((in_elems + VEC - 1) / VEC) * VEC + L * row_vecs(k) * VEC) * sizeof(T);
  }
};

template <typename T, int L, int M>
__global__ void __launch_bounds__(kBlockThreads)
polyphase_block_kernel(const T* __restrict__ x, long long n, const T* __restrict__ bank, int k,
                       long long n_out, T* __restrict__ out, int span, int row_vecs) {
  using S = BlockShape<T, L, M>;
  constexpr int VEC = S::VEC, BLK = S::BLK, NV = S::NV;
  extern __shared__ __align__(16) unsigned char sRaw2[];
  T* sIn = reinterpret_cast<T*>(sRaw2);                                    // padded input span
  const int in_elems = span + (span / BLK + 1) * VEC;
  T* sBank = sIn + ((in_elems + VEC - 1) / VEC) * VEC;                    // [L][row_vecs * VEC], zero tail
  const long long c = blockIdx.y;
  const long long j0 = (long long)blockIdx.x * (kBlockThreads * kCycles);  // first cycle of the tile
  const T* xs = x + c * n;
  const int taps = 2 * k + 1;
  const long long lo = M * j0 - k;                                         // source index of staged element 0
  for (int q = threadIdx.x; q < span; q += kBlockThreads) {
    const long long src = lo + q;
    sIn[q + (q / BLK) * VEC] = (src >= 0 && src < n) ? __ldg(xs + src) : T(0);
  }
  for (int q = threadIdx.x; q < L * row_vecs * VEC; q += kBlockThreads) {
    const int r = q / (row_vecs * VEC), t = q - r * row_vecs * VEC;
    sBank[q] = t < taps ? __ldg(bank + (long long)r * taps + t) : T(0);
  }
  __syncthreads();

  T acc[kCycles][L];
#pragma unroll
  for (int j = 0; j < kCycles; ++j)
#pragma unroll
    for (int pp = 0; pp < L; ++pp) acc[j][pp] = T(0);
  // staged element of (cycle j, phase p, tap s): base + M j + o_p + s, base a multiple of VEC
  const int base = (int)threadIdx.x * kCycles * M;
  auto load_vec = [&](int elem) {                                  // elem is a multiple of VEC
    return *reinterpret_cast<const Vec16<T>*>(sIn + elem + (elem / BLK) * VEC);
  };
  // ring of NV vectors: at chunk t, ring[(t + i) % NV] holds vector t + i of the thread's span
  Vec16<T> ring[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) ring[i] = load_vec(base + i * VEC);
  for (int t0 = 0; t0 < row_vecs; t0 += NV) {
#pragma unroll
    for (int u = 0; u < NV; ++u) {
      const int t = t0 + u;                                        // chunk: taps [t VEC, (t + 1) VEC)
      if (t < row_vecs) {                                          // (uniform)
        Vec16<T> h[L];
#pragma unroll
        for (int pp = 0; pp < L; ++pp)
          h[pp] = *reinterpret_cast<const Vec16<T>*>(sBank + (((pp * M) % L) * row_vecs + t) * VEC);
#pragma unroll
        for (int e = 0; e < VEC; ++e)
#pragma unroll
          for (int j = 0; j < kCycles; ++j)
#pragma unroll
            for (int pp = 0; pp < L; ++pp) {
              const int w = M * j + (pp * M) / L + e;              // element of the chunk's window
              acc[j][pp] = fma(ring[(u + w / VEC) % NV].v[w % VEC], h[pp].v[e], acc[j][pp]);
            }
        ring[u] = load_vec(base + (t + NV) * VEC);                 // vector t is done: bring in t + NV
      }
    }
  }
  // kCycles * L consecutive outputs per thread
  const long long i0 = (j0 + (long long)threadIdx.x * kCycles) * L;
  T* o = out + c * n_out + i0;
#pragma unroll
  for (int j = 0; j < kCycles; ++j)
#pragma unroll
    for (int pp = 0; pp < L; ++pp)
      if (i0 + j * L + pp < n_out) o[j * L + pp] = acc[j][pp];
}

template <typename T, int L, int M>
static cudaError_t launch_block(const T* x, long long batch, long long n, const T* bank, int k,
                                long long n_out, T* out, cudaStream_t st) {
  using S = BlockShape<T, L, M>;
  const size_t smem = S::smem(k);
  cudaError_t e = cudaFuncSetAttribute(polyphase_block_kernel<T, L, M>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const long long cycles = (n_out + L - 1) / L;
  const long long tiles = (cycles + kBlockThreads * kCycles - 1) / (kBlockThreads * kCycles);
  for (long long b0 = 0; b0 < batch; b0 += 65535) {
    const long long nb = batch - b0 < 65535 ? batch - b0 : 65535;
    dim3 grid((unsigned)tiles, (unsigned)nb);
    polyphase_block_kernel<T, L, M><<<grid, kBlockThreads, smem, st>>>(
        x + b0 * n, n, bank, k, n_out, out + b0 * n_out, S::span(k), S::row_vecs(k));
    ++g_launch_count;
  }
  return cudaGetLastError();
}

// the blocked kernel takes ratios with L, M <= 4 whose tile fits shared memory
template <typename T>
static bool try_block(const T* x, long long batch, long long n, const T* bank, int l, int m, int k,
                      long long n_out, T* out, cudaStream_t st, cudaError_t* err) {
#define SMB_TRY(LL, MM)                                                                    \
  if (l == LL && m == MM) {                                                                \
    if (BlockShape<T, LL, MM>::smem(k) > 200 * 1024) return false;                         \
    *err = launch_block<T, LL, MM>(x, batch, n, bank, k, n_out, out, st);                  \
    return true;                                                                           \
  }
  SMB_TRY(1, 1) SMB_TRY(1, 2) SMB_TRY(1, 3) SMB_TRY(1, 4) SMB_TRY(2, 1) SMB_TRY(3, 1) SMB_TRY(4, 1)
  SMB_TRY(2, 3) SMB_TRY(3, 2) SMB_TRY(3, 4) SMB_TRY(4, 3)
#undef SMB_TRY
  return false;
}

}  // namespace

template <typename T>
static cudaError_t launch_direct_t(const T* x, long long batch, long long n, const T* bank, int l,
                                   int m, int k, long long n_out, T* out, cudaStream_t st) {
  if (batch == 0 || n_out == 0) return cudaSuccess;
  cudaError_t blocked = cudaSuccess;
  if (try_block<T>(x, batch, n, bank, l, m, k, n_out, out, st, &blocked)) return blocked;
  const long long span_cap = ((long long)(kOutPerCta - 1) * m) / l + 2 + 2LL * k + 1;
  const size_t smem = (size_t)span_cap * sizeof(T);
  if (smem > 200 * 1024) return cudaErrorInvalidConfiguration;
  cudaError_t e = cudaFuncSetAttribute(polyphase_direct_kernel<T>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const long long tiles = (n_out + kOutPerCta - 1) / kOutPerCta;
  for (long long b0 = 0; b0 < batch; b0 += 65535) {
    const long long nb = batch - b0 < 65535 ? batch - b0 : 65535;
    dim3 grid((unsigned)tiles, (unsigned)nb);
    polyphase_direct_kernel<T><<<grid, kOutPerCta, smem, st>>>(x + b0 * n, n, bank, l, m, k, n_out,
                                                               out + b0 * n_out, (int)span_cap);
    ++g_launch_count;
  }
  return cudaGetLastError();
}

cudaError_t launch_polyphase_direct(const float* x, long long batch, long long n,
                                    const float* bank, int l, int m, int k,
                                    long long n_out, float* out, cudaStream_t st) {
  return launch_direct_t<float>(x, batch, n, bank, l, m, k, n_out, out, st);
}

cudaError_t launch_polyphase_direct_f64(const double* x, long long batch, long long n,
                                        const double* bank, int l, int m, int k,
                                        long long n_out, double* out, cudaStream_t st) {
  return launch_direct_t<double>(x, batch, n, bank, l, m, k, n_out, out, st);
}

}  // namespace smb
