// Least-squares STFT synthesis for fft_size = 2048, complex64 -> float32 (sm_100a).
//
// Same synthesis equation and envelope as istft_kernels.cu (Stft.invert,
// stft.ml:693-939), with the inverse transforms on the register FFT of the fused
// analysis kernel.  A CTA of 16 warps owns a run of R hops of output; with C =
// ceil(2048 / hop) frames overlapping one position, R = 16 - (C - 1) when runs
// start on a frame boundary (left width a multiple of the hop) and 16 - C
// otherwise, so at most 16 frames reach a run.  They are
//   * fetched together, [bins][16 frames] along the contiguous frame axis, into a
//     padded shared-memory tile (the spectrum is stored frames-last, so a single
//     frame is a stride-`frames` column: the tile is what keeps the reads
//     coalesced),
//   * inverted one per warp: Zinv[k] = (Y[k] + conj Y[1024-k]) + i W^-k (Y[k] -
//     conj Y[1024-k]) for the bin pair each lane holds, the 1024-k halves moved
//     into place by warp shuffle, then the 32 x 32 forward FFT of conj(Zinv)
//     (the tile's memory is reused for the transposes),
//   * windowed (1/2048 folded into the window) and left in the warp's transpose
//     buffer; after one barrier every output position gathers the taps of the
//     frames that reach it, newest first (fixed order, deterministic), divides
//     by the envelope and is written once.
// 3 of every 16 transforms (hop 512) are recomputed by the neighbouring run.
//
// Frame sizes 1024 ... 128 ride along: the inverse of a 2048-point spectrum that
// carries X[k] at bin k * (2048 / fft) and zeros elsewhere is the fft-point inverse
// repeated, so the kernel spreads the fft / 2 + 1 input bins while it reads the
// tile and uses the first fft samples of each frame (window tail zero, 1 / fft
// folded into the window).
#include <cstdint>

#include "fft32.cuh"
#include "kernels.h"

namespace smb {

namespace {

using namespace fft32impl;

constexpr int kN = 2048;
constexpr int kHalf = 1024;
constexpr int kBins = 1025;
constexpr int kWarps = 16;
constexpr int kTileStride = 17;                     // float2 per bin row: 16 frames + 1 pad
constexpr int kExFloats = 32 * kFft1024ExStride * 2;
// shared by the spectrum tile [1025][17] complex and, after it, the 16 transposes
constexpr int kWorkFloats = ((kBins * kTileStride * 2 + 3) / 4) * 4;
static_assert(kWorkFloats >= kWarps * kExFloats, "transposes fit the tile space");

__device__ __forceinline__ long long ceil_div_ll(long long a, long long b) {   // b > 0
  return a >= 0 ? (a + b - 1) / b : -((-a) / b);
}

struct Istft2048Params {
  IstftArgs a;
  const float* window;       // [2048] analysis window / 2048
  const float2* tw_pass;     // [32][32]  W_1024^(k1 n2)
  const float2* tw_base;     // [32]      W_2048^l
  int classes;               // C = ceil(2048 / hop)
  int run_hops;              // R
  long long runs_per_signal, total_runs;
};

template <int STEP>                                     // 2048 / fft_size
__global__ void __launch_bounds__(kWarps * 32, 1)
istft2048_kernel(const Istft2048Params p) {
  extern __shared__ __align__(16) float smem[];
  float2* sTwPass = reinterpret_cast<float2*>(smem);                  // [16][32][2]
  float2* sTwBase = sTwPass + 1024;                                   // [32]
  float* sWindow = reinterpret_cast<float*>(sTwBase + 32);            // [2048]
  float* sWork = sWindow + kN;                 // spectrum tile [1025][17] float2, then 16 transposes
  float* sInvEnv = sWork + kWorkFloats;        // [hop] 1 / envelope of the fully covered positions
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const IstftArgs& a = p.a;
  for (int i = tid; i < 1024; i += blockDim.x) {
    const int l = i & 31, k1 = i >> 5;
    sTwPass[(((k1 >> 1) * 32 + l) << 1) + (k1 & 1)] = p.tw_pass[i];
  }
  if (tid < 32) sTwBase[tid] = p.tw_base[tid];
  for (int i = tid; i < kN; i += blockDim.x) sWindow[i] = p.window[i];
  for (int i = tid; i < p.a.hop; i += blockDim.x) {
    const double e = p.a.folded[i];
    sInvEnv[i] = (float)(1.0 / (e == 0.0 ? 1.0 : e));
  }
  __syncthreads();

  float2* tile = reinterpret_cast<float2*>(sWork);
  float2* ex = reinterpret_cast<float2*>(sWork + warp * kExFloats);
  const float4* tw4 = reinterpret_cast<const float4*>(sTwPass);
  const float2 wl = sTwBase[lane];
  const int partner = (32 - lane) & 31;
  const int hop = a.hop;
  const int run_len = p.run_hops * hop;
  constexpr int fft = kN / STEP;                          // frame length
  constexpr int bin_mask = STEP - 1;
  constexpr int bin_shift = STEP == 1 ? 0 : STEP == 2 ? 1 : STEP == 4 ? 2 : STEP == 8 ? 3 : 4;
  constexpr int bins = fft / 2 + 1;
  const long long span = (a.count - 1) * (long long)hop + fft;
  const unsigned tile_base = (unsigned)__cvta_generic_to_shared(tile);

  for (long long run = blockIdx.x; run < p.total_runs; run += gridDim.x) {
    const long long b = run / p.runs_per_signal;
    const long long m0 = (run - b * p.runs_per_signal) * run_len;
    const long long m1 = min(m0 + run_len, a.out_len);
    const long long q0 = m0 + a.left;
    const long long q1 = min(m1 + a.left, span);                      // positions [q0, q1) receive taps
    const float2* z = reinterpret_cast<const float2*>(a.z) + b * bins * a.frames;
    float* out = reinterpret_cast<float*>(a.out) + b * a.out_len;
    long long p_lo = 0, p_hi = -1;
    if (q1 > q0) {
      p_hi = min(a.count - 1, (q1 - 1) / hop);
      p_lo = max(0LL, ceil_div_ll(q0 - fft + 1, hop));
    }
    const int nf = (int)(p_hi - p_lo + 1);                             // <= 16 by construction

    // ---- spectrum tile: bins x nf frames, frames contiguous in global memory
    for (int i = tid; i < bins * 16; i += blockDim.x) {
      const int k = i >> 4, t = i & 15;
      if (t < nf)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(tile_base + 8u * (k * kTileStride + t)),
                     "l"(z + (long long)k * a.frames + p_lo + t) : "memory");
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();

    float2 v[32];
    const bool active = warp < nf;
    float2 r[16];
    float2 mid = make_float2(0.f, 0.f);
    if (active) {
      // lane l, register k2 < 16 holds the bin pair k = l + 32 k2 and 1024 - k
#pragma unroll
      for (int k2 = 0; k2 < 16; ++k2) {
        const int k = lane + 32 * k2, nk = kHalf - k;
        const float2 zero = make_float2(0.f, 0.f);
        v[k2] = (k & bin_mask) == 0 ? tile[(k >> bin_shift) * kTileStride + warp] : zero;
        r[k2] = (nk & bin_mask) == 0 ? tile[(nk >> bin_shift) * kTileStride + warp] : zero;
      }
      mid = tile[(512 >> bin_shift) * kTileStride + warp];
      if (lane == 0) { v[0].y = 0.0f; r[0].y = 0.0f; }                // DC and Nyquist are real
    }
    __syncthreads();                                                   // the tile becomes transpose space
    if (active) {
#pragma unroll
      for (int k2 = 0; k2 < 16; ++k2) {
        const float2 yk = v[k2], yn = r[k2];
        const float2 w = k2 == 0 ? wl
                                 : make_float2(wl.x * kW64C[k2] - wl.y * kW64S[k2],
                                               wl.x * kW64S[k2] + wl.y * kW64C[k2]);   // W_2048^k
        const float2 E = make_float2(yk.x + yn.x, yk.y - yn.y);       // Y[k] + conj Y[nk]
        const float2 O = make_float2(yk.x - yn.x, yk.y + yn.y);       // Y[k] - conj Y[nk]
        const float2 co = make_float2(w.x * O.x + w.y * O.y, w.x * O.y - w.y * O.x);    // conj(w) O
        const float2 wo = make_float2(co.x, -co.y);                                      // w conj(O)
        const float2 zk = make_float2(E.x - co.y, E.y + co.x);        // Zinv[k]
        const float2 zn = make_float2(E.x - wo.y, -E.y + wo.x);       // Zinv[1024-k]
        v[k2] = make_float2(zk.x, -zk.y);
        r[k2] = make_float2(zn.x, -zn.y);
      }
      mid = make_float2(2.0f * mid.x, 2.0f * mid.y);                  // conj(Zinv[512]) = 2 Y[512]
#pragma unroll
      for (int R = 16; R < 32; ++R) {
        const float2 own = r[31 - R];
        const float2 alt = R == 16 ? mid : r[(32 - R) & 15];
        const float sx = lane == 0 ? alt.x : own.x;
        const float sy = lane == 0 ? alt.y : own.y;
        v[R].x = __shfl_sync(0xffffffffu, sx, partner);
        v[R].y = __shfl_sync(0xffffffffu, sy, partner);
      }
      fft1024(v, ex, tw4, lane);
      // v[q] = conj(z[n]), n = lane + 32 q:  y[2n] = v.x, y[2n+1] = -v.y; window now
      // windowed frame -> this warp's (now idle) transpose buffer, natural order
      const float2* w2 = reinterpret_cast<const float2*>(sWindow);
#pragma unroll
      for (int q = 0; q < 32; ++q) {
        const float2 w = w2[lane + 32 * q];
        ex[lane + 32 * q] = make_float2(v[q].x * w.x, -v[q].y * w.y);
      }
    }
    __syncthreads();
    // ---- overlap-add as a gather: every output position sums the taps of the
    // frames that reach it, newest frame first (the order in which the
    // reference's block planes arrive, stft.ml:806-838), then the envelope
    // division, trim and zero extension (stft.ml:846-894)
    const long long head = min(span, (long long)(fft - hop));
    const long long stop = max(head, min(span, a.count * (long long)hop));
    const int n_out = (int)(m1 - m0);
    const long long full_lo = max(head, q0), full_hi = min(stop, q0 + n_out);
    const int rel0 = (int)(q0 - p_lo * hop);          // run position 0 relative to frame p_lo's tap 0
    int res = (int)((q0 + tid) % hop);
    const int rstep = (int)(blockDim.x % hop);
    // newest frame reaching position i and the tap it lands on, walked without a
    // division per sample: (tq, tj) = divmod(rel0 + i, hop), i advancing by blockDim.x
    const int tq_step = (int)(blockDim.x / hop);
    int tq = (rel0 + tid) / hop, tj = (rel0 + tid) - tq * hop;
    for (int i = tid; i < n_out; i += blockDim.x) {
      const long long q = q0 + i;
      float val = 0.0f;
      if (q < span) {
        int t = min(nf - 1, tq);
        int j = tj + (tq - t) * hop;
        float sum = 0.0f;
        const float* tap = sWork + t * kExFloats + j;
        for (; t >= 0 && j < fft; --t, j += hop, tap -= kExFloats - hop) sum += *tap;
        if (q >= full_lo && q < full_hi) {
          // every residue class reaches the position completely: tabulated reciprocal
          val = sum * sInvEnv[res];
        } else {
          const long long first = max(0LL, ceil_div_ll(q - fft + 1, hop));
          const long long last = min(a.count - 1, q / hop);
          double e = 0.0;
          for (long long pp = first; pp <= last; ++pp) {
            const double w = a.window[q - pp * hop];
            e += w * w;
          }
          if (e == 0.0) e = 1.0;
          val = (float)((double)sum / e);
        }
      }
      out[m0 + i] = val;
      res += rstep;
      if (res >= hop) res -= hop;
      tq += tq_step;
      tj += rstep;
      if (tj >= hop) { tj -= hop; ++tq; }
    }
    __syncthreads();
  }
}

}  // namespace

bool istft2048_supports(const IstftArgs& a) {
  if (a.fft < 128 || a.fft > kN || kN % a.fft != 0) return false;
  if (a.in_f64 || a.out_f64 || a.hop < 1 || a.hop > a.fft) return false;
  const int classes = (a.fft + a.hop - 1) / a.hop;
  const int run_hops = 16 - classes + (a.left % a.hop == 0 ? 1 : 0);
  if (run_hops < 1) return false;
  return true;
}

cudaError_t launch_istft2048(const IstftArgs& a, const float* window_scaled, const float2* tw_pass,
                             const float2* tw_base, long long batch, int sm_count,
                             cudaStream_t st) {
  if (batch == 0 || a.out_len == 0) return cudaSuccess;
  Istft2048Params p;
  p.a = a;
  p.window = window_scaled;
  p.tw_pass = tw_pass;
  p.tw_base = tw_base;
  p.classes = (a.fft + a.hop - 1) / a.hop;
  p.run_hops = 16 - p.classes + (a.left % a.hop == 0 ? 1 : 0);
  const long long run_len = (long long)p.run_hops * a.hop;
  p.runs_per_signal = (a.out_len + run_len - 1) / run_len;
  p.total_runs = p.runs_per_signal * batch;
  const size_t smem = (size_t)(1024 + 32) * sizeof(float2) + (size_t)kN * 4 +
                      (size_t)kWorkFloats * 4 + (size_t)a.hop * 4;
  const int grid = (int)(p.total_runs < sm_count ? p.total_runs : sm_count);
  cudaError_t e = cudaSuccess;
#define SMB_LAUNCH_ISTFT2048(STEP)                                                          \
  e = cudaFuncSetAttribute(istft2048_kernel<STEP>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                           (int)smem);                                                      \
  if (e != cudaSuccess) return e;                                                           \
  istft2048_kernel<STEP><<<grid, kWarps * 32, smem, st>>>(p);
  switch (kN / a.fft) {
    case 1: SMB_LAUNCH_ISTFT2048(1) break;
    case 2: SMB_LAUNCH_ISTFT2048(2) break;
    case 4: SMB_LAUNCH_ISTFT2048(4) break;
    case 8: SMB_LAUNCH_ISTFT2048(8) break;
    case 16: SMB_LAUNCH_ISTFT2048(16) break;
    default: return cudaErrorInvalidConfiguration;
  }
#undef SMB_LAUNCH_ISTFT2048
  ++g_launch_count;
  return cudaGetLastError();
}

}  // namespace smb
