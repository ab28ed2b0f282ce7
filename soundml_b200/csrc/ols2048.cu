// Overlap-save stage with block length N = 2048, one warp per block (sm_100a).
//
// Same filter and block geometry as ols_kernels.cu (reference: resample.ml:279-300,
// 1309-1319, 1456-1599; spectrum shaping resample_stubs.c:329-372), specialised
// to block length 2048: what the planner picks for 44.1 -> 22.05 kHz (K = 190),
// and what this build picks for every decimating stage whose filter fits (any M:
// 48 -> 16 kHz is /3) and for FIRs of up to 1025 taps.  Plain (L = M = 1), /M and
// xL stages; an interpolating stage runs as its L polyphase branches
// y[jL + p] = sum_t x[j + K - t] g_p[t], g_p[t] = h[p + tL] -- L plain filters at
// the input rate, one (block, branch) pair per warp, each with its own spectrum.
//
// A warp owns a block from the first load to the last store -- no CTA-level
// synchronisation, so the 16 warps of an SM drift apart and overlap each other's
// memory and FMA phases:
//   * z[n] = x[2n] + i x[2n+1] is read straight from global memory (blocks
//     overlap by only 2K samples, L2 absorbs the re-reads), transformed as
//     32 x 32 with the register fft32 of the fused STFT kernel and one padded
//     shared-memory transpose;
//   * the real-input split pairs bin k with 1024-k by warp shuffle; each lane
//     multiplies its 16 pairs by the plan spectrum;
//   * the inverse runs at the full length 2048 -- Zinv[k] = (Y[k] + conj Y[1024-k])
//     + i W^-k (Y[k] - conj Y[1024-k]), forward FFT of conj(Zinv) -- through the same
//     32 x 32 machinery; a /M stage keeps every M-th sample, which is exactly the
//     reference's alias fold onto N/M bins followed by the short inverse (the 1/M
//     and 1/W weights are folded into the plan spectrum on the host);
//   * block b writes outputs (hi(b-1), hi(b)], as in the reference.
#include <cstdint>

#include "fft32.cuh"
#include "kernels.h"

namespace smb {

namespace {

using namespace fft32impl;

constexpr int kN = 2048;
constexpr int kHalf = 1024;
constexpr int kWarps = 16;
constexpr int kExFloats = 32 * kFft1024ExStride * 2;   // per-warp transpose buffer

__device__ __forceinline__ float2 cmulf(float2 a, float2 b) {
  return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}

struct Ols2048Params {
  OlsArgs a;
  const float2* tw_pass;     // [32][32]  W_1024^(k1 n2)
  const float2* tw_base;     // [32]      W_2048^l
  long long total_blocks;
};

__global__ void __launch_bounds__(kWarps * 32, 1)
ols2048_kernel(const Ols2048Params p) {
  extern __shared__ __align__(16) float smem[];
  float2* sTwPass = reinterpret_cast<float2*>(smem);          // [16][32][2] pairs (k1, k1+1) per lane
  float2* sTwBase = sTwPass + 1024;                           // [32]
  float2* sH = sTwBase + 32;                                  // [L][1025 (+1)] plan spectra x 1/2
  float* sEx = reinterpret_cast<float*>(sH + 1026 * p.a.L);   // [16 warps][32][34] complex
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < 1024; i += blockDim.x) {
    const int l = i & 31, k1 = i >> 5;
    sTwPass[(((k1 >> 1) * 32 + l) << 1) + (k1 & 1)] = p.tw_pass[i];
  }
  if (tid < 32) sTwBase[tid] = p.tw_base[tid];
  // the real split below yields 2 X[k]: the missing 1/2 rides on the spectrum
  for (int i = tid; i < 1025 * p.a.L; i += blockDim.x) {
    const int ph = i / 1025, k = i - ph * 1025;
    const float2 h = p.a.H[i];
    sH[ph * 1026 + k] = make_float2(0.5f * h.x, 0.5f * h.y);
  }
  __syncthreads();

  const OlsArgs& a = p.a;
  float2* ex = reinterpret_cast<float2*>(sEx + warp * kExFloats);
  const float4* tw4 = reinterpret_cast<const float4*>(sTwPass);
  const float2 wl = sTwBase[lane];
  const int partner = (32 - lane) & 31;
  const long long wstride = (long long)gridDim.x * kWarps;

  for (long long id = (long long)blockIdx.x * kWarps + warp; id < p.total_blocks; id += wstride) {
    // work item = (signal c, block b, polyphase branch ph)
    const long long cb = id / a.L;
    const int ph = (int)(id - cb * a.L);
    const long long c = cb / a.blocks;
    const long long b = cb - c * a.blocks;
    const float* xs = a.x + c * a.n;
    float* out = a.out + c * a.n_out;
    const float2* sHp = sH + ph * 1026;

    // ---- block b reads stage inputs [b B - 2K - delta, +2048), zeros outside the signal
    const long long start = b * a.B - 2LL * a.K - a.delta;
    float2 v[32];
    if (start >= 0 && start + kN <= a.n) {
      const float* src = xs + start + 2 * lane;
      if ((reinterpret_cast<uintptr_t>(src) & 7) == 0) {
#pragma unroll
        for (int n1 = 0; n1 < 32; ++n1) v[n1] = __ldg(reinterpret_cast<const float2*>(src + 64 * n1));
      } else {
#pragma unroll
        for (int n1 = 0; n1 < 32; ++n1) v[n1] = make_float2(__ldg(src + 64 * n1), __ldg(src + 64 * n1 + 1));
      }
    } else {
#pragma unroll
      for (int n1 = 0; n1 < 32; ++n1) {
        const long long s = start + 64 * n1 + 2 * lane;
        v[n1].x = (s >= 0 && s < a.n) ? __ldg(xs + s) : 0.0f;
        v[n1].y = (s + 1 >= 0 && s + 1 < a.n) ? __ldg(xs + s + 1) : 0.0f;
      }
    }
    fft1024(v, ex, tw4, lane);

    // ---- real split, spectrum product, inverse pre-twiddle.  Lane l, register k2
    // < 16 handles the bin pair k = l + 32 k2 and 1024 - k.
    float2 r[16];
#pragma unroll
    for (int k2 = 0; k2 < 16; ++k2) {
      // lanes != 0 need the partner's register 31-k2; lane 0 pairs with itself
      // through register (32-k2) mod 32.
      const float2 own = v[31 - k2];
      const float2 alt = v[(32 - k2) & 31];
      const float sx = lane == 0 ? alt.x : own.x;
      const float sy = lane == 0 ? alt.y : own.y;
      r[k2].x = __shfl_sync(0xffffffffu, sx, partner);
      r[k2].y = __shfl_sync(0xffffffffu, sy, partner);
    }
    // lane 0 only: bin 512 pairs with itself; Zinv[512] = 2 conj(Y[512]), kept conjugated
    float2 mid;
    {
      const float2 xm = make_float2(2.0f * v[16].x, -2.0f * v[16].y);   // 2 X[512]
      const float2 ym = cmulf(xm, sHp[512]);
      mid = make_float2(2.0f * ym.x, 2.0f * ym.y);                       // conj(2 conj(Y)) = 2 Y
    }
#pragma unroll
    for (int k2 = 0; k2 < 16; ++k2) {
      const float2 A = v[k2];
      const float2 S = make_float2(A.x + r[k2].x, A.y - r[k2].y);
      const float2 D = make_float2(A.x - r[k2].x, A.y + r[k2].y);
      const float2 w = k2 == 0 ? wl
                               : make_float2(wl.x * kW64C[k2] - wl.y * kW64S[k2],
                                             wl.x * kW64S[k2] + wl.y * kW64C[k2]);   // W_2048^k
      const float tr = w.x * D.y + w.y * D.x;
      const float ti = w.y * D.y - w.x * D.x;
      const float2 xk = make_float2(S.x + tr, S.y + ti);      // 2 X[k]
      const float2 xn = make_float2(S.x - tr, ti - S.y);      // 2 X[1024-k]
      const int k = lane + 32 * k2;
      const float2 yk = cmulf(xk, sHp[k]);                    // Y[k]
      const float2 yn = cmulf(xn, sHp[kHalf - k]);            // Y[1024-k]
      // E = Y[k] + conj Y[nk], O = Y[k] - conj Y[nk]
      const float2 E = make_float2(yk.x + yn.x, yk.y - yn.y);
      const float2 O = make_float2(yk.x - yn.x, yk.y + yn.y);
      // Zinv[k] = E + i conj(w) O ;  Zinv[nk] = conj(E) + i w conj(O)
      //   (W^-(1024-k) = -w and Y[nk] - conj Y[k] = -conj(O))
      const float2 co = make_float2(w.x * O.x + w.y * O.y, w.x * O.y - w.y * O.x);    // conj(w) O
      const float2 wo = make_float2(w.x * O.x + w.y * O.y, -(w.x * O.y - w.y * O.x)); // w conj(O)
      const float2 zk = make_float2(E.x - co.y, E.y + co.x);
      const float2 zn = make_float2(E.x - wo.y, -E.y + wo.x);
      v[k2] = make_float2(zk.x, -zk.y);                       // conj: forward FFT gives conj(z)
      r[k2] = make_float2(zn.x, -zn.y);                       // belongs to lane 32-l, register 31-k2
    }
    // move the 1024-k halves into place: lane L, register R in [16, 32) takes the
    // value lane (32-L) mod 32 computed for k2 = 31-R (k2 = 32-R when L = 0)
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
    // v[q] = conj(z[n]), n = lane + 32 q:  y[2n] = v.x,  y[2n+1] = -v.y

    // ---- block b extends the output run to hi(b) (resample.ml:1309-1319)
    const long long num = b * a.B + kN - 3LL * a.K - a.delta - 1;
    long long hi = num >= 0 ? num / a.M : -1;
    const long long prev = (b - 1) * a.B + kN - 3LL * a.K - a.delta - 1;
    const long long lo = (b == 0 || prev < 0) ? 0 : prev / a.M + 1;
    if (hi >= a.n_out) hi = a.n_out - 1;
    // output i sits at full-rate block position i M + cpos (cpos divisible by M)
    const long long cpos = 3LL * a.K + a.delta - b * a.B;
    if (a.L > 1) {
      // interpolating stage: branch ph of input-rate sample j lands on j L + ph
      const long long hi_j = min(b * a.B + kN - 3LL * a.K - 1, a.n - 1);
      const long long lo_j = b == 0 ? 0 : (b - 1) * a.B + kN - 3LL * a.K;
#pragma unroll
      for (int q = 0; q < 32; ++q) {
        const long long j = 2LL * (lane + 32 * q) - cpos;
        if (j >= lo_j && j <= hi_j) out[j * a.L + ph] = v[q].x;
        if (j + 1 >= lo_j && j + 1 <= hi_j) out[(j + 1) * a.L + ph] = -v[q].y;
      }
    } else if (a.M == 1) {
      const bool vec = ((cpos & 1) == 0) && ((reinterpret_cast<uintptr_t>(out) & 7) == 0);
#pragma unroll
      for (int q = 0; q < 32; ++q) {
        const long long i = 2LL * (lane + 32 * q) - cpos;
        const float y0 = v[q].x, y1 = -v[q].y;
        if (vec && i >= lo && i + 1 <= hi) {
          *reinterpret_cast<float2*>(out + i) = make_float2(y0, y1);
        } else {
          if (i >= lo && i <= hi) out[i] = y0;
          if (i + 1 >= lo && i + 1 <= hi) out[i + 1] = y1;
        }
      }
    } else if (a.M == 2) {
      const long long half_c = cpos / 2;          // cpos is even
#pragma unroll
      for (int q = 0; q < 32; ++q) {
        const long long i = (long long)(lane + 32 * q) - half_c;
        if (i >= lo && i <= hi) out[i] = v[q].x;
      }
    } else {
      // any other M: lay the block out in the (now idle) transpose buffer and let
      // consecutive lanes pick consecutive outputs, i.e. every M-th sample
      float2* yb2 = ex;
#pragma unroll
      for (int q = 0; q < 32; ++q) yb2[lane + 32 * q] = make_float2(v[q].x, -v[q].y);
      __syncwarp();
      const float* yb = reinterpret_cast<const float*>(ex);
      const long long ibase = -cpos / a.M;                    // exact: M divides cpos
      const long long i_first = max(lo, ibase);
      const long long i_last = min(hi, ibase + (kN - 1) / a.M);
      for (long long i = i_first + lane; i <= i_last; i += 32)
        out[i] = yb[(int)(i - ibase) * a.M];
    }
    __syncwarp();
  }
}

}  // namespace

bool ols2048_supports(const OlsArgs& a) {
  if (a.N != kN || a.B < 1 || 2 * a.K + a.delta >= kN) return false;
  if (a.L > 1) return a.M == 1 && a.delta == 0 && a.L <= 8 && a.polyphase;
  return a.M >= 1 && a.B % a.M == 0 && (3 * a.K + a.delta) % a.M == 0;
}

cudaError_t launch_ols2048(const OlsArgs& a, const float2* tw_pass, const float2* tw_base,
                           long long batch, int sm_count, cudaStream_t st) {
  if (batch == 0 || a.n_out == 0 || a.blocks == 0) return cudaSuccess;
  Ols2048Params p;
  p.a = a;
  p.tw_pass = tw_pass;
  p.tw_base = tw_base;
  p.total_blocks = a.blocks * batch * a.L;
  const size_t smem = (size_t)(1024 + 32 + 1026 * a.L) * sizeof(float2) +
                      (size_t)kWarps * kExFloats * 4;
  cudaError_t e = cudaFuncSetAttribute(ols2048_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem);
  if (e != cudaSuccess) return e;
  const long long want = (p.total_blocks + kWarps - 1) / kWarps;
  const int grid = (int)(want < sm_count ? want : sm_count);
  ols2048_kernel<<<grid, kWarps * 32, smem, st>>>(p);
  ++g_launch_count;
  return cudaGetLastError();
}

}  // namespace smb
