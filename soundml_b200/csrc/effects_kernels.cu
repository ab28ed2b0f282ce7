// Phase vocoder (librosa 0.11 phase_vocoder, the reference's Effects.time_stretch
// stage between Stft.transform and Stft.invert) on the GPU.
//
// Output frame t reads source position s_t = t * rate (double, as np.arange), with
// i_t = floor(s_t), alpha_t = s_t - i_t, and two all-zero frames past the end:
//
//   |out[t]|   = (1 - alpha_t) |D[i_t]| + alpha_t |D[i_t + 1]|
//   arg out[t] = theta[i_(t-1) + 1] + sum_{u=1}^{t-1} (theta[i_(u-1) + 1] - theta[i_u])   (mod 2 pi)
//
// with theta = arg D.  The expected phase advance of librosa's recurrence cancels
// modulo 2 pi, so the accumulated phase carries only the gap terms, and every one of
// them is exactly zero where the walk steps by one frame: at rate 1 the phase is
// theta[t].  Nothing here grows with the absolute phase (DESIGN.md 4.8).
//
// One warp owns one row (clip, bin), contiguous in time, and walks it in tiles of
// kTile output frames.  The tile's source frames are staged once in shared memory as
// (|D|, theta), so outputs that share a frame (rate < 1) share its atan2 / hypot;
// the gap terms are summed by a warp scan in double whose carry crosses the tiles.
// Stores are coalesced: lane l writes outputs t0 + 32 k + l.
#include "kernels.h"

namespace smb {

namespace {

constexpr int kWarps = 8;              // rows per CTA, one per warp
constexpr int kPer = 4;                // outputs per lane per tile
constexpr int kTile = 32 * kPer;       // outputs per tile
constexpr int kStage = 3 * kTile;      // staged source frames per warp: covers rate <= 3
constexpr double kTwoPi = 6.283185307179586476925286766559;
constexpr unsigned kFull = 0xffffffffu;

template <typename T> struct Cplx;
template <> struct Cplx<float> { using type = float2; };
template <> struct Cplx<double> { using type = double2; };

__device__ __forceinline__ void polar(float2 v, float& m, float& th) {
  m = hypotf(v.x, v.y);
  th = atan2f(v.y, v.x);
}
__device__ __forceinline__ void polar(double2 v, double& m, double& th) {
  m = hypot(v.x, v.y);
  th = atan2(v.y, v.x);
}
__device__ __forceinline__ void sincos_(float a, float* s, float* c) { sincosf(a, s, c); }
__device__ __forceinline__ void sincos_(double a, double* s, double* c) { sincos(a, s, c); }

// frame f of a row; frames at and past `frames` are the zero padding
template <typename T>
__device__ __forceinline__ void frame_polar(const typename Cplx<T>::type* row, long long frames,
                                            long long f, T& m, T& th) {
  if (f < frames) {
    polar(row[f], m, th);
  } else {
    m = T(0);
    th = T(0);
  }
}

__device__ __forceinline__ long long src_floor(long long t, double rate) {
  return (long long)floor((double)t * rate);
}

template <typename T>
__global__ void __launch_bounds__(32 * kWarps)
phase_vocoder_kernel(const typename Cplx<T>::type* __restrict__ z,
                     typename Cplx<T>::type* __restrict__ out, long long rows, long long frames,
                     long long out_frames, double rate) {
  using C = typename Cplx<T>::type;
  __shared__ T sm_mag[kWarps][kStage];
  __shared__ T sm_th[kWarps][kStage];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * kWarps + warp;
  if (row >= rows) return;
  const C* zr = z + row * frames;
  C* orow = out + row * out_frames;
  T* mag = sm_mag[warp];
  T* th = sm_th[warp];
  double carry = 0.0;   // sum of the gap terms of the tiles before, reduced modulo 2 pi
  for (long long t0 = 0; t0 < out_frames; t0 += kTile) {
    const long long tlast = min(t0 + kTile, out_frames) - 1;
    const long long lo = t0 == 0 ? 0 : min(src_floor(t0, rate), src_floor(t0 - 1, rate) + 1);
    const long long span = src_floor(tlast, rate) + 2 - lo;
    const bool staged = span <= kStage;
    if (staged) {
      // every source frame of the tile once: loads first, then atan2 / hypot
      C v[kStage / 32];
#pragma unroll
      for (int c = 0; c < kStage / 32; ++c) {
        const long long f = lo + c * 32 + lane;
        v[c] = c * 32 + lane < span && f < frames ? zr[f] : C{};
      }
#pragma unroll
      for (int c = 0; c < kStage / 32; ++c) {
        const int j = c * 32 + lane;
        if (j < span) polar(v[c], mag[j], th[j]);
      }
      __syncwarp();
    }
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      const long long t = t0 + 32 * k + lane;
      const bool valid = t <= tlast;
      double g = 0.0, alpha = 0.0;
      T m0 = T(0), m1 = T(0), thp = T(0);
      if (valid) {
        const double s = (double)t * rate;
        const long long i = (long long)floor(s);
        alpha = s - (double)i;
        const long long ip = t == 0 ? 0 : src_floor(t - 1, rate) + 1;   // i_(t-1) + 1
        T thi;
        if (staged) {
          m0 = mag[i - lo];
          m1 = mag[i + 1 - lo];
          thi = th[i - lo];
          thp = th[ip - lo];
        } else {
          T unused;
          frame_polar<T>(zr, frames, i, m0, thi);
          frame_polar<T>(zr, frames, i + 1, m1, unused);
          frame_polar<T>(zr, frames, ip, unused, thp);
        }
        if (t > 0) g = (double)thp - (double)thi;    // exactly 0 when ip == i
      }
      // inclusive scan of the gap terms; the exclusive sum is the lane below's
      double incl = g;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const double o = __shfl_up_sync(kFull, incl, d);
        if (lane >= d) incl += o;
      }
      double excl = __shfl_up_sync(kFull, incl, 1);
      if (lane == 0) excl = 0.0;
      if (valid) {
        double ph = (double)thp + (carry + excl);
        ph -= kTwoPi * rint(ph * (1.0 / kTwoPi));
        const T mg = (T)((1.0 - alpha) * (double)m0 + alpha * (double)m1);
        T sn, cs;
        sincos_((T)ph, &sn, &cs);
        C o;
        o.x = mg * cs;
        o.y = mg * sn;
        orow[t] = o;
      }
      carry += __shfl_sync(kFull, incl, 31);
      carry -= kTwoPi * rint(carry * (1.0 / kTwoPi));
    }
    __syncwarp();      // the next tile overwrites the staged frames
  }
}

}  // namespace

cudaError_t launch_phase_vocoder(const PhaseVocoderArgs& a, cudaStream_t st) {
  if (a.rows == 0 || a.out_frames == 0) return cudaSuccess;
  const long long blocks = (a.rows + kWarps - 1) / kWarps;
  if (blocks > 2147483647LL) return cudaErrorInvalidConfiguration;
  if (a.f64)
    phase_vocoder_kernel<double><<<(unsigned)blocks, 32 * kWarps, 0, st>>>(
        (const double2*)a.z, (double2*)a.out, a.rows, a.frames, a.out_frames, a.rate);
  else
    phase_vocoder_kernel<float><<<(unsigned)blocks, 32 * kWarps, 0, st>>>(
        (const float2*)a.z, (float2*)a.out, a.rows, a.frames, a.out_frames, a.rate);
  ++g_launch_count;
  return cudaGetLastError();
}

}  // namespace smb
