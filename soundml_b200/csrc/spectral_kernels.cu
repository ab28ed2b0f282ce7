// Per-frame spectral descriptors (librosa 0.11 feature.spectral_centroid, _bandwidth,
// _rolloff and _flatness) of a non-negative magnitude spectrogram S [batch, bins, frames],
// with f_k = k * bin_hz (numpy rfftfreq's arithmetic) and L = sum_k S_k, taken as 1 when
// below the smallest normal number of S's type (librosa util.normalize, fill=None):
//
//   centroid  c  = sum_k f_k S_k / L
//   bandwidth    = (sum_k S'_k |f_k - c|^p)^(1/p),  S' = S / L (norm) or S
//   rolloff      = f_k of the first k with !(cum_k < thr): cum_k = S_0 + ... + S_k added
//                  in order in S's precision, thr = T(roll_percent) * cum_(bins-1)
//   flatness     = exp(mean_k ln m_k) / mean_k m_k,  m_k = max(amin, S_k^power)
//
// One thread owns one (clip, frame); consecutive threads take consecutive frames, so each
// bin row is one coalesced load per warp.  Pass 1 reads every element once and sums, in
// double, L, sum_k k S_k (exact products for float32: f_k's factor bin_hz is applied once
// at the end) and flatness's sum_k ln m_k and sum_k m_k (each m_k in double: exact for
// float32 S at power 1 and 2).  It also carries rolloff's sequential sum in S's type and
// stores it in shared memory at the end of every chunk of `chunk` bins.  Once the total is
// known, rolloff re-walks only the first chunk whose end reaches the threshold, from the
// checkpoint before it: the same additions in the same order, so the same bits as the full
// walk.  For S >= 0 the running sum never decreases, so that chunk holds the crossing; a
// NaN total makes chunk 0 the answer, as the literal rule does (no comparison with NaN
// holds).  Negative S is outside the domain: there the first crossing may lie in an
// earlier chunk, and a frame that never reaches the threshold gives NaN (librosa's nanmin
// of nothing).  Pass 2, only for the bandwidth, re-reads the frame's bins and sums
// S_k |f_k - c|^p in double (DESIGN.md 4.10 has why the moment form is not used).
#include <cfloat>

#include "../../include/soundml_b200.h"
#include "kernels.h"

namespace smb {

namespace {

// Threads per CTA: a build parameter so that other sizes can be measured
// (build.py -DSMB_SPECTRAL_THREADS=256 --out=...; DESIGN.md 4.10).
#ifndef SMB_SPECTRAL_THREADS
#define SMB_SPECTRAL_THREADS 128
#endif
constexpr int kThreads = SMB_SPECTRAL_THREADS;
// Bins each thread loads before it adds any of them: the loads of one batch are in flight
// together, which a walk of dependent sums would otherwise serialise.  A build parameter
// (-DSMB_SPECTRAL_LOADS=8; DESIGN.md 4.10); it divides kChunk, so checkpoints fall between
// batches.
#ifndef SMB_SPECTRAL_LOADS
#define SMB_SPECTRAL_LOADS 16
#endif
constexpr int kLoads = SMB_SPECTRAL_LOADS;
constexpr int kChunk = 32;                         // bins between rolloff checkpoints (at least)
static_assert(kChunk % kLoads == 0, "whole load batches fill every chunk but the last");
constexpr size_t kCheckpointBytes = 48 << 10;      // checkpoints of one CTA: no opt-in needed

template <typename T> struct Tiny;
template <> struct Tiny<float> { static constexpr double value = FLT_MIN; };
template <> struct Tiny<double> { static constexpr double value = DBL_MIN; };

// x^p with numpy's exact forms of the default exponents
__device__ __forceinline__ double raise(double x, double p) {
  return p == 2.0 ? x * x : p == 1.0 ? x : pow(x, p);
}
// y^(1/p): numpy's ** 0.5 is sqrt, ** 1.0 the identity
__device__ __forceinline__ double root(double y, double p) {
  return p == 2.0 ? sqrt(y) : p == 1.0 ? y : pow(y, 1.0 / p);
}

// body(k, S_k) for k in [k0, k1) in order, the loads issued kLoads at a time
template <typename T, typename Body>
__device__ __forceinline__ void walk(const T* __restrict__ col, long long F, long long k0, long long k1,
                                     Body&& body) {
  long long k = k0;
  for (; k + kLoads <= k1; k += kLoads) {
    T v[kLoads];
#pragma unroll
    for (int u = 0; u < kLoads; ++u) v[u] = __ldg(col + (k + u) * F);
#pragma unroll
    for (int u = 0; u < kLoads; ++u) body(k + u, v[u]);
  }
  for (; k < k1; ++k) body(k, __ldg(col + k * F));
}

template <typename T>
__global__ void __launch_bounds__(kThreads) spectral_kernel(const SpectralArgs a, long long chunk) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* checkpoint = reinterpret_cast<T*>(smem_raw);   // [chunks][kThreads]
  const long long i = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (i >= a.batch * a.frames) return;
  const long long F = a.frames, bins = a.bins;
  const long long b = i / F, f = i - b * F;
  const T* col = static_cast<const T*>(a.s) + b * bins * F + f;
  const bool flat = a.what & SMB_SPECTRAL_FLATNESS, roll = a.what & SMB_SPECTRAL_ROLLOFF;

  double len = 0.0, moment = 0.0, log_sum = 0.0, m_sum = 0.0;
  T cum = T(0);
  for (long long k0 = 0, j = 0; k0 < bins; k0 += chunk, ++j) {
    walk(col, F, k0, min(k0 + chunk, bins), [&](long long k, T s) {
      const double sd = (double)s;
      len += sd;
      moment += (double)k * sd;
      cum += s;
      if (flat) {
        double m = raise(sd, a.power);
        m = m < a.amin ? a.amin : m;                // keeps a NaN, as np.maximum does
        log_sum += log(m);
        m_sum += m;
      }
    });
    if (roll) checkpoint[j * kThreads + threadIdx.x] = cum;
  }

  const double scale = len < Tiny<T>::value ? 1.0 : len;
  const double c = moment * a.bin_hz / scale;
  T* out = static_cast<T*>(a.out) + b * (long long)__popc(a.what) * F + f;
  if (a.what & SMB_SPECTRAL_CENTROID) {
    *out = T(c);
    out += F;
  }
  if (a.what & SMB_SPECTRAL_BANDWIDTH) {
    double acc = 0.0;
    walk(col, F, 0, bins, [&](long long k, T s) {
      acc += (double)s * raise(fabs((double)k * a.bin_hz - c), a.p);
    });
    if (a.norm) acc /= scale;
    *out = T(root(acc, a.p));
    out += F;
  }
  if (roll) {
    const T thr = T(a.roll_percent) * cum;
    const long long chunks = (bins + chunk - 1) / chunk;
    long long j = 0;
    while (j < chunks && checkpoint[j * kThreads + threadIdx.x] < thr) ++j;
    double freq = NAN;
    if (j < chunks) {
      T run = j ? checkpoint[(j - 1) * kThreads + threadIdx.x] : T(0);
      const long long k1 = min((j + 1) * chunk, bins);
      long long k = j * chunk;
      for (; k < k1; ++k) {
        run += col[k * F];
        if (!(run < thr)) break;
      }
      if (k < k1) freq = (double)k * a.bin_hz;
    }
    *out = T(freq);
    out += F;
  }
  if (flat) *out = T(exp(log_sum / (double)bins) / (m_sum / (double)bins));
}

template <typename T>
cudaError_t launch_typed(const SpectralArgs& a, cudaStream_t st) {
  // checkpoint spacing: kChunk bins, or a multiple of it when the CTA's checkpoints at that
  // spacing would pass kCheckpointBytes
  const long long cap = (long long)(kCheckpointBytes / (kThreads * sizeof(T)));
  const long long base = (a.bins + kChunk - 1) / kChunk;
  const long long chunk = kChunk * ((base + cap - 1) / cap);
  const size_t smem = (a.what & SMB_SPECTRAL_ROLLOFF)
                          ? (size_t)((a.bins + chunk - 1) / chunk) * kThreads * sizeof(T) : 0;
  const long long blocks = (a.batch * a.frames + kThreads - 1) / kThreads;
  if (blocks > 2147483647LL) return cudaErrorInvalidConfiguration;
  spectral_kernel<T><<<(unsigned)blocks, kThreads, smem, st>>>(a, chunk);
  return cudaSuccess;
}

}  // namespace

cudaError_t launch_spectral(const SpectralArgs& a, cudaStream_t st) {
  if (a.batch == 0 || a.frames == 0) return cudaSuccess;
  const cudaError_t e = a.f64 ? launch_typed<double>(a, st) : launch_typed<float>(a, st);
  if (e != cudaSuccess) return e;
  ++g_launch_count;
  return cudaGetLastError();
}

}  // namespace smb
