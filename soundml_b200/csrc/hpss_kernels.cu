// Harmonic-percussive separation (librosa 0.11 decompose.hpss) on the GPU.
//
// harm = median over win_harm frames along the frame axis, perc = median over win_perc
// bins along the bin axis, both under scipy's mode="reflect" (half-sample symmetric,
// any number of wraps); the median of w values is element floor(w / 2) of the sorted
// window (the upper median for even w), a pure selection and so exact.  The masks are
// librosa.util.softmask in the input's precision:
//
//   mask_harm = softmask(harm, perc * margin_harm),  mask_perc = softmask(perc, harm * margin_perc)
//
// and the outputs S * mask (real input) or (S * mask) * phase (complex input, librosa
// magphase).  Two kernels compute the same values:
//
// hpss_tile_kernel (both windows <= kHpssFastWindow): one CTA owns a tile of kTileB bins
// x kTileF frames of one clip.  It stages the tile's magnitudes with their halos in
// shared memory, then each thread walks a run of kRun outputs along one axis with its
// window kept sorted in registers: the sorted array has kK slots, the window padded with
// the smallest key below and the largest above so that its median always sits in slot
// kMid, and one step
// removes the outgoing value and inserts the incoming one with fixed compare/select
// sweeps (no dynamic register index).  The harmonic medians go to shared memory; the
// threads that walk the percussive medians then evaluate both masks and write the tile.
//
// hpss_exact_kernel (any window, e.g. longer than the axis): one thread per output,
// each median by counting ranks over its window read from global memory.
#include <algorithm>
#include <cfloat>

#include "../../include/soundml_b200.h"
#include "kernels.h"

namespace smb {

namespace {

constexpr int kK = (int)kHpssFastWindow;   // sorted slots per window
constexpr int kMid = kK / 2;               // the slot the median of any w <= kK lands in
// Bins = frames of a tile: a build parameter so that other tiles can be measured
// (build.py -DSMB_HPSS_TILE=32 --out=...; DESIGN.md 4.9).  128 fits float32 only.
#ifndef SMB_HPSS_TILE
#define SMB_HPSS_TILE 64
#endif
constexpr int kTileB = SMB_HPSS_TILE, kTileF = SMB_HPSS_TILE;
constexpr int kRun = SMB_HPSS_TILE / 2;    // outputs one thread walks per median
constexpr int kThreads = kTileB * kTileF / kRun;
constexpr int kHarmPitch = kTileF + 1;     // odd: lanes on consecutive rows hit distinct banks
static_assert(kThreads == 2 * kTileB && kThreads == 2 * kTileF, "two runs per row and per column");

template <typename T> struct Num;
template <> struct Num<float> {
  using C = float2;
  static constexpr float tiny = FLT_MIN;
};
template <> struct Num<double> {
  using C = double2;
  static constexpr double tiny = DBL_MIN;
};

// The integer key of a value in np.sort's order: every NaN above +inf (and all NaNs
// equal), zeros of either sign in their IEEE order.  Integer min / max / compare keep a
// NaN in its place, where float min / max would drop it; the key maps back exactly.
template <typename T> struct Bits;
template <> struct Bits<float> {
  using U = unsigned int;
  static constexpr U top = 0x80000000u;
  static __device__ __forceinline__ U of(float x) { return __float_as_uint(x); }
  static __device__ __forceinline__ float from(U b) { return __uint_as_float(b); }
};
template <> struct Bits<double> {
  using U = unsigned long long;
  static constexpr U top = 0x8000000000000000ull;
  static __device__ __forceinline__ U of(double x) { return (U)__double_as_longlong(x); }
  static __device__ __forceinline__ double from(U b) { return __longlong_as_double((long long)b); }
};
template <typename T>
__device__ __forceinline__ typename Bits<T>::U order_key(T x) {
  using U = typename Bits<T>::U;
  if (isnan(x)) return ~U(0);
  const U b = Bits<T>::of(x);
  return (b & Bits<T>::top) ? ~b : (b | Bits<T>::top);
}
template <typename T>
__device__ __forceinline__ T from_key(typename Bits<T>::U k) {
  return Bits<T>::from((k & Bits<T>::top) ? (k & ~Bits<T>::top) : ~k);
}

__device__ __forceinline__ float hypot_(float x, float y) { return hypotf(x, y); }
__device__ __forceinline__ double hypot_(double x, double y) { return hypot(x, y); }
__device__ __forceinline__ float pow_(float x, float p) { return powf(x, p); }
__device__ __forceinline__ double pow_(double x, double p) { return pow(x, p); }

// scipy mode="reflect": m = q mod 2n, index m < n ? m : 2n - 1 - m
__device__ __forceinline__ long long hpss_reflect(long long q, long long n) {
  if (q >= 0 && q < n) return q;
  long long m = q % (2 * n);
  if (m < 0) m += 2 * n;
  return m < n ? m : 2 * n - 1 - m;
}

// |s[i]|: the value itself for real input, hypot(re, im) for complex (numpy's abs)
template <typename T>
__device__ __forceinline__ T magnitude(const void* s, long long i, int cplx) {
  if (!cplx) return static_cast<const T*>(s)[i];
  const typename Num<T>::C v = static_cast<const typename Num<T>::C*>(s)[i];
  return hypot_(v.x, v.y);
}

// (x / z)^p as numpy evaluates `a ** p` for an array a: squares and square roots are
// the correctly rounded operations numpy's scalar-power shortcut uses
template <typename T>
__device__ __forceinline__ T ratio_pow(T x, double p) {
  if (p == 2.0) return x * x;
  if (p == 1.0) return x;
  if (p == 0.5) return sqrt(x);
  return pow_(x, (T)p);
}

// librosa.util.softmask(x, xr, power=p, split_zeros=split)
template <typename T>
__device__ __forceinline__ T softmask(T x, T xr, double p, bool split) {
  if (isinf(p)) return x > xr ? T(1) : T(0);
  const T z = x > xr || isnan(x) ? x : xr;        // np.maximum: NaN wins
  if (z < Num<T>::tiny) return split ? T(0.5) : T(0);
  const T a = ratio_pow(x / z, p), b = ratio_pow(xr / z, p);
  return a / (a + b);
}

// Both masks of one element and the outputs `what` asks for.  cell is the element's
// offset inside its clip's [bins, frames] plane; mag its magnitude S.
template <typename T>
__device__ __forceinline__ void emit(const HpssArgs& a, long long b, long long cell, T mag, T harm,
                                     T perc) {
  const bool split = a.margin_harm == 1.0 && a.margin_perc == 1.0;
  const T mh = softmask(harm, perc * (T)a.margin_harm, a.power, split);
  const T mp = softmask(perc, harm * (T)a.margin_perc, a.power, split);
  const long long plane = a.bins * a.frames;
  const int parts = a.what == SMB_HPSS_BOTH || a.what == SMB_HPSS_MASKS ? 2 : 1;
  const long long o = b * parts * plane + cell;
  if (a.what == SMB_HPSS_MASKS) {
    static_cast<T*>(a.out)[o] = mh;
    static_cast<T*>(a.out)[o + plane] = mp;
    return;
  }
  const T m0 = a.what == SMB_HPSS_PERCUSSIVE ? mp : mh;
  if (!a.complex_in) {
    static_cast<T*>(a.out)[o] = mag * m0;
    if (parts == 2) static_cast<T*>(a.out)[o + plane] = mag * mp;
    return;
  }
  // librosa magphase: phase = (re / S' + [S == 0], im / S'), S' = S + [S == 0]
  using C = typename Num<T>::C;
  const C d = static_cast<const C*>(a.s)[b * plane + cell];
  const bool zero = mag == T(0);
  const T den = mag + (zero ? T(1) : T(0));
  const T pr = d.x / den + (zero ? T(1) : T(0)), pi = d.y / den;
  const T v0 = mag * m0;
  static_cast<C*>(a.out)[o] = C{v0 * pr, v0 * pi};
  if (parts == 2) {
    const T v1 = mag * mp;
    static_cast<C*>(a.out)[o + plane] = C{v1 * pr, v1 * pi};
  }
}

// kK keys sorted ascending in registers (bitonic network, compile-time indices)
template <typename U>
__device__ __forceinline__ void sort_slots(U (&v)[kK]) {
#pragma unroll
  for (int k = 2; k <= kK; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll
      for (int i = 0; i < kK; ++i) {
        const int l = i ^ j;
        if (l > i) {
          const U x = v[i], y = v[l];
          const bool up = (i & k) == 0;
          v[i] = up ? min(x, y) : max(x, y);
          v[l] = up ? max(x, y) : min(x, y);
        }
      }
    }
  }
}

// The medians of kRun consecutive outputs along one axis of the staged tile: output s
// reads src[(s + j) * step], j < w.  put(s, median) takes each one.  The window is kept
// as order keys, padded with the smallest key below and the largest above (the largest
// is also every NaN's: a NaN and a pad are interchangeable, and slot kMid holds a NaN
// exactly when element floor(w / 2) of the window in np.sort's order is one).
template <typename T, typename Put>
__device__ __forceinline__ void run_medians(const T* src, int step, int w, Put&& put) {
  using U = typename Bits<T>::U;
  const U lo_fill = 0, hi_fill = ~U(0);
  const int lo = kMid - w / 2;               // smallest-key slots below the window
  U v[kK];
#pragma unroll
  for (int k = 0; k < kK; ++k)
    v[k] = k < lo ? lo_fill : (k < lo + w ? order_key(src[(k - lo) * step]) : hi_fill);
  sort_slots(v);
#pragma unroll 1
  for (int s = 0; s < kRun; ++s) {
    put(s, from_key<T>(v[kMid]));
    if (s + 1 == kRun) break;
    const U gone = order_key(src[s * step]), in = order_key(src[(s + w) * step]);
    // drop one copy of `gone` (the first slot not below it holds it) ...
#pragma unroll
    for (int k = 0; k < kK - 1; ++k) v[k] = v[k] < gone ? v[k] : v[k + 1];
    // ... and insert `in` among the kK - 1 slots left: slot k takes max(b[k-1], min(b[k], in))
    U below = lo_fill;
#pragma unroll
    for (int k = 0; k < kK; ++k) {
      const U here = k < kK - 1 ? v[k] : hi_fill;
      v[k] = max(below, min(here, in));
      below = here;
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(kThreads)
hpss_tile_kernel(const HpssArgs a, long long tiles_b, long long tiles_f) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* stage = reinterpret_cast<T*>(smem_raw);
  const int hh = (int)(a.win_harm / 2), hp = (int)(a.win_perc / 2);
  const int rows = kTileB + (int)a.win_perc - 1, cols = kTileF + (int)a.win_harm - 1;
  const int pitch = cols | 1;                 // odd: lanes on consecutive rows hit distinct banks
  T* harm = stage + rows * pitch;             // [kTileB][kHarmPitch]
  long long t = blockIdx.x;
  const long long tf = t % tiles_f;
  t /= tiles_f;
  const long long tb = t % tiles_b, b = t / tiles_b;
  const long long b0 = tb * kTileB, f0 = tf * kTileF;
  const long long clip = b * a.bins * a.frames;

  // 1. magnitudes of the tile and its halos (the corners no window reaches are skipped)
  for (int i = threadIdx.x; i < rows * cols; i += kThreads) {
    const int r = i / cols, c = i - r * cols;
    const bool core_r = r >= hp && r < hp + kTileB, core_c = c >= hh && c < hh + kTileF;
    if (!core_r && !core_c) continue;
    const long long br = hpss_reflect(b0 - hp + r, a.bins), fc = hpss_reflect(f0 - hh + c, a.frames);
    stage[r * pitch + c] = magnitude<T>(a.s, clip + br * a.frames + fc, a.complex_in);
  }
  __syncthreads();

  // 2. harmonic medians: thread (r, half) walks frames [kRun half, kRun (half + 1)) of row r
  {
    const int r = threadIdx.x % kTileB, c0 = (threadIdx.x / kTileB) * kRun;
    T* dst = harm + r * kHarmPitch + c0;
    run_medians<T>(stage + (hp + r) * pitch + c0, 1, (int)a.win_harm,
                   [&](int s, T m) { dst[s] = m; });
  }
  __syncthreads();

  // 3. percussive medians down each column, then both masks and the outputs
  {
    const int c = threadIdx.x % kTileF, r0 = (threadIdx.x / kTileF) * kRun;
    const long long f = f0 + c;
    run_medians<T>(stage + r0 * pitch + hh + c, pitch, (int)a.win_perc, [&](int s, T m) {
      const int r = r0 + s;
      const long long bin = b0 + r;
      if (bin < a.bins && f < a.frames)
        emit<T>(a, b, bin * a.frames + f, stage[(hp + r) * pitch + hh + c], harm[r * kHarmPitch + c], m);
    });
  }
}

// Element h = floor(w / 2) of the sorted window of w values at positions i - h ...
// i - h + w - 1 of an axis of n values (origin + stride * index), by counting ranks in
// the order of the keys (np.sort's, NaN last).
template <typename T>
__device__ T exact_median(const void* s, int cplx, long long origin, long long stride, long long n,
                          long long i, long long w) {
  const long long h = w / 2, period = 2 * n;
  long long m0 = (i - h) % period;
  if (m0 < 0) m0 += period;
  auto at = [&](long long m) {
    return magnitude<T>(s, origin + stride * (m < n ? m : period - 1 - m), cplx);
  };
  for (long long j = 0, mj = m0; j < w; ++j, mj = mj + 1 == period ? 0 : mj + 1) {
    const T vj = at(mj);
    const auto kj = order_key(vj);
    long long below = 0, same = 0;
    for (long long k = 0, mk = m0; k < w; ++k, mk = mk + 1 == period ? 0 : mk + 1) {
      const auto kk = order_key(at(mk));
      below += kk < kj;
      same += kk == kj;
    }
    if (below <= h && h < below + same) return from_key<T>(kj);
  }
  return T(NAN);     // not reached: the key order is total, so some value has rank h
}

template <typename T>
__global__ void __launch_bounds__(256) hpss_exact_kernel(const HpssArgs a) {
  const long long plane = a.bins * a.frames, total = a.batch * plane;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long b = i / plane, cell = i - b * plane;
    const long long r = cell / a.frames, f = cell - r * a.frames;
    const long long clip = b * plane;
    const T harm = exact_median<T>(a.s, a.complex_in, clip + r * a.frames, 1, a.frames, f, a.win_harm);
    const T perc = exact_median<T>(a.s, a.complex_in, clip + f, a.frames, a.bins, r, a.win_perc);
    emit<T>(a, b, cell, magnitude<T>(a.s, i, a.complex_in), harm, perc);
  }
}

template <typename T>
cudaError_t launch_typed(const HpssArgs& a, cudaStream_t st) {
  if (hpss_fast_supports(a.win_harm, a.win_perc)) {
    const long long tiles_b = (a.bins + kTileB - 1) / kTileB, tiles_f = (a.frames + kTileF - 1) / kTileF;
    const long long blocks = a.batch * tiles_b * tiles_f;
    if (blocks > 2147483647LL) return cudaErrorInvalidConfiguration;
    const int rows = kTileB + (int)a.win_perc - 1, pitch = (kTileF + (int)a.win_harm - 1) | 1;
    const size_t smem = ((size_t)rows * pitch + (size_t)kTileB * kHarmPitch) * sizeof(T);
    cudaError_t e = cudaFuncSetAttribute(hpss_tile_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    hpss_tile_kernel<T><<<(unsigned)blocks, kThreads, smem, st>>>(a, tiles_b, tiles_f);
  } else {
    const long long total = a.batch * a.bins * a.frames;
    const long long blocks = std::min<long long>((total + 255) / 256, 1LL << 20);
    hpss_exact_kernel<T><<<(unsigned)blocks, 256, 0, st>>>(a);
  }
  return cudaSuccess;
}

}  // namespace

bool hpss_fast_supports(long long win_harm, long long win_perc) {
  return win_harm >= 1 && win_perc >= 1 && win_harm <= kHpssFastWindow && win_perc <= kHpssFastWindow;
}

cudaError_t launch_hpss(const HpssArgs& a, cudaStream_t st) {
  if (a.batch == 0 || a.bins == 0 || a.frames == 0) return cudaSuccess;
  const cudaError_t e = a.f64 ? launch_typed<double>(a, st) : launch_typed<float>(a, st);
  if (e != cudaSuccess) return e;
  ++g_launch_count;
  return cudaGetLastError();
}

}  // namespace smb
