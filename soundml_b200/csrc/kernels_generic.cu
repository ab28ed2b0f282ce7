// Generic STFT and mel kernels: any fft size / hop / window / padding, float32
// or float64 audio, float64 interior.  This is the reference's precision
// contract taken literally (window multiply and transform in double, one
// rounding into the output dtype: stft.ml:28-35,345-364; mel product in
// double: mel.ml:228-231).  It is the always-available path; fft 2048 float32
// dispatches to the fused kernel in stft2048.cu instead.
#include "kernels.h"
#include "stft_stage.cuh"

#include <cstdio>

namespace smb {

std::atomic<long long> g_launch_count{0};

template <typename T> struct OutTraits;
template <> struct OutTraits<float> {
  typedef float2 complex_t;
  __device__ static float mag(float re, float im) { return hypotf(re, im); }
  __device__ static float pw(float m, float p) { return powf(m, p); }
};
template <> struct OutTraits<double> {
  typedef double2 complex_t;
  __device__ static double mag(double re, double im) { return hypot(re, im); }
  __device__ static double pw(double m, double p) { return pow(m, p); }
};

// One CTA per (tile of TF frames, signal).  Each frame: gather + window in
// double into shared memory, transform (radix-2 in place for powers of two,
// direct DFT otherwise), round once, stage the bins of the tile so the global
// writes run along the contiguous frame axis.
template <typename T, int MODE>
__global__ void stft_generic_kernel(const T* __restrict__ x, FrameGeom g,
                                    const double* __restrict__ window,
                                    const double2* __restrict__ twiddle, int log2n,
                                    int tile_frames, double power, void* __restrict__ out_) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double2* buf = reinterpret_cast<double2*>(smem_raw);
  const int N = g.fft;
  const int bins = N / 2 + 1;
  typedef typename OutTraits<T>::complex_t C;
  // output tile [bins][tile_frames] after the transform buffer(s)
  const bool pow2 = log2n >= 0;
  double2* spec = pow2 ? buf : buf + N;          // direct DFT writes to a second array
  unsigned char* tile_raw = reinterpret_cast<unsigned char*>(buf + (pow2 ? N : N + bins));
  C* tile_c = reinterpret_cast<C*>(tile_raw);
  T* tile_r = reinterpret_cast<T*>(tile_raw);

  const long long b = blockIdx.y;
  const long long p0 = (long long)blockIdx.x * tile_frames;
  const int nf = (int)min((long long)tile_frames, g.frames - p0);
  const T* xs = x + b * g.n;

  for (int f = 0; f < nf; ++f) {
    const long long start = (p0 + f) * g.hop;
    for (int j = threadIdx.x; j < N; j += blockDim.x) {
      const long long s = stage::src_index(g, start + j);
      const double v = s >= 0 ? (double)xs[s] : g.pad_value;
      const double wv = window[j] * v;
      int dst = j;
      if (pow2 && log2n > 0) dst = (int)(__brev((unsigned)j) >> (32 - log2n));
      buf[dst] = make_double2(wv, 0.0);
    }
    __syncthreads();
    if (pow2) {
      for (int s = 1; s <= log2n; ++s) {
        const int half = 1 << (s - 1);
        const int stride = N >> s;                 // twiddle step
        for (int idx = threadIdx.x; idx < N / 2; idx += blockDim.x) {
          const int j = idx & (half - 1);
          const int base = (idx >> (s - 1)) << s;
          const double2 w = twiddle[j * stride];
          const double2 a = buf[base + j];
          const double2 c = buf[base + j + half];
          const double tr = w.x * c.x - w.y * c.y;
          const double ti = w.x * c.y + w.y * c.x;
          buf[base + j] = make_double2(a.x + tr, a.y + ti);
          buf[base + j + half] = make_double2(a.x - tr, a.y - ti);
        }
        __syncthreads();
      }
    } else {
      for (int k = threadIdx.x; k < bins; k += blockDim.x) {
        double re = 0.0, im = 0.0;
        int idx = 0;                                // (j * k) mod N, incrementally
        for (int j = 0; j < N; ++j) {
          const double2 w = twiddle[idx];
          const double v = buf[j].x;
          re += v * w.x;
          im += v * w.y;
          idx += k;
          if (idx >= N) idx -= N;
        }
        spec[k] = make_double2(re, im);
      }
      __syncthreads();
    }
    for (int k = threadIdx.x; k < bins; k += blockDim.x) {
      const double2 z = spec[k];
      const T re = (T)z.x, im = (T)z.y;             // the one rounding
      if (MODE == kModeComplex) {
        C c;
        c.x = re;
        c.y = im;
        tile_c[k * tile_frames + f] = c;
      } else {
        const T m = OutTraits<T>::mag(re, im);      // stft.ml:670-674
        T v;
        if (power == 2.0) v = m * m;
        else if (power == 1.0) v = m;
        else v = OutTraits<T>::pw(m, (T)power);
        tile_r[k * tile_frames + f] = v;
      }
    }
    __syncthreads();
  }
  // [batch, bins, frames]
  const long long total = (long long)bins * nf;
  if (MODE == kModeComplex) {
    C* out = reinterpret_cast<C*>(out_) + b * bins * g.frames;
    for (long long i = threadIdx.x; i < total; i += blockDim.x) {
      const int k = (int)(i / nf), f = (int)(i % nf);
      out[(long long)k * g.frames + p0 + f] = tile_c[k * tile_frames + f];
    }
  } else {
    T* out = reinterpret_cast<T*>(out_) + b * bins * g.frames;
    for (long long i = threadIdx.x; i < total; i += blockDim.x) {
      const int k = (int)(i / nf), f = (int)(i % nf);
      out[(long long)k * g.frames + p0 + f] = tile_r[k * tile_frames + f];
    }
  }
}

static int ilog2_exact(int n) {
  if (n < 1 || (n & (n - 1))) return -1;
  int l = 0;
  while ((1 << l) < n) ++l;
  return l;
}

cudaError_t launch_stft_generic(const void* x, int dtype, long long batch, FrameGeom g,
                                const double* window, const double2* twiddle,
                                int mode, double power, void* out, cudaStream_t st) {
  if (batch == 0 || g.frames == 0) return cudaSuccess;
  const int N = g.fft, bins = N / 2 + 1;
  const int log2n = ilog2_exact(N);
  const size_t elem = (dtype == 0 ? 4 : 8) * (mode == kModeComplex ? 2 : 1);
  const size_t fixed = (size_t)(log2n >= 0 ? N : N + bins) * sizeof(double2);
  const size_t budget = 200 * 1024;
  if (fixed + (size_t)bins * elem > budget) return cudaErrorInvalidConfiguration;
  int tile = (int)((budget - fixed) / ((size_t)bins * elem));
  if (tile > 8) tile = 8;
  if (tile < 1) tile = 1;
  const size_t smem = fixed + (size_t)bins * elem * tile;
  const long long tiles = (g.frames + tile - 1) / tile;
  if (tiles > 2147483647LL || batch > 65535) {
    // fold the batch over several launches to respect grid limits
    for (long long b0 = 0; b0 < batch; b0 += 65535) {
      const long long nb = batch - b0 < 65535 ? batch - b0 : 65535;
      const char* xb = (const char*)x + (size_t)b0 * g.n * (dtype == 0 ? 4 : 8);
      char* ob = (char*)out + (size_t)b0 * bins * g.frames * elem;
      cudaError_t e = launch_stft_generic(xb, dtype, nb, g, window, twiddle, mode, power, ob, st);
      if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
  }
  dim3 grid((unsigned)tiles, (unsigned)batch);
  const int threads = N >= 512 ? 256 : (N >= 128 ? 128 : 64);
#define SMB_LAUNCH(T, M)                                                                  \
  do {                                                                                    \
    cudaError_t e = cudaFuncSetAttribute(stft_generic_kernel<T, M>,                       \
                                         cudaFuncAttributeMaxDynamicSharedMemorySize,     \
                                         (int)smem);                                      \
    if (e != cudaSuccess) return e;                                                       \
    stft_generic_kernel<T, M><<<grid, threads, smem, st>>>((const T*)x, g, window,        \
                                                           twiddle, log2n, tile, power,   \
                                                           out);                          \
  } while (0)
  if (dtype == 0) {
    if (mode == kModeComplex) SMB_LAUNCH(float, kModeComplex);
    else SMB_LAUNCH(float, kModePower);
  } else {
    if (mode == kModeComplex) SMB_LAUNCH(double, kModeComplex);
    else SMB_LAUNCH(double, kModePower);
  }
#undef SMB_LAUNCH
  ++g_launch_count;
  return cudaGetLastError();
}

// Mel.apply (mel.ml:202-231): out[b, m, p] = (T) sum_k W[m, k] * (double) S[b, k, p].
// One thread per output; threads of a warp run along the contiguous frame axis
// so every S row segment is one coalesced read, and only the filter's nonzero
// band is visited.
template <typename T>
__global__ void mel_apply_kernel(const T* __restrict__ s, int bins, long long frames,
                                 int n_mels, const double* __restrict__ w,
                                 const int* __restrict__ band_lo,
                                 const int* __restrict__ band_hi, T* __restrict__ out) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int m = blockIdx.y;
  const long long b = blockIdx.z;
  if (p >= frames) return;
  const T* sb = s + b * bins * frames;
  const double* wr = w + (long long)m * bins;
  double acc = 0.0;
  const int lo = band_lo[m], hi = band_hi[m];
  for (int k = lo; k < hi; ++k) acc += wr[k] * (double)sb[(long long)k * frames + p];
  out[(b * n_mels + m) * frames + p] = (T)acc;
}

cudaError_t launch_mel_apply(const void* s, int dtype, long long batch, int bins,
                             long long frames, int n_mels, const double* weights,
                             const int* band_lo, const int* band_hi, void* out,
                             cudaStream_t st) {
  if (batch == 0 || frames == 0) return cudaSuccess;
  const int threads = 128;
  const size_t esz = dtype == 0 ? 4 : 8;
  for (long long b0 = 0; b0 < batch; b0 += 65535) {
    const long long nb = batch - b0 < 65535 ? batch - b0 : 65535;
    dim3 grid((unsigned)((frames + threads - 1) / threads), (unsigned)n_mels, (unsigned)nb);
    const char* sb = (const char*)s + (size_t)b0 * bins * frames * esz;
    char* ob = (char*)out + (size_t)b0 * n_mels * frames * esz;
    if (dtype == 0)
      mel_apply_kernel<float><<<grid, threads, 0, st>>>((const float*)sb, bins, frames, n_mels,
                                                        weights, band_lo, band_hi, (float*)ob);
    else
      mel_apply_kernel<double><<<grid, threads, 0, st>>>((const double*)sb, bins, frames,
                                                         n_mels, weights, band_lo, band_hi,
                                                         (double*)ob);
    ++g_launch_count;
  }
  return cudaGetLastError();
}

}  // namespace smb
