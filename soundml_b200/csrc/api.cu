// C ABI of libsoundml_b200.so (see include/soundml_b200.h).
//
// Plans own: the host-side design (window / weights / filter banks, double),
// its device copies, a CUDA stream, and staging buffers for host-memory calls.
// Preconditions are checked in the reference's order and with its messages
// (SMB_EINVAL = Invalid_argument); CUDA failures are SMB_ECUDA.  There is no
// CPU execution path in this library.
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <memory>
#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/soundml_b200.h"
#include "host_design.h"
#include "kernels.h"

namespace {

thread_local std::string t_error;

struct cuda_failure : std::runtime_error {
  using std::runtime_error::runtime_error;
};

void cuda_check(cudaError_t e, const char* what) {
  if (e != cudaSuccess)
    throw cuda_failure(smb::format("soundml_b200: %s failed: %s", what, cudaGetErrorString(e)));
}
#define CK(call) cuda_check((call), #call)

template <typename F>
int guarded(F&& f) {
  try {
    f();
    return SMB_OK;
  } catch (const smb::invalid_argument& e) {
    t_error = e.what();
    return SMB_EINVAL;
  } catch (const cuda_failure& e) {
    t_error = e.what();
    return SMB_ECUDA;
  } catch (const std::bad_alloc&) {
    t_error = "soundml_b200: out of host memory";
    return SMB_ENOMEM;
  } catch (const std::exception& e) {
    t_error = e.what();
    return SMB_ECUDA;
  }
}

void require_device() {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    throw cuda_failure(
        "soundml_b200: no CUDA device is available (this library has no CPU fallback)");
}

// A device buffer that only ever grows.
struct DeviceBuffer {
  void* ptr = nullptr;
  size_t cap = 0;
  void* ensure(size_t bytes) {
    if (bytes > cap) {
      if (ptr) cudaFree(ptr);
      ptr = nullptr;
      cap = 0;
      CK(cudaMalloc(&ptr, bytes));
      cap = bytes;
    }
    return ptr;
  }
  void release() {
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
  }
};

template <typename T>
T* upload(const std::vector<T>& v) {
  T* d = nullptr;
  if (v.empty()) return d;
  CK(cudaMalloc(&d, v.size() * sizeof(T)));
  CK(cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  return d;
}

struct StreamOwner {
  cudaStream_t own = nullptr, use = nullptr;
  void create() {
    CK(cudaStreamCreateWithFlags(&own, cudaStreamNonBlocking));
    use = own;
  }
  // SMB_STREAM_OWN restores the plan's stream; anything else (NULL = the CUDA
  // default stream) is used as given.  Plans own scratch (the generic mel path's power
  // spectrogram, the cascade's hand-off buffer, the dB maximum, host-call staging) that
  // the next call reuses without an event, which is safe on ONE stream: when the stream
  // changes, work queued on the previous one is drained first, so the scratch is never
  // shared by two streams in flight.  The previous stream must still exist -- or have
  // been synchronised before it was destroyed (cudaErrorInvalidResourceHandle from a
  // stream already gone is swallowed: nothing can be pending on it).
  void set(void* external) {
    cudaStream_t next = external == SMB_STREAM_OWN ? own : (cudaStream_t)external;
    if (next != use) {
      const cudaError_t e = cudaStreamSynchronize(use);
      if (e != cudaSuccess) {
        cudaGetLastError();
        if (e != cudaErrorInvalidResourceHandle && e != cudaErrorContextIsDestroyed) CK(e);
      }
    }
    use = next;
  }
  void destroy() {
    if (own) cudaStreamDestroy(own);
    own = use = nullptr;
  }
};

// Host-memory calls stage the batch through the device in slices on three
// streams (H2D, compute, D2H) with two buffer slots, so the PCIe transfers of
// neighbouring slices overlap each other and the kernels (full-duplex link).
// With pageable host memory the copies degrade to synchronous staging; pinned
// memory (smb_host_alloc_pinned) gets the full overlap.
struct HostPipe {
  cudaStream_t h2d = nullptr, d2h = nullptr;
  cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_run[2] = {nullptr, nullptr},
              ev_out[2] = {nullptr, nullptr};
  DeviceBuffer in[2], out[2];
  bool ready = false;
  void ensure() {
    if (ready) return;
    CK(cudaStreamCreateWithFlags(&h2d, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&d2h, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      CK(cudaEventCreateWithFlags(&ev_in[i], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&ev_run[i], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&ev_out[i], cudaEventDisableTiming));
    }
    ready = true;
  }
  void release() {
    for (int i = 0; i < 2; ++i) {      // the buffers may have been used without the streams (smb_mfcc)
      in[i].release();
      out[i].release();
    }
    if (!ready) return;
    for (int i = 0; i < 2; ++i) {
      cudaEventDestroy(ev_in[i]);
      cudaEventDestroy(ev_run[i]);
      cudaEventDestroy(ev_out[i]);
    }
    cudaStreamDestroy(h2d);
    cudaStreamDestroy(d2h);
    ready = false;
  }
  // run(din, dout, items) enqueues the kernels for `items` batch items on `compute`.
  template <typename Run>
  void execute(cudaStream_t compute, const void* x, void* out_host, int64_t batch,
               size_t in_item, size_t out_item, Run&& run) {
    ensure();
    const size_t slice_bytes = (size_t)64 << 20;
    int64_t per = (int64_t)(slice_bytes / std::max<size_t>(1, in_item + out_item));
    per = std::max<int64_t>(1, std::min<int64_t>(per, batch));
    const int64_t slices = (batch + per - 1) / per;
    for (int64_t i = 0; i < slices; ++i) {
      const int slot = (int)(i & 1);
      const int64_t b0 = i * per, nb = std::min<int64_t>(per, batch - b0);
      void* din = in[slot].ensure((size_t)per * in_item);
      void* dout = out[slot].ensure((size_t)per * out_item);
      if (i >= 2) CK(cudaStreamWaitEvent(h2d, ev_run[slot], 0));      // input slot consumed
      CK(cudaMemcpyAsync(din, (const char*)x + (size_t)b0 * in_item, (size_t)nb * in_item,
                         cudaMemcpyHostToDevice, h2d));
      CK(cudaEventRecord(ev_in[slot], h2d));
      CK(cudaStreamWaitEvent(compute, ev_in[slot], 0));
      if (i >= 2) CK(cudaStreamWaitEvent(compute, ev_out[slot], 0));  // output slot drained
      run(din, dout, nb);
      CK(cudaEventRecord(ev_run[slot], compute));
      CK(cudaStreamWaitEvent(d2h, ev_run[slot], 0));
      CK(cudaMemcpyAsync((char*)out_host + (size_t)b0 * out_item, dout, (size_t)nb * out_item,
                         cudaMemcpyDeviceToHost, d2h));
      CK(cudaEventRecord(ev_out[slot], d2h));
    }
    CK(cudaStreamSynchronize(d2h));
    CK(cudaStreamSynchronize(compute));
  }
};

size_t dtype_size(int dtype) {
  if (dtype == SMB_F32) return 4;
  if (dtype == SMB_F64) return 8;
  throw smb::invalid_argument("soundml_b200: dtype must be SMB_F32 or SMB_F64");
}

const double kTwoPi = 6.283185307179586476925286766559;

}  // namespace

// A plan's tables, scratch and stream belong to the device that was current when it was
// first used; a later call under another current device would hand kernels pointers of
// the wrong device.
void same_device(int bound) {
  int now = -1;
  CK(cudaGetDevice(&now));
  if (now != bound)
    throw smb::invalid_argument(smb::format(
        "soundml_b200: the plan is bound to CUDA device %d but device %d is current "
        "(one plan per device; cudaSetDevice before the call)", bound, now));
}

// ============================ plan types =====================================

struct smb_stft_plan {
  smb::StftGeometry geom;
  std::vector<double> window;        // analysis window, fft doubles
  bool device_ready = false;
  int device = 0, sm_count = 0, path = SMB_PATH_AUTO;
  StreamOwner stream;
  double* d_window64 = nullptr;
  double2* d_twiddle64 = nullptr;
  double* d_folded = nullptr;        // synthesis: folded squared window, one entry per residue
  float* d_window_inv = nullptr;     // synthesis fast path: window / 2048
  float* d_window32 = nullptr;       // fast path tables (fft 2048 only)
  float2* d_tw_pass = nullptr;
  float2* d_tw_post = nullptr;
  void* d_dft_images = nullptr;      // tensor-core kernel: split-fp16 images of the 32-point DFT
  HostPipe pipe;
  DeviceBuffer tmp;        // power spectrogram of the generic mel path
  DeviceBuffer cepstral;   // mel spectrogram (+ host-call output) of the MFCC path

  void ensure_device() {
    if (device_ready) return same_device(device);
    require_device();
    CK(cudaGetDevice(&device));
    CK(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device));
    stream.create();
    d_window64 = upload(window);
    const int64_t n = geom.fft;
    std::vector<double2> tw((size_t)n);
    for (int64_t j = 0; j < n; ++j) {
      const double a = kTwoPi * double(j) / double(n);
      tw[(size_t)j] = make_double2(std::cos(a), -std::sin(a));
    }
    d_twiddle64 = upload(tw);
    if (fast_step() > 0) {
      // shorter frames run zero-padded to 2048: the window's tail is zero
      std::vector<float> w32(2048, 0.0f);
      for (int64_t j = 0; j < n; ++j) w32[(size_t)j] = (float)window[(size_t)j];
      d_window32 = upload(w32);
      std::vector<float2> pass(1024), post(512);
      for (int k1 = 0; k1 < 32; ++k1)
        for (int n2 = 0; n2 < 32; ++n2) {
          const double a = kTwoPi * double(k1 * n2) / 1024.0;
          pass[(size_t)(k1 * 32 + n2)] = make_float2((float)std::cos(a), (float)-std::sin(a));
        }
      for (int j = 0; j < 16; ++j)
        for (int l = 0; l < 32; ++l) {
          const double a = kTwoPi * double(l + 32 * j) / 2048.0;
          post[(size_t)(j * 32 + l)] = make_float2((float)std::cos(a), (float)-std::sin(a));
        }
      d_tw_pass = upload(pass);
      d_tw_post = upload(post);
      // The 32-point DFT in real arithmetic, F[n = (k, c')][j = (m, c)] with
      // (re, im) interleaved: out_re = sum in_re cos + in_im sin, out_im = sum
      // in_im cos - in_re sin (angle 2 pi m k / 32).  Two fp16 images (leading 11
      // bits, remainder) in the K-major SWIZZLE_128B operand layout: row n is
      // 128 bytes, its 16-byte chunk q sits at position q ^ (n mod 8).
      std::vector<__half> images(2 * 64 * 64);
      for (int n = 0; n < 64; ++n)
        for (int j = 0; j < 64; ++j) {
          const int k = n >> 1, co = n & 1, m = j >> 1, ci = j & 1;
          const double a = kTwoPi * double((m * k) % 32) / 32.0;
          const double v = ci == co ? std::cos(a) : (ci == 1 ? std::sin(a) : -std::sin(a));
          const __half hi = __float2half_rn((float)v);
          const __half lo = __float2half_rn((float)(v - (double)__half2float(hi)));
          const size_t at = (size_t)n * 64 + (size_t)((((j >> 3) ^ (n & 7)) << 3) | (j & 7));
          images[at] = hi;
          images[64 * 64 + at] = lo;
        }
      d_dft_images = upload(images);
    }
    device_ready = true;
  }
  // stft.ml:712-721: position m receives w[j]^2 for the j congruent to m modulo the hop
  std::vector<double> folded_square_window() const {
    std::vector<double> folded((size_t)geom.hop, 0.0);
    for (int64_t j = 0; j < geom.fft; ++j)
      folded[(size_t)(j % geom.hop)] += window[(size_t)j] * window[(size_t)j];
    return folded;
  }
  bool nola() const {                                    // stft.ml:731-742
    if (geom.hop > geom.fft) return false;
    const std::vector<double> folded = folded_square_window();
    double lo = HUGE_VAL, hi = 0.0;
    for (double v : folded) {
      if (v < lo) lo = v;
      if (v > hi) hi = v;
    }
    return lo > 1e-10 * hi;
  }
  int64_t output_length(int64_t frames) const {          // stft.ml:790-794
    if (frames == 0) return 0;
    return (frames - 1) * geom.hop + geom.fft - geom.left_width() - geom.right_width();
  }
  // 2048 / fft when the frame embeds in the fused kernel's 2048-point transform
  int fast_step() const {
    return geom.fft >= 128 && geom.fft <= 2048 && 2048 % geom.fft == 0 ? (int)(2048 / geom.fft) : 0;
  }
  smb::FrameGeom frame_geom(int64_t n) const {
    smb::FrameGeom g;
    g.n = n;
    g.frames = geom.frames(n);
    g.fft = (int)geom.fft;
    g.hop = (int)geom.hop;
    g.left = (int)geom.left_width();
    g.pad = geom.pad;
    g.pad_value = geom.pad_value;
    return g;
  }
  ~smb_stft_plan() {
    if (!device_ready) return;
    cudaFree(d_window64);
    cudaFree(d_twiddle64);
    cudaFree(d_folded);
    cudaFree(d_window_inv);
    cudaFree(d_window32);
    cudaFree(d_tw_pass);
    cudaFree(d_tw_post);
    cudaFree(d_dft_images);
    pipe.release();
    tmp.release();
    cepstral.release();
    stream.destroy();
  }
};

struct smb_mel_plan {
  int bound_device = 0;              // the device the tables live on (first use)
  int64_t n_mels = 0, fft = 0, bins = 0, sample_rate = 0;
  double f_min = 0, f_max = 0;
  int scale = 0, norm = 0;
  std::vector<double> weights;       // [n_mels][bins]
  std::vector<int> band_lo, band_hi;
  // Mel schedule of a fused kernel: every filter's band cut into pieces of at most
  // `ps` float4 steps, a lane carries one piece for all the frames of the tile.
  struct PieceSchedule {
    std::vector<float> vals;               // [round][step][lane] float4 weights
    std::vector<smb::MelPiece> pieces;     // [warps][rounds][32]
    std::vector<unsigned char> pcnt;       // [n_mels]: pieces (= partial sums) of each filter, 1..4
    int rounds = 0, mpad = 0;              // partial-sum slot of (piece j, filter m) = j * mpad + m
    float* d_vals = nullptr;
    smb::MelPiece* d_pieces = nullptr;
    unsigned char* d_pcnt = nullptr;
    void clear() { vals.clear(); pieces.clear(); pcnt.clear(); rounds = mpad = 0; }
    void to_device() { d_vals = upload(vals); d_pieces = upload(pieces); d_pcnt = upload(pcnt); }
    void free_device() { cudaFree(d_vals); cudaFree(d_pieces); cudaFree(d_pcnt); }
  };
  // Mel schedule of the frame-pair kernel (stft2048p.cu): whole filters, eight per
  // round, a lane = (filter, frame pair); rounds dealt to the group's four warps.
  struct PairSchedule {
    std::vector<float> w;                  // [round][step][8 filters] x float4
    std::vector<smb::PairMelItem> items;   // [4 warps][rounds][8]
    int rounds = 0;
    float* d_w = nullptr;
    smb::PairMelItem* d_items = nullptr;
    void clear() { w.clear(); items.clear(); rounds = 0; }
    void to_device() { if (!items.empty()) { d_w = upload(w); d_items = upload(items); } }
    void free_device() { cudaFree(d_w); cudaFree(d_items); }
  };
  PairSchedule sched_pair;
  PieceSchedule sched_cc;   // CUDA-core kernel: kFastTile warps, 8 frames per lane
  PieceSchedule sched_tc;   // tensor-core kernel: kTcTile warps, 4 frames per lane
  // 2048 / fft_size when the fused kernel can carry this filterbank (1 for fft
  // 2048, 2 for 1024, ...), else 0
  int fast_step = 0;
  bool device_ready = false;
  StreamOwner stream;
  double* d_weights = nullptr;
  int *d_band_lo = nullptr, *d_band_hi = nullptr;
  DeviceBuffer in, out;
  // MFCC epilogue: DCT table of the last (n_mfcc, lifter) asked for, max scratch
  double* d_dct = nullptr;
  unsigned long long* d_max = nullptr;
  int64_t dct_n_mfcc = -1;
  double dct_lifter = -1.0;
  const double* dct_table(int64_t n_mfcc, double lifter) {
    if (d_dct && dct_n_mfcc == n_mfcc && dct_lifter == lifter) return d_dct;
    // raw DCT-II rows 2 cos(pi k (2m+1) / 2N), orthonormal scales and lifter folded
    // in (soundml.ml:26-43, 84-93), all in double
    std::vector<double> t((size_t)(n_mfcc * n_mels));
    const double pi = 3.14159265358979323846;
    for (int64_t k = 0; k < n_mfcc; ++k) {
      double w = k == 0 ? 1.0 / std::sqrt(4.0 * double(n_mels)) : 1.0 / std::sqrt(2.0 * double(n_mels));
      if (lifter > 0.0) w *= 1.0 + lifter / 2.0 * std::sin(pi * double(k + 1) / lifter);
      for (int64_t m = 0; m < n_mels; ++m)
        t[(size_t)(k * n_mels + m)] =
            2.0 * std::cos(pi * double(k) * double(2 * m + 1) / (2.0 * double(n_mels))) * w;
    }
    cudaFree(d_dct);
    d_dct = upload(t);
    dct_n_mfcc = n_mfcc;
    dct_lifter = lifter;
    return d_dct;
  }

  void finish_host() {
    band_lo.assign((size_t)n_mels, 0);
    band_hi.assign((size_t)n_mels, 0);
    const bool small = bins <= 32767 && n_mels <= 32767;
    for (int64_t m = 0; m < n_mels; ++m) {
      int lo = (int)bins, hi = 0;
      for (int64_t k = 0; k < bins; ++k)
        if (weights[(size_t)(m * bins + k)] != 0.0) {
          lo = std::min(lo, (int)k);
          hi = (int)k + 1;
        }
      if (hi == 0) lo = 0;
      band_lo[(size_t)m] = lo;
      band_hi[(size_t)m] = hi;
    }
    if (!small || bins + 3 > 32767) return;
    // the fused kernel takes frames of 2048 / step samples, step a power of two
    // (shorter frames run zero-padded and keep every step-th bin in the power row)
    if (bins < 65 || bins > 1025 || 1024 % (bins - 1) != 0) return;
    const int step = (int)(1024 / (bins - 1));
    if (step == 1 && !build_pair_schedule(sched_pair)) sched_pair.clear();
    // the CUDA-core kernel trades a few padded steps for conflict-free octets
    // (whole list as the window); the tensor-core kernel has no shared memory to
    // spare for longer weight tables and keeps the strict longest-first rounds
    if (!build_schedule(sched_cc, smb::kFastTile, smb::kFastPieceSteps, 1 << 30) ||
        !build_schedule(sched_tc, smb::kTcTile, smb::kTcPieceSteps, 32)) {
      sched_cc.clear();
      sched_tc.clear();
      return;
    }
    fast_step = step;
  }
  // Mel schedule of the frame-pair kernel.  Filter m's band [band_lo, band_hi) is read
  // in 4-bin steps from an even bin b0 <= band_lo; eight consecutive filters make a
  // round (neighbouring bands have similar lengths), lane (i, j) of the round's warp
  // carries filter i for frame pair j.  The two filters of a quarter-warp start on
  // 16-byte groups of opposite parity (b0 / 2 odd against even; one of them moves two
  // bins down, weights zero there) so that the eight 16-byte loads of a quarter-warp,
  // whose four frame pairs sit 32 bytes apart, fall in eight distinct bank groups.
  // Weights are stored [round][step][filter] x float4 = one 128-byte run per warp
  // load.  Rounds go longest-first onto the lightest of the four warps.
  bool build_pair_schedule(PairSchedule& sc) const {
    sc.clear();
    const int kBins = 1032;                                  // power row incl. zeroed tail (stft2048p.cu)
    if (bins != 1025 || n_mels > 32767) return false;
    constexpr int F = smb::kPairFilters;                     // filters per round (lane = filter, frame pair)
    const int rounds_total = (int)((n_mels + F - 1) / F);
    struct Round { int steps; size_t base; int b0[F]; int m[F]; };
    std::vector<Round> built((size_t)rounds_total);
    for (int q = 0; q < rounds_total; ++q) {
      Round& rd = built[(size_t)q];
      int hi[F];
      for (int i = 0; i < F; ++i) {
        const int64_t m = (int64_t)q * F + i;
        rd.m[i] = m < n_mels ? (int)m : -1;
        rd.b0[i] = m < n_mels ? band_lo[(size_t)m] & ~1 : 0;
        hi[i] = m < n_mels ? std::max(band_hi[(size_t)m], rd.b0[i]) : 0;
      }
      for (int i = 0; i < F; i += 2) {
        if (rd.m[i] < 0 || rd.m[i + 1] < 0) continue;
        if ((((rd.b0[i] >> 1) + (rd.b0[i + 1] >> 1)) & 1) != 0) continue;
        if (rd.b0[i + 1] >= 2) rd.b0[i + 1] -= 2;
        else if (rd.b0[i] >= 2) rd.b0[i] -= 2;
      }
      rd.steps = 1;                                        // 0 marks an idle round in the kernel
      for (int i = 0; i < F; ++i)
        if (rd.m[i] >= 0) rd.steps = std::max(rd.steps, (hi[i] - rd.b0[i] + 3) / 4);
      rd.steps = (rd.steps + 1) & ~1;                      // the kernel runs two steps per iteration
      if (rd.steps > 510 || 4 * rd.steps > kBins) return false;
      // every lane runs the round's step count: keep its reads inside the row
      for (int i = 0; i < F; ++i) rd.b0[i] = std::min(rd.b0[i], (kBins - 4 * rd.steps) & ~1);
      rd.base = sc.w.size();
      sc.w.resize(rd.base + (size_t)rd.steps * F * 4, 0.0f);
      for (int i = 0; i < F; ++i) {
        if (rd.m[i] < 0) continue;
        for (int k = band_lo[(size_t)rd.m[i]]; k < band_hi[(size_t)rd.m[i]]; ++k) {
          const int u = k - rd.b0[i];
          sc.w[rd.base + ((size_t)(u >> 2) * F + (size_t)i) * 4 + (size_t)(u & 3)] =
              (float)weights[(size_t)((int64_t)rd.m[i] * bins + k)];
        }
      }
    }
    sc.w.resize(sc.w.size() + F * 4, 0.0f);                // the kernel's prefetch reads one step ahead
    if (sc.w.size() >= (1u << 24)) return false;
    const int warps = smb::kPairTile / 2;
    std::vector<int> by_len((size_t)rounds_total);
    for (int q = 0; q < rounds_total; ++q) by_len[(size_t)q] = q;
    std::stable_sort(by_len.begin(), by_len.end(),
                     [&](int a, int b) { return built[(size_t)a].steps > built[(size_t)b].steps; });
    std::vector<std::vector<int>> lists((size_t)warps);
    std::vector<long long> load((size_t)warps, 0);
    for (int q : by_len) {
      const size_t wi = (size_t)(std::min_element(load.begin(), load.end()) - load.begin());
      lists[wi].push_back(q);
      load[wi] += built[(size_t)q].steps * 10 + 30;
    }
    sc.rounds = 0;
    for (const auto& l : lists) sc.rounds = std::max(sc.rounds, (int)l.size());
    sc.items.assign((size_t)(warps * sc.rounds * F), smb::PairMelItem{0, 0, -1});   // idle: no steps
    for (int wi = 0; wi < warps; ++wi)
      for (size_t r = 0; r < lists[(size_t)wi].size(); ++r) {
        const Round& rd = built[(size_t)lists[(size_t)wi][r]];
        for (int i = 0; i < F; ++i) {
          smb::PairMelItem& it = sc.items[((size_t)wi * (size_t)sc.rounds + r) * F + (size_t)i];
          it.w4_steps = (int)(rd.base / 4 + (size_t)i) | ((rd.steps / 2) << 24);
          it.h0 = (unsigned short)(rd.b0[i] >> 1);
          it.m = (short)rd.m[i];
        }
      }
    return true;
  }
  // Mel schedule of the fused kernels.  Every filter's band, starting on a float4
  // of the power row, is cut into pieces of at most `ps` float4 steps; a lane
  // carries one piece for all the frames of its tile (one weight load feeds 4 FMAs
  // per frame) and leaves a partial sum in slot `pid` = j * mpad + m for the j-th
  // piece of filter m (at most four per filter: `ps` grows with the longest band;
  // the write-out adds the pcnt[m] of them up).  Rounds of 32 lanes share one
  // step count.  They are filled longest pieces first out of a window of
  // candidates, so that the lanes of a quarter-warp get distinct start residues
  // (start / 4 mod 8) where the window allows: their 16-byte power-row loads then
  // fall in distinct bank groups.  Weights are stored
  // [round][step][lane] x float4, a contiguous run per warp-wide load.  Rounds go
  // to the group's warps longest-first onto the lightest warp.
  bool build_schedule(PieceSchedule& sc, int warps, int ps, int window) const {
    sc.clear();
    const int row_floats = (int)((bins + 3) / 4 * 4);        // the kernel zeroes the row tail
    struct Piece { int m, start, steps, pid; };
    std::vector<Piece> pieces;
    sc.pcnt.assign((size_t)n_mels, 1);
    sc.mpad = (int)((n_mels + 7) / 8 * 8);
    int longest = 1;
    for (int64_t m = 0; m < n_mels; ++m) {
      const int lo = band_lo[(size_t)m] & ~3, hi = std::max(band_hi[(size_t)m], lo + 1);
      longest = std::max(longest, (hi - lo + 3) / 4);
    }
    ps = std::max(ps, (longest + 3) / 4);                // no filter in more than four pieces
    if (ps > 255) return false;
    for (int64_t m = 0; m < n_mels; ++m) {
      const int lo = band_lo[(size_t)m] & ~3, hi = std::max(band_hi[(size_t)m], lo + 1);
      const int total = (hi - lo + 3) / 4;
      int j = 0;
      for (int s0 = 0; s0 < total; s0 += ps, ++j)
        pieces.push_back(Piece{(int)m, lo + 4 * s0, std::min(ps, total - s0), j * sc.mpad + (int)m});
      sc.pcnt[(size_t)m] = (unsigned char)j;
    }
    const int scratch = 4 * sc.mpad;                     // idle lanes drop their zeros here
    // pieces longest first; a round is picked from the first `window` of them
    std::vector<int> rest(pieces.size());
    for (size_t i = 0; i < rest.size(); ++i) rest[i] = (int)i;
    std::stable_sort(rest.begin(), rest.end(),
                     [&](int a, int b) { return pieces[(size_t)a].steps > pieces[(size_t)b].steps; });
    struct Round { int steps; size_t base; int member[32]; int start[32]; };
    std::vector<Round> built;
    while (!rest.empty()) {
      Round rd;
      for (int t = 0; t < 32; ++t) rd.member[t] = -1;
      const size_t nc = std::min(rest.size(), (size_t)window);
      std::vector<char> used(nc, 0);
      // four octets, each scanning the candidates for eight distinct residues ...
      for (int o = 0; o < 4; ++o) {
        unsigned seen = 0;
        int lane = o * 8;
        for (size_t c = 0; c < nc && lane < o * 8 + 8; ++c) {
          if (used[c]) continue;
          const unsigned r = (unsigned)((pieces[(size_t)rest[c]].start >> 2) & 7);
          if (seen & (1u << r)) continue;
          seen |= 1u << r;
          used[c] = 1;
          rd.member[lane++] = rest[c];
        }
      }
      // ... then the free lanes take the longest candidates left
      for (int t = 0; t < 32; ++t) {
        if (rd.member[t] >= 0) continue;
        size_t c = 0;
        while (c < nc && used[c]) ++c;
        if (c == nc) break;
        used[c] = 1;
        rd.member[t] = rest[c];
      }
      std::vector<int> keep;
      for (size_t c = 0; c < rest.size(); ++c)
        if (c >= nc || !used[c]) keep.push_back(rest[c]);
      rest.swap(keep);
      rd.steps = 1;
      for (int t = 0; t < 32; ++t)
        if (rd.member[t] >= 0) rd.steps = std::max(rd.steps, pieces[(size_t)rd.member[t]].steps);
      if (rd.steps * 4 > row_floats) return false;
      rd.base = sc.vals.size();
      sc.vals.resize(rd.base + (size_t)rd.steps * 32 * 4, 0.0f);
      for (int t = 0; t < 32; ++t) {
        const int id = rd.member[t];
        rd.start[t] = 0;
        if (id < 0) continue;
        const Piece& pc = pieces[(size_t)id];
        // the stored run [start, start + 4 steps) must stay inside the row
        rd.start[t] = std::min(pc.start, row_floats - 4 * rd.steps);
        // the piece's own bins [pc.start, pc.start + 4 pc.steps), clipped to the band
        for (int k = pc.start; k < pc.start + 4 * pc.steps; ++k) {
          if (k >= bins || k < band_lo[(size_t)pc.m] || k >= band_hi[(size_t)pc.m]) continue;
          const int u = k - rd.start[t];
          sc.vals[rd.base + ((size_t)(u >> 2) * 32 + (size_t)t) * 4 + (size_t)(u & 3)] =
              (float)weights[(size_t)((int64_t)pc.m * bins + k)];
        }
      }
      built.push_back(rd);
    }
    const int rounds_total = (int)built.size();
    std::vector<int> by_len((size_t)rounds_total);
    for (int q = 0; q < rounds_total; ++q) by_len[(size_t)q] = q;
    std::stable_sort(by_len.begin(), by_len.end(),
                     [&](int a, int b) { return built[(size_t)a].steps > built[(size_t)b].steps; });
    std::vector<std::vector<int>> lists((size_t)warps);
    std::vector<long long> load((size_t)warps, 0);
    for (int q : by_len) {
      const size_t w = (size_t)(std::min_element(load.begin(), load.end()) - load.begin());
      lists[w].push_back(q);
      load[w] += built[(size_t)q].steps * 21 + 20;
    }
    sc.rounds = 0;
    for (const auto& l : lists) sc.rounds = std::max(sc.rounds, (int)l.size());
    const size_t zero_off = sc.vals.size();            // idle rounds: one step over zero weights
    sc.vals.insert(sc.vals.end(), (size_t)(32 * 4), 0.0f);
    if (sc.vals.size() >= (1u << 24)) return false;
    sc.pieces.assign((size_t)(warps * sc.rounds * 32), smb::MelPiece{});
    for (int w = 0; w < warps; ++w)
      for (int r = 0; r < sc.rounds; ++r)
        for (int t = 0; t < 32; ++t) {
          smb::MelPiece& out = sc.pieces[((size_t)w * (size_t)sc.rounds + (size_t)r) * 32 + (size_t)t];
          if ((size_t)r < lists[(size_t)w].size()) {
            const Round& rd = built[(size_t)lists[(size_t)w][(size_t)r]];
            out.off = (int)(rd.base + (size_t)t * 4) | (rd.steps << 24);
            out.lo = (short)rd.start[t];
            out.pid = (unsigned short)(rd.member[t] >= 0 ? pieces[(size_t)rd.member[t]].pid : scratch);
          } else {
            out.off = (int)(zero_off + (size_t)t * 4) | (1 << 24);
            out.lo = 0;
            out.pid = (unsigned short)scratch;
          }
        }
    return true;
  }
  void ensure_device() {
    if (device_ready) return same_device(bound_device);
    require_device();
    CK(cudaGetDevice(&bound_device));
    stream.create();
    d_weights = upload(weights);
    d_band_lo = upload(band_lo);
    d_band_hi = upload(band_hi);
    sched_cc.to_device();
    sched_tc.to_device();
    sched_pair.to_device();
    CK(cudaMalloc(&d_max, sizeof(unsigned long long)));
    device_ready = true;
  }
  ~smb_mel_plan() {
    if (!device_ready) return;
    cudaFree(d_weights);
    cudaFree(d_band_lo);
    cudaFree(d_band_hi);
    sched_cc.free_device();
    sched_tc.free_device();
    sched_pair.free_device();
    cudaFree(d_dct);
    cudaFree(d_max);
    in.release();
    out.release();
    stream.destroy();
  }
};

// Device copies of one overlap-save plan.
struct OlsDevice {
  smb::OlsPlan plan;
  float2* d_h = nullptr;
  float2* d_tw = nullptr;
  float2 *d_tw_pass = nullptr, *d_tw_base = nullptr;   // tables of the N = 2048 kernel
  int sm_count = 0;
  bool fast = true;                                     // the N = 2048 kernel may be used
  void upload_from(const smb::OlsPlan& p) {
    plan = p;
    if (!p.ok) return;
    if (p.n == 2048 && (p.l == 1 || p.polyphase)) {
      std::vector<float2> pass(1024), base(32);
      for (int k1 = 0; k1 < 32; ++k1)
        for (int n2 = 0; n2 < 32; ++n2) {
          const double a = kTwoPi * double(k1 * n2) / 1024.0;
          pass[(size_t)(k1 * 32 + n2)] = make_float2((float)std::cos(a), (float)-std::sin(a));
        }
      for (int l = 0; l < 32; ++l) {
        const double a = kTwoPi * double(l) / 2048.0;
        base[(size_t)l] = make_float2((float)std::cos(a), (float)-std::sin(a));
      }
      d_tw_pass = upload(pass);
      d_tw_base = upload(base);
      int device = 0;
      CK(cudaGetDevice(&device));
      CK(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device));
    }
    std::vector<float2> h(p.spectrum_re.size());
    for (size_t i = 0; i < h.size(); ++i)
      h[i] = make_float2((float)p.spectrum_re[i], (float)p.spectrum_im[i]);
    d_h = upload(h);
    const int64_t tn = std::max(p.n, p.w);
    std::vector<float2> tw((size_t)(tn / 2));
    for (int64_t j = 0; j < tn / 2; ++j) {
      const double a = kTwoPi * double(j) / double(tn);
      tw[(size_t)j] = make_float2((float)std::cos(a), (float)-std::sin(a));
    }
    d_tw = upload(tw);
  }
  void release() {
    cudaFree(d_h);
    cudaFree(d_tw);
    cudaFree(d_tw_pass);
    cudaFree(d_tw_base);
    d_h = d_tw = d_tw_pass = d_tw_base = nullptr;
  }
  void run(const float* x, int64_t batch, int64_t n, int64_t n_out, float* out,
           cudaStream_t st) const {
    smb::OlsArgs a{};
    a.x = x;
    a.out = out;
    a.n = n;
    a.n_out = n_out;
    a.blocks = plan.blocks_for(n_out);
    a.L = (int)plan.l; a.M = (int)plan.m; a.K = (int)plan.k;
    a.N = (int)plan.n; a.B = (int)plan.b; a.delta = (int)plan.delta; a.W = (int)plan.w;
    a.H = d_h;
    a.tw = d_tw;
    a.polyphase = plan.polyphase ? 1 : 0;
    if (fast && d_tw_pass && smb::ols2048_supports(a))
      CK(smb::launch_ols2048(a, d_tw_pass, d_tw_base, batch, sm_count, st));
    else if (plan.full_inverse || plan.polyphase)
      throw smb::invalid_argument("soundml_b200: this overlap-save plan needs the N = 2048 kernel");
    else
      CK(smb::launch_ols(a, batch, st));
  }
};

// Device image of G for the tensor-core executor of one phase-rich stage.
struct GemmDevice {
  // L <= 160 is one launch; wider stages (L = 320, 441, 640: the 44.1 k <-> 48 k
  // family) are cut into column groups of <= 160, one launch each, because the
  // three accumulators of a group must fit the 512 TMEM columns.
  struct Group {
    int col_begin = 0, width = 0, n_pad = 0, chunk_begin = 0, chunks = 0, tmem_cols = 0;
    float* d_images = nullptr;
    int4* d_meta = nullptr;
  };
  bool ok = false;
  std::vector<Group> groups;
  // Row form (resample_rows_kernel): stages whose L columns are one launch and whose
  // shift accumulators fit tensor memory.
  bool rows_ok = false;
  int rows_sm_count = 0;
  struct RowsGroup {
    smb::GemmRowsArgs a{};
    float* d_images = nullptr;
    int4 *d_chunks = nullptr, *d_slices = nullptr;
  };
  std::vector<RowsGroup> rows_groups;            // one launch per group of <= 160 columns
  void release_rows() {
    for (RowsGroup& g : rows_groups) {
      cudaFree(g.d_images);
      cudaFree(g.d_chunks);
      cudaFree(g.d_slices);
    }
    rows_groups.clear();
    rows_ok = false;
  }
  // columns [c0, c0 + l) of the stage's L (l_total below)
  // split_main: the row grid is shifted so that every column's filter centre falls into the
  // same shift (qc), and that shift's two small split terms get an accumulator of their own:
  // its main accumulator then is a chain of exact hi x hi products only (4 per chunk).  With
  // everything in one accumulator per shift, a 14-chunk stage (44.1 -> 16 kHz) measured
  // -121.9 dB THD+N in float32 against the reference's -125 dB gate (resample_quality.ml
  // Q1/Q2); the window form, which separates the small terms, -132.5 dB.
  bool build_rows_group(const smb::ResampleStage& s, int64_t c0, int64_t l, bool single_group, bool split_main) {
    const int64_t l_total = s.l, m = s.m, taps = 2 * s.k + 1;
    if (l > 160 || m < 32) return false;
    std::vector<int64_t> d((size_t)l);
    int64_t k;
    int qc = 0;
    if (split_main) {
      // row j of G for (column r, tap t) is d_r + t; the centre tap of the group's first column
      // is moved onto a multiple of M, so every centre (they span less than M rows) lies in shift qc
      const int64_t d_first = (c0 * m) / l_total, shift = (m - s.k % m) % m;
      for (int64_t r = 0; r < l; ++r) d[(size_t)r] = ((c0 + r) * m) / l_total - d_first + shift;
      k = s.k + shift - d_first;
      qc = (int)((s.k + shift) / m);
    } else {
      // the group's first column starts q0 whole input rows in: fold them into the delay
      const int64_t q0 = ((c0 * m) / l_total) / m;
      k = s.k - q0 * m;
      for (int64_t r = 0; r < l; ++r) d[(size_t)r] = ((c0 + r) * m) / l_total - q0 * m;
    }
    const int64_t p_len = taps + d[(size_t)(l - 1)];
    const int shifts = (int)((p_len + m - 1) / m);
    const int chunks = (int)((m + 31) / 32);
    const int n_pad = (int)((l + 15) / 16 * 16);
    if (shifts > 4) return false;
    // columns of G_q with a nonzero in rows [j0, j1] of the shift's block: d_r <= q m + j <= d_r + taps - 1
    auto active = [&](int q, int64_t j0, int64_t j1, int* lo, int* hi) {
      *lo = n_pad;
      *hi = -1;
      for (int64_t r = 0; r < l; ++r) {
        const int64_t first = d[(size_t)r] - (int64_t)q * m, last = first + taps - 1;
        if (first <= j1 && last >= j0) {
          *lo = std::min(*lo, (int)r);
          *hi = std::max(*hi, (int)r);
        }
      }
      return *hi >= 0;
    };
    smb::GemmRowsArgs a{};
    int total_cols = 0;
    // accumulators side by side in DESCENDING q: the active columns of D_q are a suffix
    // and those of D_(q-1) a prefix, so a chunk's nonzeros form one run of TMEM columns
    // (split_main: the outer shifts first, then the main shift, then its small-term accumulator:
    // the main shift and the tails are dealt to different issuing threads)
    std::vector<int> order;
    for (int q = shifts - 1; q >= 0; --q)
      if (!split_main || q != qc) order.push_back(q);
    if (split_main && qc >= shifts) return false;
    if (split_main) order.push_back(qc);
    int tails_cols = 0;
    for (int q : order) {
      int lo, hi;
      if (!active(q, 0, m - 1, &lo, &hi)) return false;
      if (split_main && q == qc) tails_cols = total_cols;
      a.acc_shift[q] = q;
      a.acc_lo[q] = (q == 0 && !split_main) ? 0 : lo / 16 * 16;
      a.acc_w[q] = (q == 0 && !split_main) ? n_pad : (hi + 1 - a.acc_lo[q] + 15) / 16 * 16;
      a.acc_col[q] = total_cols;
      total_cols += a.acc_w[q];
    }
    const int d_cols = total_cols;                                // the shifts' accumulators: what a run may cover
    a.n_acc = shifts;
    if (split_main) {
      a.acc_shift[shifts] = qc;
      a.acc_lo[shifts] = a.acc_lo[qc];
      a.acc_w[shifts] = a.acc_w[qc];
      a.acc_col[shifts] = total_cols;
      total_cols += a.acc_w[qc];
      a.n_acc = shifts + 1;
    }
    if (total_cols > 512 || chunks > 32 || chunks < 3) return false;   // (chunks >= stages: the loader's scratch hand-over)
    // the A tiles go to tensor memory when two stages of 64 columns fit beside the accumulators
    // (the products then read only B from shared memory: 1.99 -> 1.90 ms on configs[3]); a stage
    // cut into column groups gathers A once per group and is better off with the cheaper
    // shared-memory producers (44.1 -> 32 kHz: 0.88 against 0.93 ms).  SMB_ROWS_SMEM_A=1 /
    // SMB_ROWS_TMEM_A=1 force either.
    const bool a_tmem = total_cols + 128 <= 512 && !getenv("SMB_ROWS_SMEM_A") &&
                        (single_group || getenv("SMB_ROWS_TMEM_A"));
    int tmem_alloc = 32;
    while (tmem_alloc < total_cols + (a_tmem ? 128 : 0)) tmem_alloc *= 2;
    const int kSliceAlign = getenv("SMB_ROWS_ALIGN") ? atoi(getenv("SMB_ROWS_ALIGN")) : 8;
    std::vector<int4> chunk_meta((size_t)chunks), slice_meta;
    struct Run { int bytes_at, start, width; };                  // a chunk's stored rows: [hi | lo][width][32]
    std::vector<Run> runs;
    // per chunk: TMEM column -> run, -1 where nothing is stored
    std::vector<std::vector<int>> run_at((size_t)chunks, std::vector<int>((size_t)d_cols, -1));
    size_t total_bytes = 0;
    int stage_bytes = 0;
    for (int ch = 0; ch < chunks; ++ch) {
      // exact active columns (TMEM coordinates); a run may start on any column -- only its
      // width is a multiple of 16 -- so a chunk stores ceil16(band) columns, not the
      // band widened to 16-column boundaries on both sides
      std::vector<char> on((size_t)d_cols, 0);
      for (int q = 0; q < shifts; ++q) {
        int lo, hi;
        if (!active(q, 32 * (int64_t)ch, std::min<int64_t>(32 * (int64_t)ch + 31, m - 1), &lo, &hi)) continue;
        for (int cc = lo; cc <= hi; ++cc) on[(size_t)(a.acc_col[q] + cc - a.acc_lo[q])] = 1;
      }
      const int first_slice = (int)slice_meta.size();
      int bytes = 0;
      for (int t0 = 0; t0 < d_cols;) {
        if (!on[(size_t)t0]) { ++t0; continue; }
        int t1 = t0 + 1;                                          // one past the run's last active column
        const int t_end = split_main && t0 < tails_cols ? tails_cols : d_cols;   // a run stays with one owner
        for (int t = t0 + 1; t < t_end && t - t0 < 256; ++t) {
          if (on[(size_t)t]) t1 = t + 1;
          else if (t - t1 >= 16) break;                           // a gap of 16 columns ends the run
        }
        int start = t0 / kSliceAlign * kSliceAlign;              // the accumulator address of a product
        int width = (t1 - start + 15) / 16 * 16;
        if (width > 256) { width = 256; t1 = start + 256; }
        if (start + width > d_cols) start = d_cols - width;      // (never past the shifts' accumulators)
        if (split_main && t0 < tails_cols && start + width > tails_cols) start = tails_cols - width;
        if (split_main && t0 >= tails_cols && start < tails_cols) start = tails_cols;   // (a 16-column boundary)
        if (start < 0) return false;
        for (int t = start; t < start + width; ++t) run_at[(size_t)ch][(size_t)t] = (int)runs.size();
        runs.push_back(Run{bytes, start, width});
        const int lo_delta = width * 128;                         // from a row's hi image to its lo image
        if (!split_main) {
          slice_meta.push_back(make_int4(bytes, start, width, 0 | (lo_delta << 3)));
        } else if (start < tails_cols) {
          // the outer shifts: all three products in their own accumulators, second issuer
          slice_meta.push_back(make_int4(bytes, start, width, 0 | 4 | (lo_delta << 3)));
        } else {
          // the main shift: hi x hi into its accumulator, the small terms into the extra one
          slice_meta.push_back(make_int4(bytes, start, width, 1 | (lo_delta << 3)));
          slice_meta.push_back(make_int4(bytes, a.acc_col[shifts] + (start - a.acc_col[qc]), width, 2 | (lo_delta << 3)));
        }
        bytes += 2 * width * 128;
        t0 = std::max(t1, start + width);
      }
      chunk_meta[(size_t)ch] = make_int4((int)total_bytes, bytes, first_slice, (int)slice_meta.size() - first_slice);
      total_bytes += (size_t)bytes;
      stage_bytes = std::max(stage_bytes, bytes);
    }
    if (slice_meta.size() > 80) return false;
    stage_bytes = (stage_bytes + 1023) / 1024 * 1024;
    // static shared memory of the kernel (barriers, metadata) comes out of the same 227 KB
    const size_t budget = 227 * 1024 - 2048;
    a.a_tmem = a_tmem ? 1 : 0;
    a.a_tmem_col = total_cols;
    if (a_tmem) {
      a.a_stages = 2;
      // no more B stages than chunks: the B loader takes back the stage the epilogue borrowed
      // at chunk b_stages - 1 of the next tile, a chunk a 3-chunk tile does not have
      a.b_stages = std::min(4, chunks);
      const size_t turn = 8 * 32 * 17 * 4;                      // the producers' transposition tiles
      while (a.b_stages > 2 && smb::resample_rows_smem_bytes(0, a.b_stages, stage_bytes) + turn > budget) --a.b_stages;
      if (smb::resample_rows_smem_bytes(0, a.b_stages, stage_bytes) + turn > budget) return false;
    } else if (smb::resample_rows_smem_bytes(2, 3, stage_bytes) <= budget) { a.a_stages = 2; a.b_stages = 3; }
    else if (smb::resample_rows_smem_bytes(3, 2, stage_bytes) <= budget) { a.a_stages = 3; a.b_stages = 2; }
    else if (smb::resample_rows_smem_bytes(2, 2, stage_bytes) <= budget) { a.a_stages = 2; a.b_stages = 2; }
    else return false;
    int device = 0;
    CK(cudaGetDevice(&device));
    CK(cudaDeviceGetAttribute(&rows_sm_count, cudaDevAttrMultiProcessorCount, device));
    std::vector<float> img(total_bytes / 4, 0.0f);
    for (int64_t r = 0; r < l; ++r) {
      const int64_t ph = ((c0 + r) * m) % l_total;
      for (int64_t t = 0; t < taps; ++t) {
        const int64_t j = d[(size_t)r] + t;
        const int q = (int)(j / m);
        const int64_t jj = j % m;
        const int ch = (int)(jj / 32), kk = (int)(jj % 32);
        const int tcol = a.acc_col[q] + (int)r - a.acc_lo[q];
        const int ri = run_at[(size_t)ch][(size_t)tcol];
        if (ri < 0) return false;                               // (cannot happen: the runs cover every nonzero)
        const Run run = runs[(size_t)ri];
        const double gv = s.bank[(size_t)(ph * taps + t)];
        const float gf = (float)gv;
        uint32_t bits;
        std::memcpy(&bits, &gf, 4);
        bits &= 0xFFFFE000u;
        float hi;
        std::memcpy(&hi, &bits, 4);
        const float lo = (float)(gv - (double)hi);
        const int64_t rr = tcol - run.start;                     // row inside the run
        const size_t cell = (size_t)(rr * 32 + ((((kk >> 2) ^ (rr & 7)) << 2) | (kk & 3)));
        const size_t base = ((size_t)chunk_meta[(size_t)ch].x + (size_t)run.bytes_at) / 4;
        img[base + cell] = hi;
        img[base + (size_t)run.width * 32 + cell] = lo;
      }
    }
    a.slices = (int)slice_meta.size();
    a.two_issuers = split_main ? 1 : 0;
    a.l = (int)l;
    a.m = (int)m;
    a.k = (int)k;
    a.n_pad = n_pad;
    a.shifts = shifts;
    a.chunks = chunks;
    a.tmem_cols = tmem_alloc;
    a.b_stage_bytes = stage_bytes;
    a.l_total = (int)l_total;
    a.col_begin = (int)c0;
    RowsGroup g;
    g.d_images = upload(img);
    g.d_chunks = upload(chunk_meta);
    g.d_slices = upload(slice_meta);
    a.b_images = g.d_images;
    a.chunk_meta = g.d_chunks;
    a.slice_meta = g.d_slices;
    g.a = a;
    rows_groups.push_back(g);
    return true;
  }
  void build_rows(const smb::ResampleStage& s) {
    const int n_groups = (int)((s.l + 159) / 160);
    const int64_t base_width = ((s.l + n_groups - 1) / n_groups + 15) / 16 * 16;
    // long stages (many K-chunks = long accumulation chains) separate the small terms of the
    // main shift when tensor memory has room for the extra accumulator; SMB_ROWS_SPLIT=0/1 forces
    const bool want_split = getenv("SMB_ROWS_SPLIT") ? atoi(getenv("SMB_ROWS_SPLIT")) != 0 : (s.m + 31) / 32 >= 8;
    for (int attempt = want_split ? 0 : 1; attempt < 2; ++attempt) {
      bool ok = true;
      for (int64_t c0 = 0; c0 < s.l && ok; c0 += base_width)
        ok = build_rows_group(s, c0, std::min<int64_t>(base_width, s.l - c0), n_groups == 1, attempt == 0);
      if (ok) {
        rows_ok = true;
        return;
      }
      release_rows();
    }
  }
  void build(const smb::ResampleStage& s) {
    const int64_t l = s.l, m = s.m, k = s.k, taps = 2 * k + 1;
    if (s.exec != smb::kExecGemm || l > 1024) return;
    build_rows(s);
    const int n_groups = (int)((l + 159) / 160);
    const int base_width = (int)(((l + n_groups - 1) / n_groups + 15) / 16 * 16);
    for (int c0 = 0; c0 < l; c0 += base_width) {
      Group g;
      g.col_begin = c0;
      g.width = (int)std::min<int64_t>(base_width, l - c0);
      g.n_pad = (g.width + 15) / 16 * 16;
      // rows of G (K index) this group's columns touch: d(r) = floor(r M / L) .. + taps - 1
      const int64_t d_first = ((int64_t)c0 * m) / l;
      const int64_t d_last = ((int64_t)(c0 + g.width - 1) * m) / l + taps - 1;
      g.chunk_begin = (int)(d_first / 32);
      g.chunks = (int)(d_last / 32) - g.chunk_begin + 1;
      g.tmem_cols = 32;
      while (g.tmem_cols < 3 * g.n_pad) g.tmem_cols *= 2;
      // G is banded: chunk ch only has nonzeros in a run of columns.  Store and
      // multiply just that run, widened to multiples of 16 columns; the group's
      // first two chunks keep the full width because their first products
      // zero-initialise the accumulators.
      std::vector<int> cmin((size_t)g.chunks, g.n_pad), cmax((size_t)g.chunks, -1);
      for (int r = 0; r < g.width; ++r) {
        const int64_t d = ((int64_t)(c0 + r) * m) / l;
        for (int64_t ch = d / 32; ch <= (d + taps - 1) / 32; ++ch) {
          const size_t rel = (size_t)(ch - g.chunk_begin);
          cmin[rel] = std::min(cmin[rel], r);
          cmax[rel] = std::max(cmax[rel], r);
        }
      }
      std::vector<int4> meta((size_t)g.chunks);
      size_t total_floats = 0;
      for (int ch = 0; ch < g.chunks; ++ch) {
        int col0 = 0, ncols = g.n_pad;
        if (ch >= 2 && cmax[(size_t)ch] >= 0) {
          col0 = cmin[(size_t)ch] / 16 * 16;
          ncols = (cmax[(size_t)ch] + 1 - col0 + 15) / 16 * 16;
        } else if (ch >= 2) {
          ncols = 16;                                          // empty chunk: a zero slice
        }
        meta[(size_t)ch] = make_int4((int)(total_floats * 4), col0, ncols, 0);
        total_floats += (size_t)2 * ncols * 32;
      }
      std::vector<float> img(total_floats, 0.0f);
      for (int r = 0; r < g.width; ++r) {
        const int64_t col = c0 + r;
        const int64_t d = (col * m) / l, ph = (col * m) % l;
        for (int64_t t = 0; t < taps; ++t) {
          const int64_t j = d + t;                               // row of G
          const double gv = s.bank[(size_t)(ph * taps + t)];
          const float gf = (float)gv;
          uint32_t bits;
          std::memcpy(&bits, &gf, 4);
          bits &= 0xFFFFE000u;                                   // tf32 piece, exact
          float hi;
          std::memcpy(&hi, &bits, 4);
          const float lo = (float)(gv - (double)hi);
          const int64_t ch = j / 32 - g.chunk_begin, kk = j % 32;
          const int4 mt = meta[(size_t)ch];
          const int64_t rr = r - mt.y;                           // row inside the stored slice
          const size_t cell = (size_t)(rr * 32 + ((((kk >> 2) ^ (rr & 7)) << 2) | (kk & 3)));
          const size_t base = (size_t)mt.x / 4;
          img[base + cell] = hi;
          img[base + (size_t)mt.z * 32 + cell] = lo;
        }
      }
      g.d_meta = upload(meta);
      g.d_images = upload(img);
      groups.push_back(g);
    }
    ok = true;
  }
  void release() {
    for (Group& g : groups) {
      cudaFree(g.d_images);
      cudaFree(g.d_meta);
    }
    groups.clear();
    release_rows();
  }
};

struct smb_resample_plan {
  int bound_device = 0;              // the device the tables live on (first use)
  smb::ResamplePlan plan;
  bool device_ready = false;
  StreamOwner stream;
  std::vector<float*> d_bank;        // per stage, [l][2k+1] float32
  std::vector<double*> d_bank64;     // the same banks uncast, for float64 audio
  std::vector<OlsDevice> ols;        // per stage; plan.ok only for OLS-tagged power-of-two stages
  std::vector<GemmDevice> gemm;      // per stage; ok only for GEMM-tagged stages
  int executor = SMB_EXEC_PLANNED;   // SMB_EXEC_DIRECT forces the dot-product kernel everywhere
  DeviceBuffer in, out, mid;
  HostPipe pipe;                     // host-memory calls: sliced, copies under kernels
  void ensure_device() {
    if (device_ready) return same_device(bound_device);
    require_device();
    CK(cudaGetDevice(&bound_device));
    stream.create();
    for (const auto& s : plan.stages) {
      std::vector<float> b(s.bank.size());
      for (size_t i = 0; i < b.size(); ++i) b[i] = (float)s.bank[i];   // cast at prepare
      d_bank.push_back(upload(b));
      d_bank64.push_back(upload(s.bank));
      ols.emplace_back();
      ols.back().upload_from(smb::ols_plan_for_stage(s));
      gemm.emplace_back();
      gemm.back().build(s);
    }
    device_ready = true;
  }
  // The kernel run_stage picks for stage i (SMB_FORM_*).
  int form(size_t i) const {
    if (executor == SMB_EXEC_DIRECT) return SMB_FORM_DIRECT;
    if (ols[i].plan.ok) return SMB_FORM_OLS;
    // (SMB_GEMM_WINDOWS=1: the overlapping-window form, for A/B measurement)
    if (gemm[i].rows_ok && !getenv("SMB_GEMM_WINDOWS")) return SMB_FORM_ROW;
    if (gemm[i].ok) return SMB_FORM_WINDOW;
    return SMB_FORM_DIRECT;
  }
  // One stage over device buffers: overlap-save where the planner tagged it and
  // the GPU plan exists, the direct polyphase kernel otherwise -- the same
  // designed filter either way (resample.ml:495-497).
  void run_stage(size_t i, const float* x, int64_t batch, int64_t n, int64_t n_out, float* out,
                 cudaStream_t st) {
    const smb::ResampleStage& s = plan.stages[i];
    const int f = form(i);
    if (f == SMB_FORM_OLS) {
      ols[i].run(x, batch, n, n_out, out, st);
    } else if (f == SMB_FORM_ROW) {
      for (const GemmDevice::RowsGroup& g : gemm[i].rows_groups) {
        smb::GemmRowsArgs a = g.a;
        a.x = x;
        a.out = out;
        a.n = n;
        a.n_out = n_out;
        CK(smb::launch_resample_rows(a, batch, gemm[i].rows_sm_count, st));
      }
    } else if (f == SMB_FORM_WINDOW) {
      for (const GemmDevice::Group& g : gemm[i].groups) {
        smb::GemmResampleArgs a{};
        a.x = x;
        a.out = out;
        a.n = n;
        a.n_out = n_out;
        a.l = g.width;
        a.m = (int)s.m;
        a.k = (int)s.k - 32 * g.chunk_begin;          // the group's first K-chunk is chunk 0
        a.l_total = (int)s.l;
        a.col_begin = g.col_begin;
        a.n_pad = g.n_pad;
        a.chunks = g.chunks;
        a.tmem_cols = g.tmem_cols;
        a.b_images = g.d_images;
        a.chunk_meta = g.d_meta;
        CK(smb::launch_resample_gemm(a, batch, st));
      }
    } else
      CK(smb::launch_polyphase_direct(x, batch, n, d_bank[i], (int)s.l, (int)s.m, (int)s.k,
                                      n_out, out, st));
  }
  ~smb_resample_plan() {
    if (!device_ready) return;
    for (float* p : d_bank) cudaFree(p);
    for (double* p : d_bank64) cudaFree(p);
    for (OlsDevice& o : ols) o.release();
    for (GemmDevice& g : gemm) g.release();
    in.release();
    out.release();
    mid.release();
    pipe.release();
    stream.destroy();
  }
};

struct smb_fir_plan {
  int bound_device = 0;              // the device the tables live on (first use)
  std::vector<double> h;
  int64_t k = 0;
  bool device_ready = false;
  StreamOwner stream;
  float* d_bank = nullptr;
  OlsDevice ols;
  DeviceBuffer in, out;
  HostPipe pipe;                     // host-memory calls: sliced, copies under kernels
  void ensure_device() {
    if (device_ready) return same_device(bound_device);
    require_device();
    CK(cudaGetDevice(&bound_device));
    stream.create();
    std::vector<float> b(h.size());
    for (size_t s = 0; s < h.size(); ++s) b[s] = (float)h[h.size() - 1 - s];  // row reversed
    d_bank = upload(b);
    ols.upload_from(smb::ols_plan_for_fir(h));
    device_ready = true;
  }
  ~smb_fir_plan() {
    if (!device_ready) return;
    cudaFree(d_bank);
    ols.release();
    in.release();
    out.release();
    pipe.release();
    stream.destroy();
  }
};

// ============================ entry points ===================================

extern "C" {

const char* smb_last_error(void) { return t_error.c_str(); }
const char* smb_version(void) { return "soundml_b200 0.1 (sm_100a)"; }

int smb_device_count(int* count) {
  return guarded([&] {
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) c = 0;
    *count = c;
  });
}
int smb_set_device(int device) { return guarded([&] { CK(cudaSetDevice(device)); }); }
int smb_device_alloc(void** ptr, size_t bytes) {
  return guarded([&] { require_device(); CK(cudaMalloc(ptr, bytes ? bytes : 1)); });
}
int smb_device_free(void* ptr) { return guarded([&] { CK(cudaFree(ptr)); }); }
int smb_host_alloc_pinned(void** ptr, size_t bytes) {
  return guarded([&] { require_device(); CK(cudaMallocHost(ptr, bytes ? bytes : 1)); });
}
int smb_host_free_pinned(void* ptr) { return guarded([&] { CK(cudaFreeHost(ptr)); }); }
int smb_memcpy_h2d(void* dst, const void* src, size_t bytes) {
  return guarded([&] { CK(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice)); });
}
int smb_memcpy_d2h(void* dst, const void* src, size_t bytes) {
  return guarded([&] { CK(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost)); });
}
int smb_device_synchronize(void) { return guarded([&] { CK(cudaDeviceSynchronize()); }); }
int64_t smb_kernel_launch_count(void) { return smb::g_launch_count.load(); }

int smb_window_make(int kind, double param, int periodic, int64_t n, double* out) {
  return guarded([&] {
    std::vector<double> w = smb::window_make("make", kind, param, periodic != 0, n);
    std::memcpy(out, w.data(), w.size() * sizeof(double));
  });
}

// ---- STFT --------------------------------------------------------------------

int smb_stft_plan_create(smb_stft_plan** plan, int64_t fft_size, int64_t hop,
                         int64_t win_length, int window_kind, double window_param,
                         int alignment, int pad_kind, double pad_value, int scale) {
  return guarded([&] {
    *plan = nullptr;
    smb::StftGeometry g;
    g.fft = fft_size;
    g.hop = hop;
    g.win_length = win_length;
    g.alignment = alignment;
    g.pad = pad_kind;
    g.pad_value = pad_value;
    g.scale = scale;
    std::vector<double> w = smb::stft_analysis_window(g, window_kind, window_param);
    smb_stft_plan* p = new smb_stft_plan;
    p->geom = g;
    p->window = std::move(w);
    *plan = p;
  });
}

int smb_stft_plan_create_with_window(smb_stft_plan** plan, int64_t fft_size, int64_t hop,
                                     int alignment, int pad_kind, double pad_value,
                                     const double* analysis_window) {
  return guarded([&] {
    *plan = nullptr;
    smb::StftGeometry g;
    g.fft = fft_size;
    g.hop = hop == SMB_DEFAULT ? std::max<int64_t>(1, fft_size / 4) : hop;
    g.win_length = fft_size;
    g.alignment = alignment;
    g.pad = pad_kind;
    g.pad_value = pad_value;
    smb::stft_validate_geometry(g);
    smb_stft_plan* p = new smb_stft_plan;
    p->geom = g;
    p->window.assign(analysis_window, analysis_window + fft_size);
    *plan = p;
  });
}

int smb_stft_plan_destroy(smb_stft_plan* plan) {
  return guarded([&] { delete plan; });
}
int smb_stft_plan_set_stream(smb_stft_plan* plan, void* s) {
  return guarded([&] { plan->ensure_device(); plan->stream.set(s); });
}
int smb_stft_plan_set_path(smb_stft_plan* plan, int path) {
  return guarded([&] {
    if (path < SMB_PATH_AUTO || path > SMB_PATH_PAIR)
      throw smb::invalid_argument("set_path: unknown path");
    plan->path = path;
  });
}
int smb_stft_plan_sync(smb_stft_plan* plan) {
  return guarded([&] { if (plan->device_ready) CK(cudaStreamSynchronize(plan->stream.use)); });
}
int64_t smb_stft_fft_size(const smb_stft_plan* plan) { return plan->geom.fft; }
int64_t smb_stft_hop(const smb_stft_plan* plan) { return plan->geom.hop; }
int64_t smb_stft_bins(const smb_stft_plan* plan) { return plan->geom.bins(); }
int64_t smb_stft_frames(const smb_stft_plan* plan, int64_t n) {
  int64_t r = -1;
  guarded([&] { r = plan->geom.frames(n); });
  return r;
}
int smb_stft_analysis_window(const smb_stft_plan* plan, double* out) {
  return guarded([&] {
    std::memcpy(out, plan->window.data(), plan->window.size() * sizeof(double));
  });
}
int smb_stft_source_indices(const smb_stft_plan* plan, int64_t n, int64_t* out,
                            int64_t* padded_len) {
  return guarded([&] {
    if (n < 1) throw smb::invalid_argument("source_indices: n must be at least 1");
    const int64_t left = plan->geom.left_width(), right = plan->geom.right_width();
    if (padded_len) *padded_len = n + left + right;
    if (!out) return;
    for (int64_t q = 0; q < n + left + right; ++q) {
      const int64_t s = q - left;
      int64_t idx;
      if (s >= 0 && s < n) idx = s;
      else if (plan->geom.pad == smb::kReflect) idx = smb::reflect_index(n, s);
      else if (plan->geom.pad == smb::kEdge) idx = s < 0 ? 0 : n - 1;
      else idx = -1;
      out[q] = idx;
    }
  });
}

}  // extern "C"

namespace {

enum SpecKind { kSpecComplex, kSpecPower };

// SMB_PATH_AUTO: the tensor-core kernel when it covers the call
constexpr bool kAutoPrefersTensor = false;

void check_signal(const char* op, int64_t batch, int64_t n) {
  if (n < 0)
    throw smb::invalid_argument(smb::format(
        "%s: cannot analyse a signal of length %lld (length must be non-negative)", op,
        (long long)n));
  if (batch < 0) throw smb::invalid_argument(smb::format("%s: negative batch", op));
}

// Which fused kernel takes the call: 0 none (generic path), SMB_PATH_FAST the
// CUDA-core register-FFT kernel, SMB_PATH_TENSOR the tcgen05 kernel.
int want_fast(const smb_stft_plan* p, int dtype, const smb::FrameGeom& g, int out_kind,
              const smb_mel_plan* mel) {
  if (p->path == SMB_PATH_GENERIC) return 0;
  const int step = p->fast_step();
  smb::FrameGeom gk = g;
  gk.fft = 2048;
  const bool base = dtype == SMB_F32 && step > 0 &&
                    (!mel || (mel->fast_step == step && !mel->sched_cc.pieces.empty()));
  // the frame-pair kernel: mel output of fft 2048 proper
  const bool ok_pair = dtype == SMB_F32 && step == 1 && mel && out_kind == smb::kFastMel &&
                       !mel->sched_pair.items.empty() &&
                       smb::stft2048p_supports(gk, (int)mel->n_mels, (int)mel->sched_pair.w.size(),
                                               mel->sched_pair.rounds);
  if (p->path == SMB_PATH_PAIR) {
    if (!ok_pair)
      throw smb::invalid_argument(
          "soundml_b200: the frame-pair fft-2048 kernel does not cover this call");
    return SMB_PATH_PAIR;
  }
  if (p->path == SMB_PATH_AUTO && ok_pair) return SMB_PATH_PAIR;
  const bool ok_tc = base && smb::stft2048tc_supports(gk, out_kind, mel ? (int)mel->n_mels : 0,
                                                      mel ? (int)mel->sched_tc.vals.size() : 0,
                                                      mel ? mel->sched_tc.rounds : 0,
                                                      mel ? mel->sched_tc.mpad : 0);
  const bool ok_cc = base && smb::stft2048_supports(gk, out_kind, mel ? (int)mel->n_mels : 0,
                                                    mel ? (int)mel->sched_cc.vals.size() : 0,
                                                    mel ? mel->sched_cc.rounds : 0,
                                                    mel ? mel->sched_cc.mpad : 0);
  if (p->path == SMB_PATH_TENSOR) {
    if (!ok_tc)
      throw smb::invalid_argument(
          "soundml_b200: the tensor-core fft-2048 kernel does not cover this geometry");
    return SMB_PATH_TENSOR;
  }
  if (p->path == SMB_PATH_FAST) {
    if (!ok_cc)
      throw smb::invalid_argument(
          "soundml_b200: the fused fft-2048 kernel does not cover this geometry");
    return SMB_PATH_FAST;
  }
  if (ok_tc && kAutoPrefersTensor) return SMB_PATH_TENSOR;
  return ok_cc ? SMB_PATH_FAST : (ok_tc ? SMB_PATH_TENSOR : 0);
}

smb::Stft2048PairArgs pair_args(const smb_stft_plan* stft, const smb_mel_plan* mel, const void* din,
                                void* dout, int64_t nb, const smb::FrameGeom& g, double power) {
  smb::Stft2048PairArgs a{};
  a.x = (const float*)din;
  a.out = (float*)dout;
  a.batch = nb;
  a.g = g;
  a.g.fft = 2048;
  a.window = stft->d_window32;
  a.tw_pass = stft->d_tw_pass;
  a.tw_post = stft->d_tw_post;
  a.power = (float)power;
  if (mel) {
    a.n_mels = (int)mel->n_mels;
    a.mel_w = mel->sched_pair.d_w;
    a.mel_w_floats = (int)mel->sched_pair.w.size();
    a.mel_items = mel->sched_pair.d_items;
    a.mel_rounds = mel->sched_pair.rounds;
  }
  return a;
}

// x (device) -> spectrum (device).  kind: complex or |X|^power.
void run_spectrum(smb_stft_plan* p, const void* dx, int64_t batch, const smb::FrameGeom& g,
                  int dtype, SpecKind kind, double power, void* dout) {
  cudaStream_t st = p->stream.use;
  const int fast_kind = kind == kSpecComplex ? smb::kFastComplex : smb::kFastPower;
  if (const int which = want_fast(p, dtype, g, fast_kind, nullptr)) {
    smb::Stft2048Args a{};
    a.x = (const float*)dx;
    a.out = (float*)dout;
    a.batch = batch;
    a.g = g;
    a.g.fft = 2048;
    a.bin_step = p->fast_step();
    a.window = p->d_window32;
    a.tw_pass = p->d_tw_pass;
    a.tw_post = p->d_tw_post;
    a.power = (float)power;
    a.dft_images = p->d_dft_images;
    if (which == SMB_PATH_TENSOR) CK(smb::launch_stft2048tc(a, fast_kind, p->sm_count, st));
    else CK(smb::launch_stft2048(a, fast_kind, p->sm_count, st));
  } else {
    CK(smb::launch_stft_generic(dx, dtype, batch, g, p->d_window64, p->d_twiddle64,
                                kind == kSpecComplex ? smb::kModeComplex : smb::kModePower,
                                power, dout, st));
  }
}

void spectrum_call(const char* op, smb_stft_plan* p, const void* x, int64_t batch, int64_t n,
                   int dtype, SpecKind kind, double power, void* out, int mem,
                   int64_t p0 = 0, int64_t p1 = -1) {
  check_signal(op, batch, n);
  const size_t esz = dtype_size(dtype);
  smb::FrameGeom g = p->frame_geom(n);
  if (p1 >= 0) {
    // transform_range (stft.ml:652-666): frames [p0, p1) of the full transform.
    // Frame p0 + p' starts at padded position (p0 + p') hop, so shifting the
    // left width by p0 hop makes the kernels' frame 0 the range's first frame.
    if (p0 < 0 || p0 > p1 || p1 > g.frames)
      throw smb::invalid_argument(smb::format(
          "transform_range: cannot take frames [%lld, %lld) of a %lld-frame transform (the "
          "range must satisfy 0 <= p0 <= p1 <= frames)",
          (long long)p0, (long long)p1, (long long)g.frames));
    g.left = (int)(g.left - p0 * g.hop);
    g.frames = p1 - p0;
  }
  const size_t out_elems =
      (size_t)batch * (size_t)p->geom.bins() * (size_t)g.frames * (kind == kSpecComplex ? 2 : 1);
  if (batch == 0 || g.frames == 0) return;       // frameless spectrum: nothing to write
  p->ensure_device();
  cudaStream_t st = p->stream.use;
  if (mem == SMB_MEM_DEVICE) {
    run_spectrum(p, x, batch, g, dtype, kind, power, out);
    return;
  }
  if (mem != SMB_MEM_HOST) throw smb::invalid_argument("soundml_b200: unknown memory kind");
  p->pipe.execute(st, x, out, batch, (size_t)n * esz, out_elems / (size_t)batch * esz,
                  [&](const void* din, void* dout, int64_t nb) {
                    run_spectrum(p, din, nb, g, dtype, kind, power, dout);
                  });
}

void run_mel_apply(smb_mel_plan* m, const void* ds, int64_t batch, int64_t frames, int dtype,
                   void* dout, cudaStream_t st) {
  CK(smb::launch_mel_apply(ds, dtype, batch, (int)m->bins, frames, (int)m->n_mels, m->d_weights,
                           m->d_band_lo, m->d_band_hi, dout, st));
}

}  // namespace

extern "C" {

int smb_stft_transform(smb_stft_plan* plan, const void* x, int64_t batch, int64_t n,
                       int dtype, void* out, int mem) {
  return guarded([&] {
    spectrum_call("transform", plan, x, batch, n, dtype, kSpecComplex, 1.0, out, mem);
  });
}

int smb_stft_transform_range(smb_stft_plan* plan, const void* x, int64_t batch, int64_t n,
                             int dtype, int64_t p0, int64_t p1, void* out, int mem) {
  return guarded([&] {
    spectrum_call("transform_range", plan, x, batch, n, dtype, kSpecComplex, 1.0, out, mem, p0,
                  p1 < 0 ? 0 : p1);
  });
}

int smb_stft_power_spectrum(smb_stft_plan* plan, const void* x, int64_t batch, int64_t n,
                            int dtype, double power, void* out, int mem) {
  return guarded([&] {
    spectrum_call("power_spectrum", plan, x, batch, n, dtype, kSpecPower, power, out, mem);
  });
}

int smb_stft_nola(const smb_stft_plan* plan) { return plan->nola() ? 1 : 0; }

int64_t smb_stft_output_length(const smb_stft_plan* plan, int64_t frames) {
  int64_t r = -1;
  guarded([&] {
    if (frames < 0)
      throw smb::invalid_argument(smb::format(
          "output_length: cannot size the synthesis of %lld frames (frames must be non-negative)",
          (long long)frames));
    r = plan->output_length(frames);
  });
  return r;
}

int smb_stft_invert(smb_stft_plan* plan, const void* z, int64_t batch, int64_t frames,
                    int in_dtype, int has_length, int64_t length, int out_dtype, void* out,
                    int mem) {
  return guarded([&] {
    smb_stft_plan* p = plan;
    if (batch < 0 || frames < 0)
      throw smb::invalid_argument("invert: batch and frame counts must be non-negative");
    if (has_length && length < 0)                       // stft.ml:776-785
      throw smb::invalid_argument(smb::format(
          "invert: cannot synthesise a signal of length %lld (length must be non-negative)",
          (long long)length));
    if (!p->nola())                                     // stft.ml:744-753
      throw smb::invalid_argument(smb::format(
          "invert: cannot invert a %lld-point window advanced by %lld samples inside a "
          "%lld-point frame (the overlap-added squared window must stay above 1e-10 of its "
          "largest value at every position)",
          (long long)p->geom.win_length, (long long)p->geom.hop, (long long)p->geom.fft));
    const size_t isz = 2 * dtype_size(in_dtype), osz = dtype_size(out_dtype);
    const int64_t left = p->geom.left_width(), hop = p->geom.hop;
    const int64_t out_len = has_length ? length : p->output_length(frames);
    // only the frames the output can reach are inverted (stft.ml:907-915)
    int64_t count = frames;
    if (has_length) count = std::min(frames, (length + left + hop - 1) / hop);
    if (batch == 0 || out_len == 0) return;
    p->ensure_device();
    cudaStream_t st = p->stream.use;
    if (!p->d_folded) p->d_folded = upload(p->folded_square_window());
    auto run = [&](const void* dz, void* dout, int64_t nb) {
      if (count == 0) {                                 // nothing reaches the output: zeros
        CK(cudaMemsetAsync(dout, 0, (size_t)nb * (size_t)out_len * osz, st));
        return;
      }
      smb::IstftArgs a{};
      a.z = dz;
      a.out = dout;
      a.frames = frames;
      a.count = count;
      a.out_len = out_len;
      a.fft = (int)p->geom.fft;
      a.hop = (int)hop;
      a.left = (int)left;
      a.window = p->d_window64;
      a.twiddle = p->d_twiddle64;
      a.folded = p->d_folded;
      a.in_f64 = in_dtype == SMB_F64;
      a.out_f64 = out_dtype == SMB_F64;
      const bool fast = p->path != SMB_PATH_GENERIC && smb::istft2048_supports(a);
      if (!fast && p->path == SMB_PATH_FAST)
        throw smb::invalid_argument(
            "soundml_b200: the fft-2048 synthesis kernel does not cover this geometry");
      if (fast) {
        if (!p->d_window_inv) {
          // 1 / fft of the inverse folded in; frames shorter than 2048 leave a zero tail
          std::vector<float> w(2048, 0.0f);
          for (size_t j = 0; j < (size_t)p->geom.fft; ++j)
            w[j] = (float)(p->window[j] / double(p->geom.fft));
          p->d_window_inv = upload(w);
        }
        CK(smb::launch_istft2048(a, p->d_window_inv, p->d_tw_pass, p->d_tw_post, nb, p->sm_count,
                                 st));
        return;
      }
      CK(smb::launch_istft(a, nb, st));
    };
    if (mem == SMB_MEM_DEVICE) {
      run(z, out, batch);
      return;
    }
    if (mem != SMB_MEM_HOST) throw smb::invalid_argument("soundml_b200: unknown memory kind");
    if (frames == 0) {
      std::memset(out, 0, (size_t)batch * (size_t)out_len * osz);
      return;
    }
    p->pipe.execute(st, z, out, batch, (size_t)p->geom.bins() * (size_t)frames * isz,
                    (size_t)out_len * osz, run);
  });
}

int smb_stft_griffin_lim(smb_stft_plan* plan, const void* s, int64_t batch, int64_t frames,
                         int dtype, int64_t n_iter, double momentum, const void* init_phase,
                         int has_length, int64_t length, void* out, int mem) {
  return guarded([&] {
    smb_stft_plan* p = plan;
    if (batch < 0 || frames < 0)
      throw smb::invalid_argument("griffin_lim: batch and frame counts must be non-negative");
    if (has_length && length < 0)
      throw smb::invalid_argument(smb::format(
          "griffin_lim: cannot synthesise a signal of length %lld (length must be non-negative)",
          (long long)length));
    if (!p->nola())
      throw smb::invalid_argument(smb::format(
          "griffin_lim: cannot invert a %lld-point window advanced by %lld samples inside a "
          "%lld-point frame (the overlap-added squared window must stay above 1e-10 of its "
          "largest value at every position)",
          (long long)p->geom.win_length, (long long)p->geom.hop, (long long)p->geom.fft));
    if (n_iter < 1)
      throw smb::invalid_argument(smb::format(
          "griffin_lim: cannot run %lld iterations (n_iter must be at least 1)",
          (long long)n_iter));
    if (momentum < 0.0)
      throw smb::invalid_argument(smb::format(
          "griffin_lim: cannot use a momentum of %g (momentum must be non-negative)", momentum));
    const size_t esz = dtype_size(dtype);
    const int64_t bins = p->geom.bins(), left = p->geom.left_width(), hop = p->geom.hop;
    const int64_t natural = p->output_length(frames);
    const int64_t out_len = has_length ? length : natural;
    if (batch == 0 || out_len == 0) return;
    if (mem != SMB_MEM_DEVICE && mem != SMB_MEM_HOST)
      throw smb::invalid_argument("soundml_b200: unknown memory kind");
    if (frames == 0) {
      if (mem == SMB_MEM_HOST) std::memset(out, 0, (size_t)batch * (size_t)out_len * esz);
      else { p->ensure_device(); CK(cudaMemsetAsync(out, 0, (size_t)batch * (size_t)out_len * esz, p->stream.use)); }
      return;
    }
    p->ensure_device();
    cudaStream_t st = p->stream.use;
    if (!p->d_folded) p->d_folded = upload(p->folded_square_window());
    const size_t cells = (size_t)batch * (size_t)bins * (size_t)frames;
    // the whole problem stays resident across the iterations
    struct Temp {                       // freed when the call returns or throws
      void* ptr = nullptr;
      void reserve(size_t bytes) { CK(cudaMalloc(&ptr, bytes ? bytes : 1)); }
      ~Temp() { if (ptr) cudaFree(ptr); }
    } d_s, d_phase, d_spec, d_a, d_b, d_y, d_out;
    const void* mags = s;
    const void* phase = init_phase;
    void* dout = out;
    if (mem == SMB_MEM_HOST) {
      d_s.reserve(cells * esz);
      CK(cudaMemcpyAsync(d_s.ptr, s, cells * esz, cudaMemcpyHostToDevice, st));
      mags = d_s.ptr;
      if (init_phase) {
        d_phase.reserve(cells * esz);
        CK(cudaMemcpyAsync(d_phase.ptr, init_phase, cells * esz, cudaMemcpyHostToDevice, st));
        phase = d_phase.ptr;
      }
      d_out.reserve((size_t)batch * (size_t)out_len * esz);
      dout = d_out.ptr;
    }
    d_spec.reserve(cells * sizeof(double2));
    double2* spec = (double2*)d_spec.ptr;
    auto synth = [&](int64_t len, bool named, int out_dtype, void* dst) {
      int64_t count = frames;
      if (named) count = std::min(frames, (len + left + hop - 1) / hop);
      if (count == 0) {
        CK(cudaMemsetAsync(dst, 0, (size_t)batch * (size_t)len * dtype_size(out_dtype), st));
        return;
      }
      smb::IstftArgs a{};
      a.z = spec;
      a.out = dst;
      a.frames = frames;
      a.count = count;
      a.out_len = len;
      a.fft = (int)p->geom.fft;
      a.hop = (int)hop;
      a.left = (int)left;
      a.window = p->d_window64;
      a.twiddle = p->d_twiddle64;
      a.folded = p->d_folded;
      a.in_f64 = 1;
      a.out_f64 = out_dtype == SMB_F64;
      CK(smb::launch_istft(a, batch, st));
    };
    CK(smb::launch_gl_project(mags, phase, dtype == SMB_F64, nullptr, nullptr, 0.0, 1,
                              (long long)cells, spec, st));
    // the loop runs at the natural length, the one geometry that re-analyses to
    // exactly `frames` frames (stft.ml:1000-1008)
    if (natural > 0) {
      d_a.reserve(cells * sizeof(double2));
      d_b.reserve(cells * sizeof(double2));
      d_y.reserve((size_t)batch * (size_t)natural * sizeof(double));
      double2* rebuilt = (double2*)d_a.ptr;
      double2* previous = (double2*)d_b.ptr;
      const double beta = momentum / (1.0 + momentum);
      smb::FrameGeom g = p->frame_geom(natural);
      if (g.frames != frames)
        throw smb::invalid_argument("griffin_lim: the natural length does not re-analyse to the "
                                    "given frame count");
      for (int64_t k = 0; k < n_iter; ++k) {
        synth(natural, false, SMB_F64, d_y.ptr);
        CK(smb::launch_stft_generic(d_y.ptr, SMB_F64, batch, g, p->d_window64, p->d_twiddle64,
                                    smb::kModeComplex, 1.0, rebuilt, st));
        CK(smb::launch_gl_project(mags, nullptr, dtype == SMB_F64, rebuilt,
                                  k == 0 ? nullptr : previous, beta, 0, (long long)cells, spec, st));
        std::swap(rebuilt, previous);
      }
    }
    synth(out_len, has_length != 0, dtype, dout);
    if (mem == SMB_MEM_HOST) {
      CK(cudaMemcpyAsync(out, dout, (size_t)batch * (size_t)out_len * esz, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
    } else {
      // the temporaries die with this call: wait for the work that uses them
      CK(cudaStreamSynchronize(st));
    }
  });
}

// ---- mel ---------------------------------------------------------------------

int smb_mel_plan_create(smb_mel_plan** plan, int64_t n_mels, int64_t sample_rate,
                        int64_t fft_size, double f_min, double f_max, int scale, int norm) {
  return guarded([&] {
    *plan = nullptr;
    double fmax_used = 0.0;
    std::vector<double> w =
        smb::mel_weights(n_mels, sample_rate, fft_size, f_min, f_max, scale, norm, &fmax_used);
    smb_mel_plan* p = new smb_mel_plan;
    p->n_mels = n_mels;
    p->fft = fft_size;
    p->bins = fft_size / 2 + 1;
    p->sample_rate = sample_rate;
    p->f_min = f_min;
    p->f_max = fmax_used;
    p->scale = scale;
    p->norm = norm;
    p->weights = std::move(w);
    p->finish_host();
    *plan = p;
  });
}

int smb_mel_plan_create_with_weights(smb_mel_plan** plan, int64_t n_mels, int64_t fft_size,
                                     const double* weights) {
  return guarded([&] {
    *plan = nullptr;
    if (n_mels < 1)
      throw smb::invalid_argument(smb::format(
          "create: cannot build %lld mel bands (n_mels must be at least 1)", (long long)n_mels));
    if (fft_size < 1)
      throw smb::invalid_argument(smb::format(
          "create: cannot use an FFT of size %lld (fft_size must be at least 1)",
          (long long)fft_size));
    smb_mel_plan* p = new smb_mel_plan;
    p->n_mels = n_mels;
    p->fft = fft_size;
    p->bins = fft_size / 2 + 1;
    p->weights.assign(weights, weights + n_mels * p->bins);
    p->finish_host();
    *plan = p;
  });
}

int smb_mel_plan_destroy(smb_mel_plan* plan) { return guarded([&] { delete plan; }); }
int smb_mel_plan_set_stream(smb_mel_plan* plan, void* s) {
  return guarded([&] { plan->ensure_device(); plan->stream.set(s); });
}
int64_t smb_mel_n_mels(const smb_mel_plan* plan) { return plan->n_mels; }
int64_t smb_mel_bins(const smb_mel_plan* plan) { return plan->bins; }
int64_t smb_mel_fft_size(const smb_mel_plan* plan) { return plan->fft; }
int smb_mel_filterbank(const smb_mel_plan* plan, double* out) {
  return guarded([&] {
    std::memcpy(out, plan->weights.data(), plan->weights.size() * sizeof(double));
  });
}

int smb_mel_apply(smb_mel_plan* plan, const void* s, int64_t batch, int64_t frames, int dtype,
                  void* out, int mem) {
  return guarded([&] {
    if (batch < 0 || frames < 0) throw smb::invalid_argument("apply: negative extent");
    const size_t esz = dtype_size(dtype);
    if (batch == 0 || frames == 0) return;       // zero-size: nothing to reduce (mel.ml:221-227)
    plan->ensure_device();
    cudaStream_t st = plan->stream.use;
    if (mem == SMB_MEM_DEVICE) {
      run_mel_apply(plan, s, batch, frames, dtype, out, st);
      return;
    }
    if (mem != SMB_MEM_HOST) throw smb::invalid_argument("soundml_b200: unknown memory kind");
    const size_t in_bytes = (size_t)batch * plan->bins * frames * esz;
    const size_t out_bytes = (size_t)batch * plan->n_mels * frames * esz;
    void* din = plan->in.ensure(in_bytes);
    void* dout = plan->out.ensure(out_bytes);
    CK(cudaMemcpyAsync(din, s, in_bytes, cudaMemcpyHostToDevice, st));
    run_mel_apply(plan, din, batch, frames, dtype, dout, st);
    CK(cudaMemcpyAsync(out, dout, out_bytes, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  });
}

}  // extern "C"

// Soundml.mel_spectrogram.  max_slot (device, zeroed by the caller, may be null): where
// the kernel leaves the maximum of what it writes; the return value says whether it did
// (only the frame-pair kernel does; slices of a host batch accumulate into the one slot).
static bool mel_spectrogram_impl(smb_stft_plan* stft, smb_mel_plan* mel, const void* x, int64_t batch,
                                 int64_t n, int dtype, double power, void* out, int mem,
                                 unsigned long long* max_slot) {
  bool max_known = false;
  {
    // soundml.ml:12-20
    if (stft->geom.fft != mel->fft)
      throw smb::invalid_argument(smb::format(
          "mel_spectrogram: cannot project a %lld-point STFT through a filterbank built for "
          "an FFT of size %lld (the two configurations must agree on fft_size)",
          (long long)stft->geom.fft, (long long)mel->fft));
    check_signal("power_spectrum", batch, n);
    const size_t esz = dtype_size(dtype);
    const smb::FrameGeom g = stft->frame_geom(n);
    if (batch == 0 || g.frames == 0) return false;
    stft->ensure_device();
    mel->ensure_device();
    cudaStream_t st = stft->stream.use;
    const int fast = want_fast(stft, dtype, g, smb::kFastMel, mel);
    max_known = fast == SMB_PATH_PAIR && max_slot != nullptr;
    auto run = [&](const void* din, void* dout, int64_t nb) {
      if (fast == SMB_PATH_PAIR) {
        smb::Stft2048PairArgs a = pair_args(stft, mel, din, dout, nb, g, power);
        a.max_slot = max_slot;
        CK(smb::launch_stft2048p(a, false, stft->sm_count, st));
      } else if (fast) {
        smb::Stft2048Args a{};
        a.x = (const float*)din;
        a.out = (float*)dout;
        a.batch = nb;
        a.g = g;
        a.g.fft = 2048;
        a.bin_step = stft->fast_step();
        a.window = stft->d_window32;
        a.tw_pass = stft->d_tw_pass;
        a.tw_post = stft->d_tw_post;
        a.n_mels = (int)mel->n_mels;
        a.power = (float)power;
        a.dft_images = stft->d_dft_images;
        const auto& sc = fast == SMB_PATH_TENSOR ? mel->sched_tc : mel->sched_cc;
        a.nnz = (int)sc.vals.size();
        a.vals = sc.d_vals;
        a.mel_pieces = sc.d_pieces;
        a.mel_pcnt = sc.d_pcnt;
        a.mel_rounds = sc.rounds;
        a.mel_mpad = sc.mpad;
        if (fast == SMB_PATH_TENSOR) CK(smb::launch_stft2048tc(a, smb::kFastMel, stft->sm_count, st));
        else CK(smb::launch_stft2048(a, smb::kFastMel, stft->sm_count, st));
      } else {
        // two kernels through a plan-owned power spectrogram
        const size_t spec_bytes = (size_t)nb * stft->geom.bins() * g.frames * esz;
        void* spec = stft->tmp.ensure(spec_bytes);
        CK(smb::launch_stft_generic(din, dtype, nb, g, stft->d_window64, stft->d_twiddle64,
                                    smb::kModePower, power, spec, st));
        run_mel_apply(mel, spec, nb, g.frames, dtype, dout, st);
      }
    };
    if (mem == SMB_MEM_DEVICE) {
      run(x, out, batch);
    } else if (mem == SMB_MEM_HOST) {
      stft->pipe.execute(st, x, out, batch, (size_t)n * esz,
                         (size_t)mel->n_mels * g.frames * esz, run);
    } else {
      throw smb::invalid_argument("soundml_b200: unknown memory kind");
    }
  }
  return max_known;
}

extern "C" {

int smb_mel_spectrogram(smb_stft_plan* stft, smb_mel_plan* mel, const void* x, int64_t batch,
                        int64_t n, int dtype, double power, void* out, int mem) {
  return guarded([&] { mel_spectrogram_impl(stft, mel, x, batch, n, dtype, power, out, mem, nullptr); });
}

// Measurement only: the transform alone on the frame-pair kernel's skeleton (tile
// staging, window, both register-FFT passes, the transposition between them, one
// shared-memory store per value) -- no real-spectrum split, no |X|^2, no mel, nothing
// but one float per thread and tile written to `scratch`.  bench.py times it beside the
// real kernel as the kernel's compute floor.  x: device float32 [batch, n]; scratch:
// device, smb_stft_fft_ceiling_scratch_bytes(plan, batch, n) bytes.
int64_t smb_stft_fft_ceiling_scratch_bytes(const smb_stft_plan* plan, int64_t batch, int64_t n) {
  int64_t r = -1;
  guarded([&] {
    const int64_t frames = plan->geom.frames(n);
    r = (frames + smb::kPairTile - 1) / smb::kPairTile * batch * 128 * 4;
  });
  return r;
}
int smb_stft_fft_ceiling(smb_stft_plan* stft, const void* x, int64_t batch, int64_t n, void* scratch) {
  return guarded([&] {
    check_signal("fft_ceiling", batch, n);
    const smb::FrameGeom g = stft->frame_geom(n);
    if (stft->fast_step() != 1 || !smb::stft2048p_supports(g, 1, 0, 0))
      throw smb::invalid_argument("fft_ceiling: the frame-pair kernel takes fft 2048 with an even hop");
    if (batch == 0 || g.frames == 0) return;
    stft->ensure_device();
    CK(smb::launch_stft2048p(pair_args(stft, nullptr, x, scratch, batch, g, 2.0), true,
                             stft->sm_count, stft->stream.use));
  });
}

// ---- dB conversion and MFCC ------------------------------------------------------

}  // extern "C"

namespace {

const double kDecade = 10.0 / std::log(10.0);     // convert.ml:27

void to_db_call(const char* fn, double gain, int magnitude, const void* x, int64_t count,
                int dtype, double reference, double amin, double top_db, void* out, int mem,
                void* stream) {
  // convert.ml:8-22: checks in the reference's order and wording
  if (!(std::isfinite(reference) && reference > 0.0))
    throw smb::invalid_argument(smb::format("Soundml.Convert.%s: reference must be finite and positive", fn));
  if (!(std::isfinite(amin) && amin > 0.0))
    throw smb::invalid_argument(smb::format("Soundml.Convert.%s: amin must be finite and positive", fn));
  const bool clamp = !std::isnan(top_db);
  if (clamp && !(std::isfinite(top_db) && top_db >= 0.0))
    throw smb::invalid_argument(smb::format("Soundml.Convert.%s: top_db must be finite and non-negative", fn));
  if (count < 0) throw smb::invalid_argument("to_db: negative extent");
  const size_t esz = dtype_size(dtype);
  if (count == 0) return;
  require_device();
  // there is no plan here, hence no plan stream: SMB_STREAM_OWN means the default stream
  cudaStream_t st = stream == SMB_STREAM_OWN ? nullptr : (cudaStream_t)stream;
  const double scale = gain / 10.0 * kDecade;
  const double offset = scale * std::log(std::max(amin, reference));
  // the maximum's slot and the host call's staging are stream-ordered allocations:
  // no device-wide synchronisation, and a device-memory call stays asynchronous
  unsigned long long* slot = nullptr;
  void *din = nullptr, *dout = nullptr;
  auto release = [&] {
    if (slot) cudaFreeAsync(slot, st);
    if (din) cudaFreeAsync(din, st);
    if (dout) cudaFreeAsync(dout, st);
  };
  try {
    CK(cudaMallocAsync((void**)&slot, sizeof(unsigned long long), st));
    const void* src = x;
    void* dst = out;
    if (mem == SMB_MEM_HOST) {
      CK(cudaMallocAsync(&din, (size_t)count * esz, st));
      CK(cudaMallocAsync(&dout, (size_t)count * esz, st));
      CK(cudaMemcpyAsync(din, x, (size_t)count * esz, cudaMemcpyHostToDevice, st));
      src = din;
      dst = dout;
    } else if (mem != SMB_MEM_DEVICE) {
      throw smb::invalid_argument("soundml_b200: unknown memory kind");
    }
    CK(smb::launch_to_db(src, count, dtype, magnitude, amin, scale, offset, clamp,
                         clamp ? top_db : 0.0, slot, dst, st));
    if (mem == SMB_MEM_HOST)
      CK(cudaMemcpyAsync(out, dout, (size_t)count * esz, cudaMemcpyDeviceToHost, st));
  } catch (...) {
    release();
    throw;
  }
  release();
  if (mem == SMB_MEM_HOST) CK(cudaStreamSynchronize(st));   // the host buffer is the caller's again
}

}  // namespace

extern "C" {

int smb_power_to_db(const void* x, int64_t count, int dtype, double reference, double amin,
                    double top_db, void* out, int mem, void* cuda_stream) {
  return guarded([&] {
    to_db_call("power_to_db", 10.0, 0, x, count, dtype, reference, amin, top_db, out, mem, cuda_stream);
  });
}
int smb_amplitude_to_db(const void* x, int64_t count, int dtype, double reference, double amin,
                        double top_db, void* out, int mem, void* cuda_stream) {
  return guarded([&] {
    to_db_call("amplitude_to_db", 20.0, 1, x, count, dtype, reference, amin, top_db, out, mem,
               cuda_stream);
  });
}

int smb_mfcc(smb_stft_plan* stft, smb_mel_plan* mel, const void* x, int64_t batch, int64_t n,
             int dtype, int64_t n_mfcc, double lifter, void* out, int mem) {
  return guarded([&] {
    // soundml.ml:50-70
    if (stft->geom.fft != mel->fft)
      throw smb::invalid_argument(smb::format(
          "mfcc: cannot project a %lld-point STFT through a filterbank built for an FFT of size "
          "%lld (the two configurations must agree on fft_size)",
          (long long)stft->geom.fft, (long long)mel->fft));
    if (n_mfcc < 1 || n_mfcc > mel->n_mels)
      throw smb::invalid_argument(smb::format(
          "mfcc: cannot keep %lld cepstral coefficients of %lld mel bands (n_mfcc must lie in "
          "[1, n_mels])", (long long)n_mfcc, (long long)mel->n_mels));
    const bool has_lifter = !std::isnan(lifter);
    if (has_lifter && !(std::isfinite(lifter) && lifter >= 0.0))
      throw smb::invalid_argument(smb::format(
          "mfcc: cannot lifter with a coefficient of %g (lifter must be finite and non-negative)",
          lifter));
    check_signal("power_spectrum", batch, n);
    const size_t esz = dtype_size(dtype);
    const smb::FrameGeom g = stft->frame_geom(n);
    if (batch == 0 || g.frames == 0) return;
    stft->ensure_device();
    mel->ensure_device();
    cudaStream_t st = stft->stream.use;
    // log-mel needs the whole-tensor maximum, so the mel spectrogram is
    // materialised (plan-owned), then reduced, then transformed
    const size_t mel_bytes = (size_t)batch * mel->n_mels * g.frames * esz;
    const size_t out_bytes = (size_t)batch * n_mfcc * g.frames * esz;
    void* dmel = stft->cepstral.ensure(mel_bytes + out_bytes);
    void* dout = mem == SMB_MEM_HOST ? (void*)((char*)dmel + mel_bytes) : out;
    const int inner_mem = mem == SMB_MEM_HOST ? SMB_MEM_HOST : SMB_MEM_DEVICE;
    if (inner_mem != SMB_MEM_HOST && mem != SMB_MEM_DEVICE)
      throw smb::invalid_argument("soundml_b200: unknown memory kind");
    // the frame-pair kernel leaves the mel spectrogram's maximum in the slot as it writes
    CK(cudaMemsetAsync(mel->d_max, 0, sizeof(unsigned long long), st));
    bool max_known = true;
    if (inner_mem == SMB_MEM_HOST) {
      // host audio goes up in slices of about 64 MB (the whole-tensor maximum needs every
      // slice's mel values before the first cepstral coefficient, so those stay on the
      // device -- a quarter of the audio's size -- but the audio never does at once)
      const int64_t per = std::max<int64_t>(1, (int64_t)(64u << 20) / std::max<int64_t>(1, n * (int64_t)esz));
      for (int64_t b0 = 0; b0 < batch; b0 += per) {
        const int64_t nb = std::min(per, batch - b0);
        void* stage = stft->pipe.in[0].ensure((size_t)std::min(per, batch) * n * esz);
        CK(cudaMemcpyAsync(stage, (const char*)x + (size_t)b0 * n * esz, (size_t)nb * n * esz,
                           cudaMemcpyHostToDevice, st));
        max_known = mel_spectrogram_impl(stft, mel, stage, nb, n, dtype, 2.0,
                                         (char*)dmel + (size_t)b0 * mel->n_mels * g.frames * esz,
                                         SMB_MEM_DEVICE, mel->d_max) && max_known;
      }
    } else {
      max_known = mel_spectrogram_impl(stft, mel, x, batch, n, dtype, 2.0, dmel, SMB_MEM_DEVICE, mel->d_max);
    }
    const double scale = kDecade, offset = scale * std::log(1.0);   // reference 1, amin 1e-10
    CK(smb::launch_mfcc(dmel, dtype, batch, (int)mel->n_mels, g.frames, (int)n_mfcc,
                        mel->dct_table(n_mfcc, has_lifter ? lifter : 0.0), mel->d_max, max_known,
                        1e-10, scale, offset, 80.0, dout, st));
    if (mem == SMB_MEM_HOST) {
      CK(cudaMemcpyAsync(out, dout, out_bytes, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
    }
  });
}

// Convert.power_to_db ?reference ?amin ?top_db (Soundml.mel_spectrogram ?power stft mel x):
// the log-mel spectrogram ML front ends ingest, as the reference composes it
// (convert.ml:20-56 over soundml.ml:12-24).  The mel kernel leaves the whole-tensor
// maximum behind as it writes, so the decibel map with its top_db clamp is ONE pass in
// place over the 128-band output: two launches in all.
int smb_mel_spectrogram_db(smb_stft_plan* stft, smb_mel_plan* mel, const void* x, int64_t batch,
                           int64_t n, int dtype, double power, double reference, double amin,
                           double top_db, void* out, int mem) {
  return guarded([&] {
    const char* fn = "power_to_db";
    if (!(std::isfinite(reference) && reference > 0.0))
      throw smb::invalid_argument(smb::format("Soundml.Convert.%s: reference must be finite and positive", fn));
    if (!(std::isfinite(amin) && amin > 0.0))
      throw smb::invalid_argument(smb::format("Soundml.Convert.%s: amin must be finite and positive", fn));
    const bool clamp = !std::isnan(top_db);
    if (clamp && !(std::isfinite(top_db) && top_db >= 0.0))
      throw smb::invalid_argument(smb::format("Soundml.Convert.%s: top_db must be finite and non-negative", fn));
    if (mem != SMB_MEM_HOST && mem != SMB_MEM_DEVICE)
      throw smb::invalid_argument("soundml_b200: unknown memory kind");
    if (stft->geom.fft != mel->fft || batch < 0 || n < 0) {   // the composition's first checks, its wording
      mel_spectrogram_impl(stft, mel, x, batch, n, dtype, power, out, mem, nullptr);
      return;
    }
    const size_t esz = dtype_size(dtype);
    const smb::FrameGeom g = stft->frame_geom(n);
    if (batch == 0 || g.frames == 0) return;
    stft->ensure_device();
    mel->ensure_device();
    cudaStream_t st = stft->stream.use;
    const int64_t count = batch * mel->n_mels * g.frames;
    void* dmel = mem == SMB_MEM_HOST ? stft->cepstral.ensure((size_t)count * esz) : out;
    CK(cudaMemsetAsync(mel->d_max, 0, sizeof(unsigned long long), st));
    const void* din = x;
    if (mem == SMB_MEM_HOST) {          // the result stays on the device until it is in decibels
      void* stage = stft->pipe.in[0].ensure((size_t)batch * n * esz);
      CK(cudaMemcpyAsync(stage, x, (size_t)batch * n * esz, cudaMemcpyHostToDevice, st));
      din = stage;
    }
    const bool max_known = mel_spectrogram_impl(stft, mel, din, batch, n, dtype, power, dmel,
                                                SMB_MEM_DEVICE, mel->d_max);
    const double scale = kDecade;                                   // gain 10: powers
    const double offset = scale * std::log(std::max(amin, reference));
    if (max_known)
      CK(smb::launch_db_known_max(dmel, count, dtype, amin, scale, offset, clamp, clamp ? top_db : 0.0,
                                  mel->d_max, st));
    else
      CK(smb::launch_to_db(dmel, count, dtype, 0, amin, scale, offset, clamp, clamp ? top_db : 0.0,
                           mel->d_max, dmel, st));
    if (mem == SMB_MEM_HOST) {
      CK(cudaMemcpyAsync(out, dmel, (size_t)count * esz, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
    }
  });
}

// ---- resampler ----------------------------------------------------------------

int smb_resample_plan_create(smb_resample_plan** plan, int64_t sample_rate, int64_t target,
                             int quality, double attenuation, double passband) {
  return guarded([&] {
    *plan = nullptr;
    smb::ResamplePlan rp = smb::resample_plan(sample_rate, target, quality, attenuation, passband);
    smb_resample_plan* p = new smb_resample_plan;
    p->plan = std::move(rp);
    *plan = p;
  });
}
int smb_resample_plan_destroy(smb_resample_plan* plan) { return guarded([&] { delete plan; }); }
int smb_resample_plan_set_stream(smb_resample_plan* plan, void* s) {
  return guarded([&] { plan->ensure_device(); plan->stream.set(s); });
}
int smb_resample_plan_sync(smb_resample_plan* plan) {
  return guarded([&] { if (plan->device_ready) CK(cudaStreamSynchronize(plan->stream.use)); });
}
int smb_resample_plan_set_executor(smb_resample_plan* plan, int exec) {
  return guarded([&] {
    if (exec != SMB_EXEC_DIRECT && exec != SMB_EXEC_PLANNED)
      throw smb::invalid_argument("set_executor: SMB_EXEC_DIRECT or SMB_EXEC_PLANNED");
    plan->executor = exec;
  });
}
int smb_resample_stage_layout(smb_resample_plan* plan, int stage, int group,
                              smb_resample_layout* out) {
  return guarded([&] {
    if (stage < 0 || stage >= (int)plan->plan.stages.size())
      throw smb::invalid_argument("stage_layout: no such stage");
    plan->ensure_device();
    const GemmDevice& gd = plan->gemm[(size_t)stage];
    smb_resample_layout r{};
    r.form = plan->form((size_t)stage);
    r.groups = r.form == SMB_FORM_ROW ? (int)gd.rows_groups.size()
             : r.form == SMB_FORM_WINDOW ? (int)gd.groups.size() : 1;
    if (group < 0 || group >= r.groups) throw smb::invalid_argument("stage_layout: no such column group");
    if (r.form == SMB_FORM_ROW) {
      const smb::GemmRowsArgs& a = gd.rows_groups[(size_t)group].a;
      r.columns = a.l;
      r.col_begin = a.col_begin;
      r.two_issuers = a.two_issuers;
      r.a_tmem = a.a_tmem;
      r.a_stages = a.a_stages;
      r.b_stages = a.b_stages;
      r.shifts = a.shifts;
      r.chunks = a.chunks;
      r.slices = a.slices;
    } else if (r.form == SMB_FORM_WINDOW) {
      r.columns = gd.groups[(size_t)group].width;
      r.col_begin = gd.groups[(size_t)group].col_begin;
      r.chunks = gd.groups[(size_t)group].chunks;
    } else {
      r.columns = (int)plan->plan.stages[(size_t)stage].l;
    }
    *out = r;
  });
}
int smb_resample_describe(const smb_resample_plan* plan, char* buf, size_t cap) {
  return guarded([&] {
    const std::string s = plan->plan.describe();
    if (cap == 0) return;
    const size_t n = std::min(cap - 1, s.size());
    std::memcpy(buf, s.data(), n);
    buf[n] = 0;
  });
}
int64_t smb_resample_l(const smb_resample_plan* plan) { return plan->plan.l; }
int64_t smb_resample_m(const smb_resample_plan* plan) { return plan->plan.m; }
int64_t smb_resample_latency(const smb_resample_plan* plan) { return plan->plan.latency; }
int smb_resample_num_stages(const smb_resample_plan* plan) { return (int)plan->plan.stages.size(); }
int smb_resample_stage_info(const smb_resample_plan* plan, int stage, int64_t* l, int64_t* m,
                            int64_t* k, int* exec, int64_t* ols_n, int64_t* ols_b,
                            int64_t* ols_delta) {
  return guarded([&] {
    if (stage < 0 || stage >= (int)plan->plan.stages.size())
      throw smb::invalid_argument("stage_info: no such stage");
    const smb::ResampleStage& s = plan->plan.stages[(size_t)stage];
    if (l) *l = s.l;
    if (m) *m = s.m;
    if (k) *k = s.k;
    if (exec) *exec = s.exec;
    if (ols_n) *ols_n = s.ols_n;
    if (ols_b) *ols_b = s.ols_b;
    if (ols_delta) *ols_delta = s.ols_delta;
  });
}
int smb_resample_stage_design(const smb_resample_plan* plan, int stage, double* fc,
                              double* beta) {
  return guarded([&] {
    if (stage < 0 || stage >= (int)plan->plan.stages.size())
      throw smb::invalid_argument("stage_design: no such stage");
    if (fc) *fc = plan->plan.stages[(size_t)stage].fc;
    if (beta) *beta = plan->plan.stages[(size_t)stage].beta;
  });
}
int smb_resample_stage_prototype(const smb_resample_plan* plan, int stage, double* out,
                                 int64_t* len) {
  return guarded([&] {
    if (stage < 0 || stage >= (int)plan->plan.stages.size())
      throw smb::invalid_argument("stage_prototype: no such stage");
    const std::vector<double>& h = plan->plan.stages[(size_t)stage].proto;
    if (len) *len = (int64_t)h.size();
    if (out) std::memcpy(out, h.data(), h.size() * sizeof(double));
  });
}
int64_t smb_resample_output_frames(const smb_resample_plan* plan, int64_t n) {
  int64_t r = -1;
  guarded([&] { r = plan->plan.output_frames(n); });
  return r;
}

int smb_resample_apply(smb_resample_plan* plan, const float* x, int64_t batch, int64_t n,
                       float* out, int mem) {
  return guarded([&] {
    if (batch < 0) throw smb::invalid_argument("apply: negative batch");
    const smb::ResamplePlan& rp = plan->plan;
    const int64_t total = rp.output_frames(n);
    if (batch == 0 || n == 0 || total == 0) return;
    plan->ensure_device();
    cudaStream_t st = plan->stream.use;
    // signals are independent: a host batch goes through in slices, the copies of one
    // slice under the kernels of its neighbours (HostPipe)
    auto run = [&](const void* din_v, void* dout_v, int64_t nb) {
      const float* din = (const float*)din_v;
      float* dout = (float*)dout_v;
      if (rp.identity()) {
        CK(cudaMemcpyAsync(dout, din, (size_t)nb * n * 4, cudaMemcpyDeviceToDevice, st));
      } else if (rp.stages.size() == 1) {
        plan->run_stage(0, din, nb, n, total, dout, st);
      } else {
        // cascade (resample.ml:1819-1842): stage 1 emits its exact ceil tail,
        // stage 2 runs over it with zeros beyond and is cut to output_frames.
        const smb::ResampleStage& s1 = rp.stages[0];
        const int64_t n1 = (n * s1.l + s1.m - 1) / s1.m;
        float* mid = (float*)plan->mid.ensure((size_t)nb * n1 * 4);
        plan->run_stage(0, din, nb, n, n1, mid, st);
        plan->run_stage(1, mid, nb, n1, total, dout, st);
      }
    };
    if (mem == SMB_MEM_DEVICE) run(x, out, batch);
    else if (mem == SMB_MEM_HOST) plan->pipe.execute(st, x, out, batch, (size_t)n * 4, (size_t)total * 4, run);
    else throw smb::invalid_argument("soundml_b200: unknown memory kind");
  });
}

// float64 audio: the reference's executor carries both dtypes (resample.ml:72-84);
// here double always takes the direct kernel, in double.
int smb_resample_apply_f64(smb_resample_plan* plan, const double* x, int64_t batch, int64_t n,
                           double* out, int mem) {
  return guarded([&] {
    if (batch < 0) throw smb::invalid_argument("apply: negative batch");
    const smb::ResamplePlan& rp = plan->plan;
    const int64_t total = rp.output_frames(n);
    if (batch == 0 || n == 0 || total == 0) return;
    plan->ensure_device();
    cudaStream_t st = plan->stream.use;
    const size_t in_bytes = (size_t)batch * n * 8, out_bytes = (size_t)batch * total * 8;
    const double* din = x;
    double* dout = out;
    if (mem == SMB_MEM_HOST) {
      double* stage = (double*)plan->in.ensure(in_bytes);
      dout = (double*)plan->out.ensure(out_bytes);
      CK(cudaMemcpyAsync(stage, x, in_bytes, cudaMemcpyHostToDevice, st));
      din = stage;
    } else if (mem != SMB_MEM_DEVICE) {
      throw smb::invalid_argument("soundml_b200: unknown memory kind");
    }
    auto stage_run = [&](size_t i, const double* src, int64_t len, int64_t n_out, double* dst) {
      const smb::ResampleStage& s = rp.stages[i];
      CK(smb::launch_polyphase_direct_f64(src, batch, len, plan->d_bank64[i], (int)s.l, (int)s.m,
                                          (int)s.k, n_out, dst, st));
    };
    if (rp.identity()) {
      CK(cudaMemcpyAsync(dout, din, in_bytes, cudaMemcpyDeviceToDevice, st));
    } else if (rp.stages.size() == 1) {
      stage_run(0, din, n, total, dout);
    } else {
      const smb::ResampleStage& s1 = rp.stages[0];
      const int64_t n1 = (n * s1.l + s1.m - 1) / s1.m;
      double* mid = (double*)plan->mid.ensure((size_t)batch * n1 * 8);
      stage_run(0, din, n, n1, mid);
      stage_run(1, mid, n1, total, dout);
    }
    if (mem == SMB_MEM_HOST) {
      CK(cudaMemcpyAsync(out, dout, out_bytes, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
    }
  });
}

// ---- FIR ----------------------------------------------------------------------

// ---- Resample.Kernel: the chunked form of apply, carry resident on the device ------
//
// resample.ml:1343-1424 (prepare / step / flush / reset), 1844-1909; bound by soundml-io
// (soundml_io.ml:639, 768, 798) and cqt.ml:797-879.  The reference threads per-stage
// histories through its executors; here the state is the raw input still inside some
// future output's dependency cone, kept in device memory, and every step runs the
// offline stage pipeline over a window of it whose origin sits on a whole phase cycle of
// every stage -- so each output is computed with the same phase, taps and summation
// order as in the offline call -- and keeps the outputs whose cone lies inside the
// samples fed so far.  With the direct executor the chunks concatenate to apply's
// result bit for bit; the block executors (overlap-save, tcgen05) agree to rounding.
struct smb_resample_kernel {
  smb_resample_plan* plan = nullptr;
  int64_t channels = 0, max_block = 0;
  int dtype = SMB_F32;
  size_t esz = 4;
  int64_t l = 1, m = 1, reach = 0, grain = 1;
  int64_t fed = 0, emitted = 0, base = 0;
  bool drained = false;
  int64_t cap = 0;                 // samples per channel row of the carry
  DeviceBuffer carry[2];           // [channels][cap]: the retained input [base, fed), ping-pong
  int cur = 0;
  DeviceBuffer win, res;           // the contiguous window and its resampled image

  static int64_t floor_div(int64_t a, int64_t b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }
  int64_t avail_after(int64_t fed_now) const {           // outputs whose cone lies inside fed_now samples
    const int64_t safe = fed_now - reach;
    int64_t avail = safe <= 0 ? 0 : (safe * l + m - 1) / m;
    return std::min(avail, plan->plan.output_frames(fed_now));
  }
  void ensure_cap(int64_t need, cudaStream_t st) {
    if (need <= cap) return;
    const int64_t grown = need + need / 2 + 64;
    DeviceBuffer next;
    next.ensure((size_t)channels * grown * esz);
    if (fed > base)
      CK(cudaMemcpy2DAsync(next.ptr, (size_t)grown * esz, carry[cur].ptr, (size_t)cap * esz,
                           (size_t)(fed - base) * esz, (size_t)channels, cudaMemcpyDeviceToDevice, st));
    CK(cudaStreamSynchronize(st));
    carry[cur].release();
    carry[cur] = next;
    carry[1 - cur].release();
    carry[1 - cur].ensure((size_t)channels * grown * esz);
    cap = grown;
  }
  // outputs [emitted, upto) from a window of the retained input, written to `out`
  // ([channels, upto - emitted], host or device)
  void window(int64_t upto, void* out, int mem, cudaStream_t st) {
    const int64_t first = emitted * m / l - reach;
    const int64_t a0 = std::max<int64_t>(0, floor_div(first, grain) * grain);   // a whole number of grains
    const int64_t len = fed - a0;
    const int64_t total_w = plan->plan.output_frames(len);
    char* w = (char*)win.ensure((size_t)channels * len * esz);
    char* r = (char*)res.ensure((size_t)channels * total_w * esz);
    CK(cudaMemcpy2DAsync(w, (size_t)len * esz, (char*)carry[cur].ptr + (size_t)(a0 - base) * esz,
                         (size_t)cap * esz, (size_t)len * esz, (size_t)channels,
                         cudaMemcpyDeviceToDevice, st));
    const int rc = dtype == SMB_F32
        ? smb_resample_apply(plan, (const float*)w, channels, len, (float*)r, SMB_MEM_DEVICE)
        : smb_resample_apply_f64(plan, (const double*)w, channels, len, (double*)r, SMB_MEM_DEVICE);
    if (rc != SMB_OK) throw cuda_failure(t_error);
    const int64_t o0 = a0 * l / m;                         // a0 is a whole number of input cycles
    const int64_t count = upto - emitted;
    CK(cudaMemcpy2DAsync(out, (size_t)count * esz, r + (size_t)(emitted - o0) * esz,
                         (size_t)total_w * esz, (size_t)count * esz, (size_t)channels,
                         mem == SMB_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, st));
    emitted = upto;
    // drop what no future output can reach (kept on a grain boundary)
    const int64_t keep = std::max<int64_t>(0, floor_div(emitted * m / l - reach, grain) * grain);
    if (keep > base) {
      if (fed > keep)
        CK(cudaMemcpy2DAsync(carry[1 - cur].ptr, (size_t)cap * esz,
                             (char*)carry[cur].ptr + (size_t)(keep - base) * esz, (size_t)cap * esz,
                             (size_t)(fed - keep) * esz, (size_t)channels, cudaMemcpyDeviceToDevice, st));
      cur = 1 - cur;
      base = keep;
    }
  }
};

int smb_resample_kernel_create(smb_resample_kernel** kernel, smb_resample_plan* plan, int dtype,
                               int64_t channels, int64_t max_block) {
  return guarded([&] {
    *kernel = nullptr;
    // resample.ml:1346-1356, the reference's wording
    if (channels < 1)
      throw smb::invalid_argument(smb::format(
          "prepare: cannot resample %lld channels (channels must be at least 1)", (long long)channels));
    if (max_block < 1)
      throw smb::invalid_argument(smb::format(
          "prepare: cannot accept blocks of %lld samples (max_block must be at least 1)",
          (long long)max_block));
    smb_resample_kernel* k = new smb_resample_kernel;
    k->plan = plan;
    k->channels = channels;
    k->max_block = max_block;
    k->dtype = dtype;
    k->esz = dtype_size(dtype);
    const smb::ResamplePlan& rp = plan->plan;
    k->l = rp.l;
    k->m = rp.m;
    // dependency cone of one output, in input samples either side of floor(i M / L)
    if (rp.stages.empty()) {
      k->reach = 0;
      k->grain = 1;
    } else if (rp.stages.size() == 1) {
      k->reach = rp.stages[0].k + 1;
      k->grain = rp.stages[0].m;
    } else {
      const int64_t l1 = rp.stages[0].l, m1 = rp.stages[0].m, k1 = rp.stages[0].k;
      const int64_t m2 = rp.stages[1].m, k2 = rp.stages[1].k;
      k->reach = k1 + ((k2 + 2) * m1 + l1 - 1) / l1 + 2;
      int64_t g = m1;                                     // window origin: whole cycles of both stages
      while ((g / m1 * l1) % m2) g += m1;
      k->grain = g;
    }
    *kernel = k;
  });
}
int smb_resample_kernel_destroy(smb_resample_kernel* k) {
  return guarded([&] {
    if (!k) return;
    k->carry[0].release();
    k->carry[1].release();
    k->win.release();
    k->res.release();
    delete k;
  });
}
int smb_resample_kernel_reset(smb_resample_kernel* k) {
  return guarded([&] {
    k->fed = k->emitted = k->base = 0;
    k->drained = false;
  });
}
int64_t smb_resample_kernel_step_frames(const smb_resample_kernel* k, int64_t n) {
  if (k->drained || n <= 0) return 0;
  if (k->l == k->m) return n;
  const int64_t avail = k->avail_after(k->fed + n);
  return avail > k->emitted ? avail - k->emitted : 0;
}
int64_t smb_resample_kernel_flush_frames(const smb_resample_kernel* k) {
  if (k->drained || k->fed == 0) return 0;
  const int64_t total = k->plan->plan.output_frames(k->fed);
  return total > k->emitted ? total - k->emitted : 0;
}
int smb_resample_kernel_step(smb_resample_kernel* k, const void* chunk, int64_t n, void* out,
                             int mem) {
  return guarded([&] {
    if (k->drained)
      throw smb::invalid_argument(
          "step: cannot feed a drained kernel (flush consumed the tail; reset before reusing)");
    if (n < 0 || n > k->max_block)
      throw smb::invalid_argument(smb::format(
          "step: cannot feed a %lld-sample chunk (max_block is %lld)", (long long)n,
          (long long)k->max_block));
    if (mem != SMB_MEM_HOST && mem != SMB_MEM_DEVICE)
      throw smb::invalid_argument("soundml_b200: unknown memory kind");
    if (n == 0) return;
    k->plan->ensure_device();
    cudaStream_t st = k->plan->stream.use;
    const cudaMemcpyKind in_kind = mem == SMB_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    if (k->l == k->m) {                                   // identity: forward a copy
      CK(cudaMemcpyAsync(out, chunk, (size_t)k->channels * n * k->esz,
                         mem == SMB_MEM_HOST ? cudaMemcpyHostToHost : cudaMemcpyDeviceToDevice, st));
      k->fed += n;
      k->emitted = k->base = k->fed;
      if (mem == SMB_MEM_HOST) CK(cudaStreamSynchronize(st));
      return;
    }
    k->ensure_cap(k->fed - k->base + n, st);
    CK(cudaMemcpy2DAsync((char*)k->carry[k->cur].ptr + (size_t)(k->fed - k->base) * k->esz,
                         (size_t)k->cap * k->esz, chunk, (size_t)n * k->esz, (size_t)n * k->esz,
                         (size_t)k->channels, in_kind, st));
    k->fed += n;
    const int64_t avail = k->avail_after(k->fed);
    if (avail > k->emitted) k->window(avail, out, mem, st);
    if (mem == SMB_MEM_HOST) CK(cudaStreamSynchronize(st));
  });
}
int smb_resample_kernel_flush(smb_resample_kernel* k, void* out, int mem) {
  return guarded([&] {
    if (k->drained) return;
    k->drained = true;
    if (mem != SMB_MEM_HOST && mem != SMB_MEM_DEVICE)
      throw smb::invalid_argument("soundml_b200: unknown memory kind");
    const int64_t total = k->fed ? k->plan->plan.output_frames(k->fed) : 0;
    if (total <= k->emitted) return;
    k->plan->ensure_device();
    cudaStream_t st = k->plan->stream.use;
    k->window(total, out, mem, st);
    if (mem == SMB_MEM_HOST) CK(cudaStreamSynchronize(st));
  });
}

int smb_fir_plan_create(smb_fir_plan** plan, const double* h, int64_t taps) {
  return guarded([&] {
    *plan = nullptr;
    if (taps < 1 || (taps % 2) == 0)
      throw smb::invalid_argument(smb::format(
          "fir: cannot use a %lld-tap filter (taps must be odd and at least 1, so the group "
          "delay is integral)", (long long)taps));
    smb_fir_plan* p = new smb_fir_plan;
    p->h.assign(h, h + taps);
    p->k = (taps - 1) / 2;
    *plan = p;
  });
}
int smb_fir_plan_destroy(smb_fir_plan* plan) { return guarded([&] { delete plan; }); }
int smb_fir_plan_set_stream(smb_fir_plan* plan, void* s) {
  return guarded([&] { plan->ensure_device(); plan->stream.set(s); });
}
int smb_fir_apply(smb_fir_plan* plan, const float* x, int64_t batch, int64_t n, float* out,
                  int method, int mem) {
  return guarded([&] {
    if (batch < 0 || n < 0) throw smb::invalid_argument("fir: negative extent");
    if (method != SMB_EXEC_DIRECT && method != SMB_EXEC_OLS && method != SMB_EXEC_PLANNED)
      throw smb::invalid_argument(
          "fir: method must be SMB_EXEC_DIRECT, SMB_EXEC_OLS or SMB_EXEC_PLANNED");
    if (batch == 0 || n == 0) return;
    plan->ensure_device();
    if (method == SMB_EXEC_PLANNED)
      method = plan->ols.plan.ok && plan->k >= 8 ? SMB_EXEC_OLS : SMB_EXEC_DIRECT;
    if (method == SMB_EXEC_OLS && !plan->ols.plan.ok)
      throw smb::invalid_argument(
          "fir: this filter is too long for the overlap-save kernel (use the direct method)");
    cudaStream_t st = plan->stream.use;
    auto run = [&](const void* din, void* dout, int64_t nb) {
      if (method == SMB_EXEC_OLS)
        plan->ols.run((const float*)din, nb, n, n, (float*)dout, st);
      else
        CK(smb::launch_polyphase_direct((const float*)din, nb, n, plan->d_bank, 1, 1, (int)plan->k, n,
                                        (float*)dout, st));
    };
    if (mem == SMB_MEM_DEVICE) run(x, out, batch);
    else if (mem == SMB_MEM_HOST) plan->pipe.execute(st, x, out, batch, (size_t)n * 4, (size_t)n * 4, run);
    else throw smb::invalid_argument("soundml_b200: unknown memory kind");
  });
}
// ---- soundml-io device ingest ------------------------------------------------------
int64_t smb_ingest_block_frames(int64_t channels, int64_t elt, int64_t advertised) {
  // soundml_io.ml:532-536
  if (channels < 1 || elt < 1) return -1;
  const int64_t budget = 4194304 / (channels * elt);
  const int64_t block = std::min<int64_t>(1048576, std::max<int64_t>(4096, budget));
  return advertised > 0 ? std::min(block, std::max<int64_t>(4096, advertised)) : block;
}
int smb_ingest_layout(const void* interleaved, int64_t frames, int64_t channels, int mode,
                      int dtype, void* out, int64_t out_total, int64_t out_off, int mem_in,
                      int mem_out, void* cuda_stream) {
  return guarded([&] {
    // geometry, as soundml_io_check_geometry (soundml_io_stubs.c:1150-1172)
    if (mode != SMB_INGEST_PLANAR && mode != SMB_INGEST_DOWNMIX)
      throw smb::invalid_argument("ingest: mode must be SMB_INGEST_PLANAR or SMB_INGEST_DOWNMIX");
    if (channels < 1 || channels > 65535)
      throw smb::invalid_argument("ingest: channels must lie in [1, 65535]");
    if (frames < 0 || out_off < 0 || out_total < 0 || out_off + frames > out_total)
      throw smb::invalid_argument("ingest: the block does not fit the destination "
                                  "(need 0 <= out_off, out_off + frames <= out_total)");
    const size_t esz = dtype_size(dtype);
    if ((mem_in != SMB_MEM_HOST && mem_in != SMB_MEM_DEVICE) ||
        (mem_out != SMB_MEM_HOST && mem_out != SMB_MEM_DEVICE))
      throw smb::invalid_argument("soundml_b200: unknown memory kind");
    if (frames == 0) return;
    require_device();
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const int64_t width = mode == SMB_INGEST_PLANAR ? channels : 1;
    static thread_local DeviceBuffer stage_in, stage_out;
    const void* din = interleaved;
    if (mem_in == SMB_MEM_HOST) {
      void* up = stage_in.ensure((size_t)frames * channels * esz);
      CK(cudaMemcpyAsync(up, interleaved, (size_t)frames * channels * esz, cudaMemcpyHostToDevice, st));
      din = up;
    }
    if (mem_out == SMB_MEM_DEVICE) {
      CK(smb::launch_ingest_layout(din, dtype, frames, (int)channels, mode == SMB_INGEST_DOWNMIX,
                                   (char*)out + (size_t)out_off * esz, out_total, st));
      if (mem_in == SMB_MEM_HOST) CK(cudaStreamSynchronize(st));   // the host block may be reused
    } else {
      void* dn = stage_out.ensure((size_t)frames * width * esz);
      CK(smb::launch_ingest_layout(din, dtype, frames, (int)channels, mode == SMB_INGEST_DOWNMIX, dn,
                                   frames, st));
      CK(cudaMemcpy2DAsync((char*)out + (size_t)out_off * esz, (size_t)out_total * esz, dn,
                           (size_t)frames * esz, (size_t)frames * esz, (size_t)width,
                           cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
    }
  });
}

// ---- the reader: decode loop staging (soundml_io.ml:742-807, soundml_io_stubs.c:1175-1239) ----
//
// The decoder (libsndfile, on the CPU) fills one of two PINNED interleaved blocks while the
// other one's upload, layout pass and resampler step are still running on the device:
//   staging()  ->  sf_readf_* writes there  ->  submit(frames)  ->  staging() (the other block) ...
// submit only enqueues: the upload on a copy stream, then -- behind an event -- the layout
// kernel and the streaming resampler on the compute stream, writing straight into the caller's
// device destination.  Frame counts are integer bookkeeping known before anything runs.
struct smb_ingest {
  int bound_device = 0;
  int64_t channels = 0, width = 0, max_block = 0;
  int mode = SMB_INGEST_PLANAR, dtype = SMB_F32;
  size_t esz = 4;
  smb_resample_plan* plan = nullptr;        // null: native rate
  smb_resample_kernel* kernel = nullptr;
  void* staging[2] = {nullptr, nullptr};
  DeviceBuffer up[2], planar;
  cudaStream_t copy = nullptr, compute = nullptr;
  bool own_compute = false;
  cudaEvent_t copied[2] = {nullptr, nullptr}, consumed[2] = {nullptr, nullptr};
  bool in_flight[2] = {false, false};
  int cur = 0;
  bool finished = false;
  int64_t frames_in = 0, frames_out = 0;
};

int smb_ingest_create(smb_ingest** reader, int64_t channels, int64_t sample_rate, int64_t target,
                      int mode, int quality, int64_t max_block, int dtype) {
  return guarded([&] {
    *reader = nullptr;
    if (mode != SMB_INGEST_PLANAR && mode != SMB_INGEST_DOWNMIX)
      throw smb::invalid_argument("ingest: mode must be SMB_INGEST_PLANAR or SMB_INGEST_DOWNMIX");
    if (channels < 1 || channels > 65535)
      throw smb::invalid_argument("ingest: channels must lie in [1, 65535]");
    if (max_block < 0) throw smb::invalid_argument("ingest: max_block must not be negative");
    const size_t esz = dtype_size(dtype);
    require_device();
    std::unique_ptr<smb_ingest> r(new smb_ingest);
    CK(cudaGetDevice(&r->bound_device));
    r->channels = channels;
    r->width = mode == SMB_INGEST_PLANAR ? channels : 1;
    r->mode = mode;
    r->dtype = dtype;
    r->esz = esz;
    r->max_block = max_block > 0 ? max_block : smb_ingest_block_frames(channels, (int64_t)esz, 0);
    if (target > 0 && target != sample_rate) {
      if (smb_resample_plan_create(&r->plan, sample_rate, target, quality, 0.0, 0.0) != SMB_OK)
        throw smb::invalid_argument(t_error);
      if (smb_resample_kernel_create(&r->kernel, r->plan, dtype, r->width, r->max_block) != SMB_OK) {
        const std::string msg = t_error;
        smb_resample_plan_destroy(r->plan);
        throw smb::invalid_argument(msg);
      }
      r->plan->ensure_device();
      r->compute = r->plan->stream.use;
    } else {
      CK(cudaStreamCreateWithFlags(&r->compute, cudaStreamNonBlocking));
      r->own_compute = true;
    }
    CK(cudaStreamCreateWithFlags(&r->copy, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      CK(cudaMallocHost(&r->staging[i], (size_t)r->max_block * channels * esz));
      r->up[i].ensure((size_t)r->max_block * channels * esz);
      CK(cudaEventCreateWithFlags(&r->copied[i], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&r->consumed[i], cudaEventDisableTiming));
    }
    r->planar.ensure((size_t)r->max_block * r->width * esz);
    *reader = r.release();
  });
}
int smb_ingest_destroy(smb_ingest* r) {
  return guarded([&] {
    if (!r) return;
    if (r->copy) cudaStreamSynchronize(r->copy);
    if (r->compute) cudaStreamSynchronize(r->compute);
    for (int i = 0; i < 2; ++i) {
      if (r->staging[i]) cudaFreeHost(r->staging[i]);
      r->up[i].release();
      if (r->copied[i]) cudaEventDestroy(r->copied[i]);
      if (r->consumed[i]) cudaEventDestroy(r->consumed[i]);
    }
    r->planar.release();
    if (r->kernel) smb_resample_kernel_destroy(r->kernel);
    if (r->plan) smb_resample_plan_destroy(r->plan);
    if (r->copy) cudaStreamDestroy(r->copy);
    if (r->own_compute && r->compute) cudaStreamDestroy(r->compute);
    delete r;
  });
}
int64_t smb_ingest_max_block(const smb_ingest* r) { return r->max_block; }
int smb_ingest_staging(smb_ingest* r, void** block) {
  return guarded([&] {
    same_device(r->bound_device);
    // the upload that last read this block (two submits ago) must have left the host
    if (r->in_flight[r->cur]) {
      CK(cudaEventSynchronize(r->copied[r->cur]));
      r->in_flight[r->cur] = false;
    }
    *block = r->staging[r->cur];
  });
}
int64_t smb_ingest_submit_frames(const smb_ingest* r, int64_t frames) {
  if (r->finished || frames <= 0) return 0;
  return r->kernel ? smb_resample_kernel_step_frames(r->kernel, frames) : frames;
}
int smb_ingest_submit(smb_ingest* r, int64_t frames, void* out_device) {
  return guarded([&] {
    same_device(r->bound_device);
    if (r->finished) throw smb::invalid_argument("ingest: cannot feed a finished reader");
    if (frames < 0 || frames > r->max_block)
      throw smb::invalid_argument(smb::format("ingest: cannot feed a %lld-frame block (max_block is %lld)",
                                              (long long)frames, (long long)r->max_block));
    if (frames == 0) return;
    const int b = r->cur;
    // the layout pass that last read up[b] must be done before the copy overwrites it
    CK(cudaStreamWaitEvent(r->copy, r->consumed[b], 0));
    CK(cudaMemcpyAsync(r->up[b].ptr, r->staging[b], (size_t)frames * r->channels * r->esz,
                       cudaMemcpyHostToDevice, r->copy));
    CK(cudaEventRecord(r->copied[b], r->copy));
    r->in_flight[b] = true;
    CK(cudaStreamWaitEvent(r->compute, r->copied[b], 0));
    const int64_t released = smb_ingest_submit_frames(r, frames);
    if (r->kernel) {
      CK(smb::launch_ingest_layout(r->up[b].ptr, r->dtype, frames, (int)r->channels,
                                   r->mode == SMB_INGEST_DOWNMIX, r->planar.ptr, frames, r->compute));
      CK(cudaEventRecord(r->consumed[b], r->compute));
      if (smb_resample_kernel_step(r->kernel, r->planar.ptr, frames, out_device, SMB_MEM_DEVICE) != SMB_OK)
        throw cuda_failure(t_error);
    } else {
      CK(smb::launch_ingest_layout(r->up[b].ptr, r->dtype, frames, (int)r->channels,
                                   r->mode == SMB_INGEST_DOWNMIX, out_device, frames, r->compute));
      CK(cudaEventRecord(r->consumed[b], r->compute));
    }
    r->frames_in += frames;
    r->frames_out += released;
    r->cur = 1 - b;
  });
}
int64_t smb_ingest_finish_frames(const smb_ingest* r) {
  return (r->finished || !r->kernel) ? 0 : smb_resample_kernel_flush_frames(r->kernel);
}
int smb_ingest_finish(smb_ingest* r, void* out_device) {
  return guarded([&] {
    same_device(r->bound_device);
    if (r->finished) return;
    const int64_t tail = smb_ingest_finish_frames(r);
    r->finished = true;
    if (r->kernel && smb_resample_kernel_flush(r->kernel, out_device, SMB_MEM_DEVICE) != SMB_OK)
      throw cuda_failure(t_error);
    r->frames_out += tail;
  });
}
int smb_ingest_sync(smb_ingest* r) {
  return guarded([&] {
    CK(cudaStreamSynchronize(r->copy));
    CK(cudaStreamSynchronize(r->compute));
  });
}
void* smb_ingest_stream(smb_ingest* r) { return (void*)r->compute; }

int smb_fir_design_lowpass(int64_t k, double cutoff, double attenuation, double* out) {
  return guarded([&] {
    if (k < 1) throw smb::invalid_argument("fir: k must be at least 1");
    if (!(cutoff > 0.0 && cutoff <= 1.0))
      throw smb::invalid_argument("fir: cutoff must lie in (0, 1] Nyquist units");
    std::vector<double> h = smb::design_prototype(1, k, cutoff, smb::kaiser_beta(attenuation));
    std::memcpy(out, h.data(), h.size() * sizeof(double));
  });
}

}  // extern "C"
