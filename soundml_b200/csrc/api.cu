// C ABI of libsoundml_b200.so (see include/soundml_b200.h).
//
// Every device table, stream, event and staging buffer is held by a unique_ptr owner.
// Preconditions are checked in the reference's order and with its messages
// (SMB_EINVAL = Invalid_argument); CUDA failures are SMB_ECUDA.  There is no
// CPU execution path in this library.
#include <cuda_runtime.h>

#include <memory>
#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/soundml_b200.h"
#include "host_design.h"
#include "kernel_tables.h"
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

// Owners of CUDA resources.  The deleters ignore errors: teardown has no one to report to.
struct DeviceFree {
  void operator()(void* p) const { cudaFree(p); }
};
struct PinnedFree {
  void operator()(void* p) const { cudaFreeHost(p); }
};
struct StreamOrderedFree {                      // cudaMallocAsync scratch, freed on its stream
  cudaStream_t st = nullptr;
  void operator()(void* p) const { cudaFreeAsync(p, st); }
};
struct StreamDestroy {
  void operator()(cudaStream_t s) const { cudaStreamDestroy(s); }
};
struct EventDestroy {
  void operator()(cudaEvent_t e) const { cudaEventDestroy(e); }
};
template <typename T>
using device_ptr = std::unique_ptr<T, DeviceFree>;
using pinned_ptr = std::unique_ptr<void, PinnedFree>;
using scratch_ptr = std::unique_ptr<void, StreamOrderedFree>;
using stream_ptr = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, StreamDestroy>;
using event_ptr = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, EventDestroy>;

template <typename T = void>
device_ptr<T> device_alloc(size_t bytes) {
  void* p = nullptr;
  CK(cudaMalloc(&p, bytes));
  return device_ptr<T>(static_cast<T*>(p));
}
scratch_ptr scratch_alloc(size_t bytes, cudaStream_t st) {
  void* p = nullptr;
  CK(cudaMallocAsync(&p, bytes, st));
  return scratch_ptr(p, StreamOrderedFree{st});
}
stream_ptr new_stream() {
  cudaStream_t s = nullptr;
  CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  return stream_ptr(s);
}
event_ptr new_event() {
  cudaEvent_t e = nullptr;
  CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  return event_ptr(e);
}

// A device buffer that only ever grows.
struct DeviceBuffer {
  device_ptr<void> ptr;
  size_t cap = 0;
  void* ensure(size_t bytes) {
    if (bytes > cap) {
      ptr.reset();
      cap = 0;
      ptr = device_alloc(bytes);
      cap = bytes;
    }
    return ptr.get();
  }
};

template <typename T>
device_ptr<T> upload(const std::vector<T>& v) {
  if (v.empty()) return nullptr;
  device_ptr<T> d = device_alloc<T>(v.size() * sizeof(T));
  CK(cudaMemcpy(d.get(), v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  return d;
}

struct StreamOwner {
  stream_ptr own;
  cudaStream_t use = nullptr;
  void create() {
    own = new_stream();
    use = own.get();
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
    cudaStream_t next = external == SMB_STREAM_OWN ? own.get() : (cudaStream_t)external;
    if (next != use) {
      const cudaError_t e = cudaStreamSynchronize(use);
      if (e != cudaSuccess) {
        cudaGetLastError();
        if (e != cudaErrorInvalidResourceHandle && e != cudaErrorContextIsDestroyed) CK(e);
      }
    }
    use = next;
  }
};

// Host-memory calls stage the batch through the device in slices on three
// streams (H2D, compute, D2H) with two buffer slots, so the PCIe transfers of
// neighbouring slices overlap each other and the kernels (full-duplex link).
// With pageable host memory the copies degrade to synchronous staging; pinned
// memory (smb_host_alloc_pinned) gets the full overlap.
struct HostPipe {
  struct Streams {
    stream_ptr h2d, d2h;
    event_ptr ev_in[2], ev_run[2], ev_out[2];
  };
  std::unique_ptr<Streams> streams;  // created by the first host-memory call
  DeviceBuffer in[2], out[2];        // (the log-mel calls also stage through in[0], without the streams)
  // run(din, dout, items) enqueues the kernels for `items` batch items on `compute`.
  template <typename Run>
  void execute(cudaStream_t compute, const void* x, void* out_host, int64_t batch,
               size_t in_item, size_t out_item, Run&& run) {
    if (!streams) {
      auto s = std::make_unique<Streams>();
      s->h2d = new_stream();
      s->d2h = new_stream();
      for (int i = 0; i < 2; ++i) {
        s->ev_in[i] = new_event();
        s->ev_run[i] = new_event();
        s->ev_out[i] = new_event();
      }
      streams = std::move(s);
    }
    cudaStream_t h2d = streams->h2d.get(), d2h = streams->d2h.get();
    const size_t slice_bytes = (size_t)64 << 20;
    int64_t per = (int64_t)(slice_bytes / std::max<size_t>(1, in_item + out_item));
    per = std::max<int64_t>(1, std::min<int64_t>(per, batch));
    const int64_t slices = (batch + per - 1) / per;
    for (int64_t i = 0; i < slices; ++i) {
      const int slot = (int)(i & 1);
      cudaEvent_t ev_in = streams->ev_in[slot].get(), ev_run = streams->ev_run[slot].get(),
                  ev_out = streams->ev_out[slot].get();
      const int64_t b0 = i * per, nb = std::min<int64_t>(per, batch - b0);
      void* din = in[slot].ensure((size_t)per * in_item);
      void* dout = out[slot].ensure((size_t)per * out_item);
      if (i >= 2) CK(cudaStreamWaitEvent(h2d, ev_run, 0));      // input slot consumed
      CK(cudaMemcpyAsync(din, (const char*)x + (size_t)b0 * in_item, (size_t)nb * in_item,
                         cudaMemcpyHostToDevice, h2d));
      CK(cudaEventRecord(ev_in, h2d));
      CK(cudaStreamWaitEvent(compute, ev_in, 0));
      if (i >= 2) CK(cudaStreamWaitEvent(compute, ev_out, 0));  // output slot drained
      run(din, dout, nb);
      CK(cudaEventRecord(ev_run, compute));
      CK(cudaStreamWaitEvent(d2h, ev_run, 0));
      CK(cudaMemcpyAsync((char*)out_host + (size_t)b0 * out_item, dout, (size_t)nb * out_item,
                         cudaMemcpyDeviceToHost, d2h));
      CK(cudaEventRecord(ev_out, d2h));
    }
    CK(cudaStreamSynchronize(d2h));
    CK(cudaStreamSynchronize(compute));
  }
};

void check_mem(int mem) {
  if (mem != SMB_MEM_DEVICE && mem != SMB_MEM_HOST)
    throw smb::invalid_argument("soundml_b200: unknown memory kind");
}

// run(din, dout, items) over the caller's device buffers, or over a host batch in
// slices through `pipe`.
template <typename Run>
void dispatch(int mem, HostPipe& pipe, cudaStream_t st, const void* x, void* out, int64_t batch,
              size_t in_item, size_t out_item, Run&& run) {
  check_mem(mem);
  if (mem == SMB_MEM_DEVICE) run(x, out, batch);
  else pipe.execute(st, x, out, batch, in_item, out_item, run);
}

// A call without a plan: run(src, dst) on the caller's device buffers, or, for host
// memory, through stream-ordered scratch (as the dB conversions stage), returning once the
// result is in `out`.
template <typename Run>
void on_stream(int mem, cudaStream_t st, const void* x, size_t in_bytes, void* out, size_t out_bytes,
               Run&& run) {
  if (mem == SMB_MEM_DEVICE) return run(x, out);
  scratch_ptr din = scratch_alloc(in_bytes, st);
  scratch_ptr dout = scratch_alloc(out_bytes, st);
  CK(cudaMemcpyAsync(din.get(), x, in_bytes, cudaMemcpyHostToDevice, st));
  run(din.get(), dout.get());
  CK(cudaMemcpyAsync(out, dout.get(), out_bytes, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));   // the host buffer is the caller's again
}

size_t dtype_size(int dtype) {
  if (dtype == SMB_F32) return 4;
  if (dtype == SMB_F64) return 8;
  throw smb::invalid_argument("soundml_b200: dtype must be SMB_F32 or SMB_F64");
}

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

// A plan's Device on the current device, with its stream and the device's multiprocessor count.
template <typename Device>
std::unique_ptr<Device> new_device() {
  require_device();
  auto d = std::make_unique<Device>();
  CK(cudaGetDevice(&d->device));
  CK(cudaDeviceGetAttribute(&d->sm_count, cudaDevAttrMultiProcessorCount, d->device));
  d->stream.create();
  return d;
}

// ============================ plan types =====================================

struct smb_stft_plan {
  smb::StftGeometry geom;
  std::vector<double> window;        // analysis window, fft doubles
  int path = SMB_PATH_AUTO;
  // Everything the plan has on its device; null until the first device call.
  struct Device {
    int device = 0, sm_count = 0;
    StreamOwner stream;
    device_ptr<double> d_window64;
    device_ptr<double2> d_twiddle64;
    device_ptr<double> d_folded;       // synthesis: folded squared window, one entry per residue
    device_ptr<float> d_window_inv;    // synthesis fast path: window / 2048
    device_ptr<float> d_window32;      // fast path tables (fft 2048 only)
    device_ptr<float2> d_tw_pass;
    device_ptr<float2> d_tw_post;
    device_ptr<__half> d_dft_images;   // tensor-core kernel: split-fp16 images of the 32-point DFT
  };
  std::unique_ptr<Device> dev;       // declared before the buffers used on its stream
  HostPipe pipe;
  DeviceBuffer tmp;        // power spectrogram of the generic mel path
  DeviceBuffer cepstral;   // mel spectrogram (+ host-call output) of the MFCC path
  // the effects' spectra: the input's (effect_in) and the effect's result (effect_out):
  // time_stretch's stretched copy, hpss_audio's separated parts
  DeviceBuffer effect_in, effect_out;

  void ensure_device() {
    if (dev) return same_device(dev->device);
    auto d = new_device<Device>();
    d->d_window64 = upload(window);
    d->d_twiddle64 = upload(smb::unit_roots<double2>(geom.fft, geom.fft));
    if (fast_step() > 0) {
      // shorter frames run zero-padded to 2048: the window's tail is zero
      std::vector<float> w32(2048, 0.0f);
      for (int64_t j = 0; j < geom.fft; ++j) w32[(size_t)j] = (float)window[(size_t)j];
      d->d_window32 = upload(w32);
      d->d_tw_pass = upload(smb::fft1024_pass_twiddles());
      d->d_tw_post = upload(smb::unit_roots<float2>(512, 2048));   // W_2048^(l + 32 j) at [j][l]
      d->d_dft_images = upload(smb::dft32_split_images());
    }
    dev = std::move(d);
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
  int64_t frames_reaching(int64_t len) const {           // stft.ml:907-915
    return (len + geom.left_width() + geom.hop - 1) / geom.hop;
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
};

struct smb_mel_plan {
  int64_t n_mels = 0, fft = 0, bins = 0, sample_rate = 0;
  double f_min = 0, f_max = 0;
  int scale = 0, norm = 0;
  std::vector<double> weights;       // [n_mels][bins]
  std::vector<int> band_lo, band_hi;
  smb::PairSchedule sched_pair;
  smb::PieceSchedule sched_cc;   // CUDA-core kernel: kFastTile warps, 8 frames per lane
  smb::PieceSchedule sched_tc;   // tensor-core kernel: kTcTile warps, 4 frames per lane
  // 2048 / fft_size when the fused kernel can carry this filterbank (1 for fft
  // 2048, 2 for 1024, ...), else 0
  int fast_step = 0;
  // Everything the plan has on its device; null until the first device call.
  struct Device {
    int device = 0, sm_count = 0;
    StreamOwner stream;
    device_ptr<double> d_weights;
    device_ptr<int> d_band_lo, d_band_hi;
    struct PieceTables {
      device_ptr<float> d_vals;
      device_ptr<smb::MelPiece> d_pieces;
      device_ptr<unsigned char> d_pcnt;
    } cc, tc;
    device_ptr<float> d_pair_w;
    device_ptr<smb::PairMelItem> d_pair_items;
    // MFCC epilogue: DCT table of the last (n_mfcc, lifter) asked for, max scratch
    device_ptr<double> d_dct;
    device_ptr<unsigned long long> d_max;
  };
  std::unique_ptr<Device> dev;       // declared before the buffers used on its stream
  HostPipe pipe;                     // host-memory calls: sliced, copies under kernels
  int64_t dct_n_mfcc = -1;
  double dct_lifter = -1.0;
  const double* dct_table(int64_t n_mfcc, double lifter) {
    if (dev->d_dct && dct_n_mfcc == n_mfcc && dct_lifter == lifter) return dev->d_dct.get();
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
    dev->d_dct = upload(t);
    dct_n_mfcc = n_mfcc;
    dct_lifter = lifter;
    return dev->d_dct.get();
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
    if (step == 1) sched_pair = smb::pair_schedule(weights, band_lo, band_hi, n_mels, bins);
    // the CUDA-core kernel trades a few padded steps for conflict-free octets
    // (whole list as the window); the tensor-core kernel has no shared memory to
    // spare for longer weight tables and keeps the strict longest-first rounds
    sched_cc = smb::piece_schedule(weights, band_lo, band_hi, n_mels, bins, smb::kFastTile, smb::kFastPieceSteps,
                                   1 << 30);
    sched_tc = smb::piece_schedule(weights, band_lo, band_hi, n_mels, bins, smb::kTcTile, smb::kTcPieceSteps, 32);
    if (sched_cc.pieces.empty() || sched_tc.pieces.empty()) sched_cc = sched_tc = {};
    else fast_step = step;
  }
  void ensure_device() {
    if (dev) return same_device(dev->device);
    auto d = new_device<Device>();
    d->d_weights = upload(weights);
    d->d_band_lo = upload(band_lo);
    d->d_band_hi = upload(band_hi);
    d->cc = {upload(sched_cc.vals), upload(sched_cc.pieces), upload(sched_cc.pcnt)};
    d->tc = {upload(sched_tc.vals), upload(sched_tc.pieces), upload(sched_tc.pcnt)};
    d->d_pair_w = upload(sched_pair.w);
    d->d_pair_items = upload(sched_pair.items);
    d->d_max = device_alloc<unsigned long long>(sizeof(unsigned long long));
    dev = std::move(d);
  }
};

// The geometry fields of plan p's launch arguments (signal pointers and extents unset).
static smb::OlsArgs ols_args(const smb::OlsPlan& p) {
  smb::OlsArgs a{};
  a.L = (int)p.l; a.M = (int)p.m; a.K = (int)p.k;
  a.N = (int)p.n; a.B = (int)p.b; a.delta = (int)p.delta; a.W = (int)p.w;
  a.polyphase = p.polyphase ? 1 : 0;
  return a;
}

// The kernel that runs plan p (SMB_OLS_*): the warp-per-block kernel wherever it
// supports the geometry, the Stockham kernel otherwise.
static int ols_kernel_of(const smb::OlsPlan& p) {
  if (!p.ok) return SMB_OLS_NONE;
  if (smb::ols2048_supports(ols_args(p))) return SMB_OLS_2048;
  if (p.full_inverse || p.polyphase)
    throw smb::invalid_argument("soundml_b200: this overlap-save plan needs the N = 2048 kernel");
  return SMB_OLS_STOCKHAM;
}

// Device copies of one overlap-save plan's tables.
struct OlsDevice {
  device_ptr<float2> d_h;
  device_ptr<float2> d_tw;
  device_ptr<float2> d_tw_pass, d_tw_base;             // tables of the N = 2048 kernel
  void upload_from(const smb::OlsPlan& p) {
    if (!p.ok) return;
    if (p.n == 2048 && (p.l == 1 || p.polyphase)) {
      d_tw_pass = upload(smb::fft1024_pass_twiddles());
      d_tw_base = upload(smb::unit_roots<float2>(32, 2048));
    }
    std::vector<float2> h(p.spectrum_re.size());
    for (size_t i = 0; i < h.size(); ++i)
      h[i] = make_float2((float)p.spectrum_re[i], (float)p.spectrum_im[i]);
    d_h = upload(h);
    const int64_t tn = std::max(p.n, p.w);
    d_tw = upload(smb::unit_roots<float2>(tn / 2, tn));
  }
  void run(const smb::OlsPlan& plan, const float* x, int64_t batch, int64_t n, int64_t n_out, float* out,
           int sm_count, cudaStream_t st) const {
    smb::OlsArgs a = ols_args(plan);
    a.x = x;
    a.out = out;
    a.n = n;
    a.n_out = n_out;
    a.blocks = plan.blocks_for(n_out);
    a.H = d_h.get();
    a.tw = d_tw.get();
    if (ols_kernel_of(plan) == SMB_OLS_2048)
      CK(smb::launch_ols2048(a, d_tw_pass.get(), d_tw_base.get(), batch, sm_count, st));
    else
      CK(smb::launch_ols(a, batch, st));
  }
};

// Device copies of one column group's tcgen05 resampler images (smb::GemmLayout).
struct GemmImages {
  device_ptr<float> d_images;
  device_ptr<int4> d_meta, d_slices;   // chunk meta; slice meta (row form only)
};

struct smb_resample_plan {
  smb::ResamplePlan plan;
  // Host tables per stage, built by the first layout() or device call (the SMB_ROWS_*
  // switches are read then); once uploaded, the host keeps the launch arguments only.
  struct StageTables { smb::OlsPlan ols; smb::GemmLayout gemm; };
  std::vector<StageTables> tables;
  // Everything the plan has on its device; null until the first device call.
  struct Device {
    int device = 0, sm_count = 0;
    StreamOwner stream;
    struct Stage {
      device_ptr<float> d_bank;                // [l][2k+1] float32
      device_ptr<double> d_bank64;             // the same bank uncast, for float64 audio
      OlsDevice ols;
      std::vector<GemmImages> rows, windows;   // per column group of the stage's GemmLayout
    };
    std::vector<Stage> stages;
  };
  std::unique_ptr<Device> dev;       // declared before the buffers used on its stream
  int executor = SMB_EXEC_PLANNED;   // SMB_EXEC_DIRECT forces the dot-product kernel everywhere
  DeviceBuffer mid;
  HostPipe pipe;                     // host-memory calls: sliced, copies under kernels
  void build_tables() {
    for (size_t i = tables.size(); i < plan.stages.size(); ++i)
      tables.push_back({smb::ols_plan_for_stage(plan.stages[i]), smb::gemm_layout(plan.stages[i])});
  }
  void ensure_device() {
    if (dev) return same_device(dev->device);
    build_tables();
    auto d = new_device<Device>();
    for (size_t i = 0; i < plan.stages.size(); ++i) {
      const std::vector<double>& bank = plan.stages[i].bank;
      Device::Stage& ds = d->stages.emplace_back();
      ds.d_bank = upload(std::vector<float>(bank.begin(), bank.end()));   // cast at prepare
      ds.d_bank64 = upload(bank);
      ds.ols.upload_from(tables[i].ols);
      for (const auto& g : tables[i].gemm.rows)
        ds.rows.push_back({upload(g.images), upload(g.chunk_meta), upload(g.slice_meta)});
      for (const auto& g : tables[i].gemm.windows) ds.windows.push_back({upload(g.images), upload(g.chunk_meta)});
    }
    for (StageTables& t : tables) {
      for (auto& g : t.gemm.rows) g = {g.a};
      for (auto& g : t.gemm.windows) g = {g.a};
    }
    dev = std::move(d);
  }
  // The kernel run_stage picks for stage i (SMB_FORM_*); the host tables must be built.
  int form(size_t i) const {
    if (executor == SMB_EXEC_DIRECT) return SMB_FORM_DIRECT;
    if (tables[i].ols.ok) return SMB_FORM_OLS;
    // (SMB_GEMM_WINDOWS=1: the overlapping-window form, for A/B measurement)
    if (!tables[i].gemm.rows.empty() && !getenv("SMB_GEMM_WINDOWS")) return SMB_FORM_ROW;
    if (!tables[i].gemm.windows.empty()) return SMB_FORM_WINDOW;
    return SMB_FORM_DIRECT;
  }
  // One stage over device buffers: overlap-save where the planner tagged it and
  // the GPU plan exists, the direct polyphase kernel otherwise -- the same
  // designed filter either way (resample.ml:495-497).
  void run_stage(size_t i, const float* x, int64_t batch, int64_t n, int64_t n_out, float* out,
                 cudaStream_t st) {
    const smb::ResampleStage& s = plan.stages[i];
    const smb::GemmLayout& gl = tables[i].gemm;
    const Device::Stage& ds = dev->stages[i];
    // the launch arguments of a tcgen05 column group over x -> out
    auto bind = [&](auto a, const GemmImages& im) {
      a.x = x;
      a.out = out;
      a.n = n;
      a.n_out = n_out;
      a.b_images = im.d_images.get();
      a.chunk_meta = im.d_meta.get();
      return a;
    };
    const int f = form(i);
    if (f == SMB_FORM_OLS) {
      ds.ols.run(tables[i].ols, x, batch, n, n_out, out, dev->sm_count, st);
    } else if (f == SMB_FORM_ROW) {
      for (size_t g = 0; g < gl.rows.size(); ++g) {
        smb::GemmRowsArgs a = bind(gl.rows[g].a, ds.rows[g]);
        a.slice_meta = ds.rows[g].d_slices.get();
        CK(smb::launch_resample_rows(a, batch, dev->sm_count, st));
      }
    } else if (f == SMB_FORM_WINDOW) {
      for (size_t g = 0; g < gl.windows.size(); ++g)
        CK(smb::launch_resample_gemm(bind(gl.windows[g].a, ds.windows[g]), batch, st));
    } else
      CK(smb::launch_polyphase_direct(x, batch, n, ds.d_bank.get(), (int)s.l, (int)s.m, (int)s.k, n_out, out, st));
  }
};

struct smb_fir_plan {
  std::vector<double> h;
  int64_t k = 0;
  // Everything the plan has on its device; null until the first device call.
  struct Device {
    int device = 0, sm_count = 0;
    StreamOwner stream;
    device_ptr<float> d_bank;
    smb::OlsPlan ols_plan;
    OlsDevice ols;
  };
  std::unique_ptr<Device> dev;       // declared before the buffers used on its stream
  HostPipe pipe;                     // host-memory calls: sliced, copies under kernels
  void ensure_device() {
    if (dev) return same_device(dev->device);
    auto d = new_device<Device>();
    d->d_bank = upload(std::vector<float>(h.rbegin(), h.rend()));   // row reversed
    d->ols_plan = smb::ols_plan_for_fir(h);
    d->ols.upload_from(d->ols_plan);
    dev = std::move(d);
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
  return guarded([&] { plan->ensure_device(); plan->dev->stream.set(s); });
}
int smb_stft_plan_set_path(smb_stft_plan* plan, int path) {
  return guarded([&] {
    if (path < SMB_PATH_AUTO || path > SMB_PATH_PAIR)
      throw smb::invalid_argument("set_path: unknown path");
    plan->path = path;
  });
}
int smb_stft_plan_sync(smb_stft_plan* plan) {
  return guarded([&] { if (plan->dev) CK(cudaStreamSynchronize(plan->dev->stream.use)); });
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

void check_signal(const char* op, int64_t batch, int64_t n) {
  if (n < 0)
    throw smb::invalid_argument(smb::format(
        "%s: cannot analyse a signal of length %lld (length must be non-negative)", op,
        (long long)n));
  if (batch < 0) throw smb::invalid_argument(smb::format("%s: negative batch", op));
}

void require_nola(const char* op, const smb_stft_plan* p) {     // stft.ml:744-753
  if (!p->nola())
    throw smb::invalid_argument(smb::format(
        "%s: cannot invert a %lld-point window advanced by %lld samples inside a "
        "%lld-point frame (the overlap-added squared window must stay above 1e-10 of its "
        "largest value at every position)",
        op, (long long)p->geom.win_length, (long long)p->geom.hop, (long long)p->geom.fft));
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
  const smb::PieceSchedule none{};
  const smb::PieceSchedule& tc = mel ? mel->sched_tc : none;
  const smb::PieceSchedule& cc = mel ? mel->sched_cc : none;
  const int n_mels = mel ? (int)mel->n_mels : 0;
  const bool ok_tc = base && smb::stft2048tc_supports(gk, out_kind, n_mels, (int)tc.vals.size(), tc.rounds, tc.mpad);
  const bool ok_cc = base && smb::stft2048_supports(gk, out_kind, n_mels, (int)cc.vals.size(), cc.rounds, cc.mpad);
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
  return ok_cc ? SMB_PATH_FAST : (ok_tc ? SMB_PATH_TENSOR : 0);
}

// The launch arguments of a fused fft-2048 kernel without a mel schedule: Stft2048Args for the
// CUDA-core and tensor-core kernels, Stft2048PairArgs for the frame-pair kernel.
template <typename Args = smb::Stft2048Args>
Args fused_args(const smb_stft_plan* stft, const void* din, void* dout, int64_t nb, const smb::FrameGeom& g,
                double power) {
  Args a{};
  a.x = (const float*)din;
  a.out = (float*)dout;
  a.batch = nb;
  a.g = g;
  a.g.fft = 2048;
  a.window = stft->dev->d_window32.get();
  a.tw_pass = stft->dev->d_tw_pass.get();
  a.tw_post = stft->dev->d_tw_post.get();
  a.power = (float)power;
  if constexpr (std::is_same_v<Args, smb::Stft2048Args>) {
    a.bin_step = stft->fast_step();
    a.dft_images = stft->dev->d_dft_images.get();
  }
  return a;
}

smb::Stft2048PairArgs pair_args(const smb_stft_plan* stft, const smb_mel_plan* mel, const void* din,
                                void* dout, int64_t nb, const smb::FrameGeom& g, double power) {
  auto a = fused_args<smb::Stft2048PairArgs>(stft, din, dout, nb, g, power);
  if (mel) {
    a.n_mels = (int)mel->n_mels;
    a.mel_w = mel->dev->d_pair_w.get();
    a.mel_w_floats = (int)mel->sched_pair.w.size();
    a.mel_items = mel->dev->d_pair_items.get();
    a.mel_rounds = mel->sched_pair.rounds;
  }
  return a;
}

// x (device) -> spectrum (device).  kind: complex or |X|^power.
void run_spectrum(smb_stft_plan* p, const void* dx, int64_t batch, const smb::FrameGeom& g,
                  int dtype, SpecKind kind, double power, void* dout) {
  const smb_stft_plan::Device& d = *p->dev;
  cudaStream_t st = d.stream.use;
  const int fast_kind = kind == kSpecComplex ? smb::kFastComplex : smb::kFastPower;
  if (const int which = want_fast(p, dtype, g, fast_kind, nullptr)) {
    const smb::Stft2048Args a = fused_args(p, dx, dout, batch, g, power);
    if (which == SMB_PATH_TENSOR) CK(smb::launch_stft2048tc(a, fast_kind, d.sm_count, st));
    else CK(smb::launch_stft2048(a, fast_kind, d.sm_count, st));
  } else {
    CK(smb::launch_stft_generic(dx, dtype, batch, g, d.d_window64.get(), d.d_twiddle64.get(),
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
  dispatch(mem, p->pipe, p->dev->stream.use, x, out, batch, (size_t)n * esz, out_elems / (size_t)batch * esz,
           [&](const void* din, void* dout, int64_t nb) {
             run_spectrum(p, din, nb, g, dtype, kind, power, dout);
           });
}

void run_mel_apply(smb_mel_plan* m, const void* ds, int64_t batch, int64_t frames, int dtype,
                   void* dout, cudaStream_t st) {
  CK(smb::launch_mel_apply(ds, dtype, batch, (int)m->bins, frames, (int)m->n_mels, m->dev->d_weights.get(),
                           m->dev->d_band_lo.get(), m->dev->d_band_hi.get(), dout, st));
}

// The synthesis arguments of Stft.invert for `nb` items z (device) -> out (device) on the
// plan's stream.  Only the frames the output can reach are inverted; when none does, out
// is zero-filled here and the count is 0: nothing is left to launch.
smb::IstftArgs istft_args(smb_stft_plan* p, const void* dz, void* dout, int64_t nb, int64_t frames,
                          bool has_length, int64_t out_len, int in_dtype, int out_dtype) {
  smb_stft_plan::Device& d = *p->dev;
  smb::IstftArgs a{};
  a.count = has_length ? std::min(frames, p->frames_reaching(out_len)) : frames;
  if (a.count == 0) {
    CK(cudaMemsetAsync(dout, 0, (size_t)nb * (size_t)out_len * dtype_size(out_dtype), d.stream.use));
    return a;
  }
  if (!d.d_folded) d.d_folded = upload(p->folded_square_window());
  a.z = dz;
  a.out = dout;
  a.frames = frames;
  a.out_len = out_len;
  a.fft = (int)p->geom.fft;
  a.hop = (int)p->geom.hop;
  a.left = (int)p->geom.left_width();
  a.window = d.d_window64.get();
  a.twiddle = d.d_twiddle64.get();
  a.folded = d.d_folded.get();
  a.in_f64 = in_dtype == SMB_F64;
  a.out_f64 = out_dtype == SMB_F64;
  return a;
}

// z (device) -> out (device): Stft.invert of `nb` items on the plan's stream (the
// synthesis kernels of smb_stft_invert; time_stretch's last stage)
void run_invert(smb_stft_plan* p, const void* dz, void* dout, int64_t nb, int64_t frames,
                bool has_length, int64_t out_len, int in_dtype, int out_dtype) {
  smb_stft_plan::Device& d = *p->dev;
  cudaStream_t st = d.stream.use;
  const smb::IstftArgs a = istft_args(p, dz, dout, nb, frames, has_length, out_len, in_dtype, out_dtype);
  if (a.count == 0) return;
  const bool fast = p->path != SMB_PATH_GENERIC && smb::istft2048_supports(a);
  if (!fast && p->path == SMB_PATH_FAST)
    throw smb::invalid_argument(
        "soundml_b200: the fft-2048 synthesis kernel does not cover this geometry");
  if (fast) {
    if (!d.d_window_inv) {
      // 1 / fft of the inverse folded in; frames shorter than 2048 leave a zero tail
      std::vector<float> w(2048, 0.0f);
      for (size_t j = 0; j < (size_t)p->geom.fft; ++j)
        w[j] = (float)(p->window[j] / double(p->geom.fft));
      d.d_window_inv = upload(w);
    }
    CK(smb::launch_istft2048(a, d.d_window_inv.get(), d.d_tw_pass.get(), d.d_tw_post.get(), nb,
                             d.sm_count, st));
    return;
  }
  CK(smb::launch_istft(a, nb, st));
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
    require_nola("invert", p);
    const size_t isz = 2 * dtype_size(in_dtype), osz = dtype_size(out_dtype);
    const int64_t out_len = has_length ? length : p->output_length(frames);
    if (batch == 0 || out_len == 0) return;
    p->ensure_device();
    if (mem == SMB_MEM_HOST && frames == 0) {
      std::memset(out, 0, (size_t)batch * (size_t)out_len * osz);
      return;
    }
    dispatch(mem, p->pipe, p->dev->stream.use, z, out, batch, (size_t)p->geom.bins() * (size_t)frames * isz,
             (size_t)out_len * osz, [&](const void* dz, void* dout, int64_t nb) {
               run_invert(p, dz, dout, nb, frames, has_length != 0, out_len, in_dtype, out_dtype);
             });
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
    require_nola("griffin_lim", p);
    if (n_iter < 1)
      throw smb::invalid_argument(smb::format(
          "griffin_lim: cannot run %lld iterations (n_iter must be at least 1)",
          (long long)n_iter));
    if (momentum < 0.0)
      throw smb::invalid_argument(smb::format(
          "griffin_lim: cannot use a momentum of %g (momentum must be non-negative)", momentum));
    const size_t esz = dtype_size(dtype);
    const int64_t bins = p->geom.bins();
    const int64_t natural = p->output_length(frames);
    const int64_t out_len = has_length ? length : natural;
    if (batch == 0 || out_len == 0) return;
    check_mem(mem);
    if (frames == 0) {
      if (mem == SMB_MEM_HOST) std::memset(out, 0, (size_t)batch * (size_t)out_len * esz);
      else { p->ensure_device(); CK(cudaMemsetAsync(out, 0, (size_t)batch * (size_t)out_len * esz, p->dev->stream.use)); }
      return;
    }
    p->ensure_device();
    smb_stft_plan::Device& d = *p->dev;
    cudaStream_t st = d.stream.use;
    const size_t cells = (size_t)batch * (size_t)bins * (size_t)frames;
    // the whole problem stays resident across the iterations; freed when the call returns or throws
    device_ptr<void> d_s, d_phase, d_out, d_a, d_b, d_y;
    const void* mags = s;
    const void* phase = init_phase;
    void* dout = out;
    if (mem == SMB_MEM_HOST) {
      d_s = device_alloc(cells * esz);
      CK(cudaMemcpyAsync(d_s.get(), s, cells * esz, cudaMemcpyHostToDevice, st));
      mags = d_s.get();
      if (init_phase) {
        d_phase = device_alloc(cells * esz);
        CK(cudaMemcpyAsync(d_phase.get(), init_phase, cells * esz, cudaMemcpyHostToDevice, st));
        phase = d_phase.get();
      }
      d_out = device_alloc((size_t)batch * (size_t)out_len * esz);
      dout = d_out.get();
    }
    const device_ptr<double2> d_spec = device_alloc<double2>(cells * sizeof(double2));
    double2* spec = d_spec.get();
    auto synth = [&](int64_t len, bool named, int out_dtype, void* dst) {
      const smb::IstftArgs a = istft_args(p, spec, dst, batch, frames, named, len, SMB_F64, out_dtype);
      if (a.count) CK(smb::launch_istft(a, batch, st));
    };
    CK(smb::launch_gl_project(mags, phase, dtype == SMB_F64, nullptr, nullptr, 0.0, 1,
                              (long long)cells, spec, st));
    // the loop runs at the natural length, the one geometry that re-analyses to
    // exactly `frames` frames (stft.ml:1000-1008)
    if (natural > 0) {
      d_a = device_alloc(cells * sizeof(double2));
      d_b = device_alloc(cells * sizeof(double2));
      d_y = device_alloc((size_t)batch * (size_t)natural * sizeof(double));
      double2* rebuilt = (double2*)d_a.get();
      double2* previous = (double2*)d_b.get();
      const double beta = momentum / (1.0 + momentum);
      smb::FrameGeom g = p->frame_geom(natural);
      if (g.frames != frames)
        throw smb::invalid_argument("griffin_lim: the natural length does not re-analyse to the "
                                    "given frame count");
      for (int64_t k = 0; k < n_iter; ++k) {
        synth(natural, false, SMB_F64, d_y.get());
        CK(smb::launch_stft_generic(d_y.get(), SMB_F64, batch, g, d.d_window64.get(), d.d_twiddle64.get(),
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

}  // extern "C"

// ---- effects: phase vocoder, time_stretch (librosa 0.11 effects; DESIGN.md 4.8) and hpss (4.9) ----

namespace {

void check_rate(const char* op, double rate) {
  if (!(rate > 0.0) || !std::isfinite(rate))
    throw smb::invalid_argument(smb::format(
        "%s: cannot stretch by a rate of %g (the rate must be positive and finite)", op, rate));
}

// ceil(frames / rate) in double: the length of np.arange(0, frames, rate)
int64_t vocoder_frames(const char* op, int64_t frames, double rate) {
  check_rate(op, rate);
  if (frames < 0)
    throw smb::invalid_argument(smb::format(
        "%s: cannot stretch %lld frames (frames must be non-negative)", op, (long long)frames));
  const double q = std::ceil((double)frames / rate);
  if (!(q <= 9007199254740992.0))
    throw smb::invalid_argument(smb::format(
        "%s: cannot stretch %lld frames by a rate of %g (the result would hold more than 2^53 "
        "frames)", op, (long long)frames, rate));
  return (int64_t)q;
}

// round(n / rate), half to even as Python's round (the current rounding mode is the
// default round-to-nearest-even)
int64_t stretch_length(int64_t n, double rate) {
  check_rate("time_stretch", rate);
  if (n < 0)
    throw smb::invalid_argument(smb::format(
        "time_stretch: cannot stretch a signal of length %lld (length must be non-negative)",
        (long long)n));
  const double q = std::nearbyint((double)n / rate);
  if (!(q <= 9007199254740992.0))
    throw smb::invalid_argument(smb::format(
        "time_stretch: cannot stretch %lld samples by a rate of %g (the result would hold more "
        "than 2^53 samples)", (long long)n, rate));
  return (int64_t)q;
}

void run_vocoder(smb_stft_plan* p, const void* dz, void* dout, int64_t nb, int64_t frames,
                 int64_t out_frames, int dtype, double rate) {
  smb::PhaseVocoderArgs a{};
  a.z = dz;
  a.out = dout;
  a.rows = nb * p->geom.bins();
  a.frames = frames;
  a.out_frames = out_frames;
  a.rate = rate;
  a.f64 = dtype == SMB_F64;
  CK(smb::launch_phase_vocoder(a, p->dev->stream.use));
}

}  // namespace

extern "C" {

int64_t smb_time_stretch_frames(const smb_stft_plan* plan, int64_t frames, double rate) {
  (void)plan;
  int64_t r = -1;
  guarded([&] { r = vocoder_frames("phase_vocoder", frames, rate); });
  return r;
}

int64_t smb_time_stretch_length(int64_t n, double rate) {
  int64_t r = -1;
  guarded([&] { r = stretch_length(n, rate); });
  return r;
}

int smb_phase_vocoder(smb_stft_plan* plan, const void* z, int64_t batch, int64_t frames,
                      int dtype, double rate, void* out, int mem) {
  return guarded([&] {
    smb_stft_plan* p = plan;
    const int64_t out_frames = vocoder_frames("phase_vocoder", frames, rate);
    if (batch < 0)
      throw smb::invalid_argument("phase_vocoder: batch must be non-negative");
    const size_t csz = 2 * dtype_size(dtype);
    check_mem(mem);
    if (batch == 0 || out_frames == 0) return;
    p->ensure_device();
    const size_t bins = (size_t)p->geom.bins();
    dispatch(mem, p->pipe, p->dev->stream.use, z, out, batch, bins * (size_t)frames * csz,
             bins * (size_t)out_frames * csz, [&](const void* dz, void* dout, int64_t nb) {
               run_vocoder(p, dz, dout, nb, frames, out_frames, dtype, rate);
             });
  });
}

int smb_time_stretch(smb_stft_plan* plan, const void* x, int64_t batch, int64_t n, int dtype,
                     double rate, void* out, int mem) {
  return guarded([&] {
    smb_stft_plan* p = plan;
    check_rate("time_stretch", rate);
    check_signal("time_stretch", batch, n);
    require_nola("invert", p);                          // Stft.invert's precondition
    const size_t esz = dtype_size(dtype);
    check_mem(mem);
    const int64_t out_len = stretch_length(n, rate);
    const smb::FrameGeom g = p->frame_geom(n);
    const int64_t out_frames = vocoder_frames("time_stretch", g.frames, rate);
    if (batch == 0 || out_len == 0) return;
    p->ensure_device();
    cudaStream_t st = p->dev->stream.use;
    const size_t bins = (size_t)p->geom.bins();
    // transform -> vocoder -> invert on the plan's stream; the two spectra stay on the
    // device in the plan's scratch (reused by the next call on the same stream)
    auto run = [&](const void* dx, void* dout, int64_t nb) {
      if (out_frames == 0) {                            // no frame: invert of nothing is zeros
        CK(cudaMemsetAsync(dout, 0, (size_t)nb * (size_t)out_len * esz, st));
        return;
      }
      void* spec = p->effect_in.ensure((size_t)nb * bins * (size_t)g.frames * 2 * esz);
      void* voc = p->effect_out.ensure((size_t)nb * bins * (size_t)out_frames * 2 * esz);
      run_spectrum(p, dx, nb, g, dtype, kSpecComplex, 1.0, spec);
      run_vocoder(p, spec, voc, nb, g.frames, out_frames, dtype, rate);
      run_invert(p, voc, dout, nb, out_frames, true, out_len, dtype, dtype);
    };
    dispatch(mem, p->pipe, st, x, out, batch, (size_t)n * esz, (size_t)out_len * esz, run);
  });
}

}  // extern "C"

namespace {

// hpss's parameters in the documented order (include/soundml_b200.h); librosa lets a NaN
// power or margin through, which would only make every mask NaN
void check_hpss(int64_t win_harm, int64_t win_perc, double power, double margin_harm,
                double margin_perc) {
  for (int64_t w : {win_harm, win_perc})
    if (w < 1)
      throw smb::invalid_argument(smb::format(
          "hpss: cannot take a median over %lld values (kernel sizes must be at least 1)", (long long)w));
  for (double m : {margin_harm, margin_perc})
    if (!(m >= 1.0) || !std::isfinite(m))
      throw smb::invalid_argument(smb::format(
          "hpss: cannot use a margin of %g (margins must be finite and at least 1)", m));
  if (!(power > 0.0))
    throw smb::invalid_argument(smb::format(
        "hpss: cannot raise the masks to a power of %g (the power must be positive; +inf gives "
        "hard masks)", power));
}

// outputs per item: 2 for SMB_HPSS_BOTH and SMB_HPSS_MASKS, else 1
int hpss_parts(int what, bool masks_allowed) {
  if (what == SMB_HPSS_HARMONIC || what == SMB_HPSS_PERCUSSIVE) return 1;
  if (what == SMB_HPSS_BOTH || (masks_allowed && what == SMB_HPSS_MASKS)) return 2;
  throw smb::invalid_argument(smb::format(
      "hpss: cannot return output kind %d (what must be SMB_HPSS_BOTH, SMB_HPSS_HARMONIC, "
      "SMB_HPSS_PERCUSSIVE%s)", what, masks_allowed ? " or SMB_HPSS_MASKS" : ""));
}

smb::HpssArgs hpss_args(const void* s, void* out, int64_t batch, int64_t bins, int64_t frames, int dtype,
                        bool complex_in, int64_t win_harm, int64_t win_perc, double power,
                        double margin_harm, double margin_perc, int what) {
  smb::HpssArgs a{};
  a.s = s;
  a.out = out;
  a.batch = batch;
  a.bins = bins;
  a.frames = frames;
  a.win_harm = win_harm;
  a.win_perc = win_perc;
  a.power = power;
  a.margin_harm = margin_harm;
  a.margin_perc = margin_perc;
  a.what = what;
  a.f64 = dtype == SMB_F64;
  a.complex_in = complex_in;
  return a;
}

}  // namespace

extern "C" {

int smb_hpss(const void* s, int64_t batch, int64_t bins, int64_t frames, int dtype, int complex_in,
             int64_t win_harm, int64_t win_perc, double power, double margin_harm,
             double margin_perc, int what, void* out, int mem, void* cuda_stream) {
  return guarded([&] {
    check_hpss(win_harm, win_perc, power, margin_harm, margin_perc);
    if (batch < 0 || bins < 0 || frames < 0)
      throw smb::invalid_argument(smb::format(
          "hpss: cannot separate a [%lld, %lld, %lld] spectrogram (extents must be non-negative)",
          (long long)batch, (long long)bins, (long long)frames));
    const size_t esz = dtype_size(dtype);
    check_mem(mem);
    const int parts = hpss_parts(what, true);
    const size_t cells = (size_t)batch * (size_t)bins * (size_t)frames;
    if (cells == 0) return;
    require_device();
    // no plan, hence no plan stream: SMB_STREAM_OWN means the default stream
    cudaStream_t st = cuda_stream == SMB_STREAM_OWN ? nullptr : (cudaStream_t)cuda_stream;
    const size_t in_bytes = cells * esz * (complex_in ? 2 : 1);
    const size_t out_bytes = cells * (size_t)parts * esz * (complex_in && what != SMB_HPSS_MASKS ? 2 : 1);
    on_stream(mem, st, s, in_bytes, out, out_bytes, [&](const void* src, void* dst) {
      CK(smb::launch_hpss(hpss_args(src, dst, batch, bins, frames, dtype, complex_in != 0, win_harm, win_perc,
                                    power, margin_harm, margin_perc, what), st));
    });
  });
}

int smb_hpss_audio(smb_stft_plan* plan, const void* x, int64_t batch, int64_t n, int dtype,
                   int64_t win_harm, int64_t win_perc, double power, double margin_harm,
                   double margin_perc, int what, void* out, int mem) {
  return guarded([&] {
    smb_stft_plan* p = plan;
    check_hpss(win_harm, win_perc, power, margin_harm, margin_perc);
    check_signal("hpss", batch, n);
    require_nola("invert", p);                          // Stft.invert's precondition
    const size_t esz = dtype_size(dtype);
    check_mem(mem);
    const int parts = hpss_parts(what, false);
    if (batch == 0 || n == 0) return;
    p->ensure_device();
    cudaStream_t st = p->dev->stream.use;
    const smb::FrameGeom g = p->frame_geom(n);
    const size_t bins = (size_t)p->geom.bins();
    // transform -> hpss -> one invert over the nb * parts separated spectra, whose
    // [nb, parts, bins, frames] layout makes the output [nb, parts, n]
    auto run = [&](const void* dx, void* dout, int64_t nb) {
      if (g.frames == 0) {                              // no frame: invert of nothing is zeros
        CK(cudaMemsetAsync(dout, 0, (size_t)nb * parts * (size_t)n * esz, st));
        return;
      }
      const size_t spectrum = bins * (size_t)g.frames * 2 * esz;
      void* spec = p->effect_in.ensure((size_t)nb * spectrum);
      void* sep = p->effect_out.ensure((size_t)nb * parts * spectrum);
      run_spectrum(p, dx, nb, g, dtype, kSpecComplex, 1.0, spec);
      CK(smb::launch_hpss(hpss_args(spec, sep, nb, (int64_t)bins, g.frames, dtype, true, win_harm, win_perc,
                                    power, margin_harm, margin_perc, what), st));
      run_invert(p, sep, dout, nb * parts, g.frames, true, n, dtype, dtype);
    };
    dispatch(mem, p->pipe, st, x, out, batch, (size_t)n * esz, (size_t)parts * (size_t)n * esz, run);
  });
}

}  // extern "C"

// ---- spectral descriptors (librosa 0.11 feature.spectral_*; DESIGN.md 4.10) ----

namespace {

constexpr int kSpectralAll = SMB_SPECTRAL_CENTROID | SMB_SPECTRAL_BANDWIDTH | SMB_SPECTRAL_ROLLOFF |
                             SMB_SPECTRAL_FLATNESS;

// the descriptors' parameters in the documented order (include/soundml_b200.h); returns the
// rows per item
int check_spectral(int what, double sample_rate, double p, double roll_percent, double amin,
                   double power) {
  if (what == 0 || (what & ~kSpectralAll))
    throw smb::invalid_argument(smb::format(
        "spectral: cannot compute descriptor set %d (what must be a nonzero combination of "
        "SMB_SPECTRAL_CENTROID, SMB_SPECTRAL_BANDWIDTH, SMB_SPECTRAL_ROLLOFF and "
        "SMB_SPECTRAL_FLATNESS)", what));
  if (!(sample_rate > 0.0) || !std::isfinite(sample_rate))
    throw smb::invalid_argument(smb::format(
        "spectral: cannot use a sample rate of %g (it must be positive and finite)", sample_rate));
  if (!(p > 0.0) || !std::isfinite(p))
    throw smb::invalid_argument(smb::format(
        "spectral: cannot take the bandwidth at p = %g (p must be positive and finite)", p));
  if (!(roll_percent > 0.0 && roll_percent < 1.0))
    throw smb::invalid_argument(smb::format(
        "spectral: cannot roll off at %g of the energy (roll_percent must lie in (0, 1))", roll_percent));
  if (!(amin > 0.0))
    throw smb::invalid_argument(smb::format(
        "spectral: cannot floor the spectrum at amin = %g (amin must be positive)", amin));
  if (!(power > 0.0))
    throw smb::invalid_argument(smb::format(
        "spectral: cannot raise the spectrum to a power of %g (the power must be positive)", power));
  return __builtin_popcount((unsigned)what);
}

smb::SpectralArgs spectral_args(const void* s, void* out, int64_t batch, int64_t bins, int64_t frames,
                                int dtype, int64_t n_fft, double sample_rate, int what, double p,
                                int norm, double roll_percent, double amin, double power) {
  smb::SpectralArgs a{};
  a.s = s;
  a.out = out;
  a.batch = batch;
  a.bins = bins;
  a.frames = frames;
  a.bin_hz = 1.0 / ((double)n_fft * (1.0 / sample_rate));   // numpy rfftfreq's 1 / (n d)
  a.what = what;
  a.p = p;
  a.norm = norm != 0;
  a.roll_percent = roll_percent;
  a.amin = amin;
  a.power = power;
  a.f64 = dtype == SMB_F64;
  return a;
}

}  // namespace

extern "C" {

int smb_spectral(const void* s, int64_t batch, int64_t bins, int64_t frames, int dtype,
                 int64_t n_fft, double sample_rate, int what, double p, int norm,
                 double roll_percent, double amin, double power, void* out, int mem,
                 void* cuda_stream) {
  return guarded([&] {
    const int rows = check_spectral(what, sample_rate, p, roll_percent, amin, power);
    if (batch < 0 || bins < 0 || frames < 0)
      throw smb::invalid_argument(smb::format(
          "spectral: cannot describe a [%lld, %lld, %lld] spectrogram (extents must be non-negative)",
          (long long)batch, (long long)bins, (long long)frames));
    if (n_fft == SMB_DEFAULT) n_fft = 2 * (bins - 1);
    if (n_fft <= 0 || n_fft / 2 + 1 != bins)
      throw smb::invalid_argument(smb::format(
          "spectral: cannot read %lld bins as the spectrum of a %lld-point transform (n_fft must "
          "be positive, with n_fft / 2 + 1 bins)", (long long)bins, (long long)n_fft));
    const size_t esz = dtype_size(dtype);
    check_mem(mem);
    if (batch == 0 || frames == 0) return;
    require_device();
    // no plan, hence no plan stream: SMB_STREAM_OWN means the default stream
    cudaStream_t st = cuda_stream == SMB_STREAM_OWN ? nullptr : (cudaStream_t)cuda_stream;
    const size_t in_bytes = (size_t)batch * (size_t)bins * (size_t)frames * esz;
    const size_t out_bytes = (size_t)batch * (size_t)rows * (size_t)frames * esz;
    on_stream(mem, st, s, in_bytes, out, out_bytes, [&](const void* src, void* dst) {
      CK(smb::launch_spectral(spectral_args(src, dst, batch, bins, frames, dtype, n_fft, sample_rate, what,
                                            p, norm, roll_percent, amin, power), st));
    });
  });
}

int smb_spectral_audio(smb_stft_plan* plan, const void* x, int64_t batch, int64_t n, int dtype,
                       double sample_rate, int what, double p, int norm, double roll_percent,
                       double amin, double power, void* out, int mem) {
  return guarded([&] {
    smb_stft_plan* pl = plan;
    const int rows = check_spectral(what, sample_rate, p, roll_percent, amin, power);
    check_signal("spectral", batch, n);
    const size_t esz = dtype_size(dtype);
    check_mem(mem);
    const smb::FrameGeom g = pl->frame_geom(n);
    if (batch == 0 || g.frames == 0) return;          // no frame: nothing to write
    pl->ensure_device();
    cudaStream_t st = pl->dev->stream.use;
    const int64_t bins = pl->geom.bins();
    // |transform| into the plan's scratch, then the descriptors
    auto run = [&](const void* dx, void* dout, int64_t nb) {
      void* mag = pl->effect_in.ensure((size_t)nb * (size_t)bins * (size_t)g.frames * esz);
      run_spectrum(pl, dx, nb, g, dtype, kSpecPower, 1.0, mag);
      CK(smb::launch_spectral(spectral_args(mag, dout, nb, bins, g.frames, dtype, pl->geom.fft, sample_rate,
                                            what, p, norm, roll_percent, amin, power), st));
    };
    dispatch(mem, pl->pipe, st, x, out, batch, (size_t)n * esz, (size_t)rows * (size_t)g.frames * esz, run);
  });
}

}  // extern "C"

extern "C" {

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
  return guarded([&] { plan->ensure_device(); plan->dev->stream.set(s); });
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
    cudaStream_t st = plan->dev->stream.use;
    dispatch(mem, plan->pipe, st, s, out, batch, (size_t)plan->bins * frames * esz,
             (size_t)plan->n_mels * frames * esz, [&](const void* din, void* dout, int64_t nb) {
               run_mel_apply(plan, din, nb, frames, dtype, dout, st);
             });
  });
}

}  // extern "C"

// soundml.ml:12-20, 50-70
static void require_same_fft(const char* op, const smb_stft_plan* stft, const smb_mel_plan* mel) {
  if (stft->geom.fft != mel->fft)
    throw smb::invalid_argument(smb::format(
        "%s: cannot project a %lld-point STFT through a filterbank built for an FFT of size "
        "%lld (the two configurations must agree on fft_size)",
        op, (long long)stft->geom.fft, (long long)mel->fft));
}

// Soundml.mel_spectrogram.  max_slot (device, zeroed by the caller, may be null): where
// the kernel leaves the maximum of what it writes; the return value says whether it did
// (only the frame-pair kernel does; slices of a host batch accumulate into the one slot).
static bool mel_spectrogram_impl(smb_stft_plan* stft, smb_mel_plan* mel, const void* x, int64_t batch,
                                 int64_t n, int dtype, double power, void* out, int mem,
                                 unsigned long long* max_slot) {
  bool max_known = false;
  {
    require_same_fft("mel_spectrogram", stft, mel);
    check_signal("power_spectrum", batch, n);
    const size_t esz = dtype_size(dtype);
    const smb::FrameGeom g = stft->frame_geom(n);
    if (batch == 0 || g.frames == 0) return false;
    stft->ensure_device();
    mel->ensure_device();
    const smb_stft_plan::Device& sd = *stft->dev;
    cudaStream_t st = sd.stream.use;
    const int fast = want_fast(stft, dtype, g, smb::kFastMel, mel);
    max_known = fast == SMB_PATH_PAIR && max_slot != nullptr;
    auto run = [&](const void* din, void* dout, int64_t nb) {
      if (fast == SMB_PATH_PAIR) {
        smb::Stft2048PairArgs a = pair_args(stft, mel, din, dout, nb, g, power);
        a.max_slot = max_slot;
        CK(smb::launch_stft2048p(a, false, sd.sm_count, st));
      } else if (fast) {
        smb::Stft2048Args a = fused_args(stft, din, dout, nb, g, power);
        a.n_mels = (int)mel->n_mels;
        const auto& sc = fast == SMB_PATH_TENSOR ? mel->sched_tc : mel->sched_cc;
        const auto& tables = fast == SMB_PATH_TENSOR ? mel->dev->tc : mel->dev->cc;
        a.nnz = (int)sc.vals.size();
        a.vals = tables.d_vals.get();
        a.mel_pieces = tables.d_pieces.get();
        a.mel_pcnt = tables.d_pcnt.get();
        a.mel_rounds = sc.rounds;
        a.mel_mpad = sc.mpad;
        if (fast == SMB_PATH_TENSOR) CK(smb::launch_stft2048tc(a, smb::kFastMel, sd.sm_count, st));
        else CK(smb::launch_stft2048(a, smb::kFastMel, sd.sm_count, st));
      } else {
        // two kernels through a plan-owned power spectrogram
        const size_t spec_bytes = (size_t)nb * stft->geom.bins() * g.frames * esz;
        void* spec = stft->tmp.ensure(spec_bytes);
        CK(smb::launch_stft_generic(din, dtype, nb, g, sd.d_window64.get(), sd.d_twiddle64.get(),
                                    smb::kModePower, power, spec, st));
        run_mel_apply(mel, spec, nb, g.frames, dtype, dout, st);
      }
    };
    dispatch(mem, stft->pipe, st, x, out, batch, (size_t)n * esz, (size_t)mel->n_mels * g.frames * esz, run);
  }
  return max_known;
}

// The mel spectrogram of host or device audio into dmel (device), its maximum in the mel
// plan's slot where the return value says so (mel_spectrogram_impl).  Host audio goes up in
// slices of about 64 MB: the whole-tensor maximum needs every slice's mel values before the
// first value in decibels, so those stay on the device -- a quarter of the audio's size --
// but the audio never does at once.
static bool mel_spectrogram_to_device(smb_stft_plan* stft, smb_mel_plan* mel, const void* x,
                                      int64_t batch, int64_t n, int dtype, double power, void* dmel,
                                      int mem) {
  const size_t esz = dtype_size(dtype);
  cudaStream_t st = stft->dev->stream.use;
  unsigned long long* d_max = mel->dev->d_max.get();
  CK(cudaMemsetAsync(d_max, 0, sizeof(unsigned long long), st));
  if (mem == SMB_MEM_DEVICE)
    return mel_spectrogram_impl(stft, mel, x, batch, n, dtype, power, dmel, SMB_MEM_DEVICE, d_max);
  const size_t mel_item = (size_t)mel->n_mels * stft->geom.frames(n) * esz;
  const int64_t per = std::max<int64_t>(1, (int64_t)(64u << 20) / std::max<int64_t>(1, n * (int64_t)esz));
  bool max_known = true;
  for (int64_t b0 = 0; b0 < batch; b0 += per) {
    const int64_t nb = std::min(per, batch - b0);
    void* stage = stft->pipe.in[0].ensure((size_t)std::min(per, batch) * n * esz);
    CK(cudaMemcpyAsync(stage, (const char*)x + (size_t)b0 * n * esz, (size_t)nb * n * esz,
                       cudaMemcpyHostToDevice, st));
    max_known = mel_spectrogram_impl(stft, mel, stage, nb, n, dtype, power,
                                     (char*)dmel + (size_t)b0 * mel_item, SMB_MEM_DEVICE, d_max) &&
                max_known;
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
                             stft->dev->sm_count, stft->dev->stream.use));
  });
}

// ---- dB conversion and MFCC ------------------------------------------------------

}  // extern "C"

namespace {

const double kDecade = 10.0 / std::log(10.0);     // convert.ml:27

// convert.ml:8-22: checks in the reference's order and wording.  Returns whether top_db
// (NaN: none) clamps.
bool check_db_args(const char* fn, double reference, double amin, double top_db) {
  if (!(std::isfinite(reference) && reference > 0.0))
    throw smb::invalid_argument(smb::format("Soundml.Convert.%s: reference must be finite and positive", fn));
  if (!(std::isfinite(amin) && amin > 0.0))
    throw smb::invalid_argument(smb::format("Soundml.Convert.%s: amin must be finite and positive", fn));
  const bool clamp = !std::isnan(top_db);
  if (clamp && !(std::isfinite(top_db) && top_db >= 0.0))
    throw smb::invalid_argument(smb::format("Soundml.Convert.%s: top_db must be finite and non-negative", fn));
  return clamp;
}

void to_db_call(const char* fn, double gain, int magnitude, const void* x, int64_t count,
                int dtype, double reference, double amin, double top_db, void* out, int mem,
                void* stream) {
  const bool clamp = check_db_args(fn, reference, amin, top_db);
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
  const scratch_ptr slot = scratch_alloc(sizeof(unsigned long long), st);
  scratch_ptr din, dout;
  const void* src = x;
  void* dst = out;
  check_mem(mem);
  if (mem == SMB_MEM_HOST) {
    din = scratch_alloc((size_t)count * esz, st);
    dout = scratch_alloc((size_t)count * esz, st);
    CK(cudaMemcpyAsync(din.get(), x, (size_t)count * esz, cudaMemcpyHostToDevice, st));
    src = din.get();
    dst = dout.get();
  }
  CK(smb::launch_to_db(src, count, dtype, magnitude, amin, scale, offset, clamp,
                       clamp ? top_db : 0.0, (unsigned long long*)slot.get(), dst, st));
  if (mem == SMB_MEM_HOST) {
    CK(cudaMemcpyAsync(out, dout.get(), (size_t)count * esz, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));   // the host buffer is the caller's again
  }
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
    require_same_fft("mfcc", stft, mel);
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
    cudaStream_t st = stft->dev->stream.use;
    unsigned long long* d_max = mel->dev->d_max.get();
    // log-mel needs the whole-tensor maximum, so the mel spectrogram is
    // materialised (plan-owned), then reduced, then transformed
    const size_t mel_bytes = (size_t)batch * mel->n_mels * g.frames * esz;
    const size_t out_bytes = (size_t)batch * n_mfcc * g.frames * esz;
    void* dmel = stft->cepstral.ensure(mel_bytes + out_bytes);
    void* dout = mem == SMB_MEM_HOST ? (void*)((char*)dmel + mel_bytes) : out;
    check_mem(mem);
    const bool max_known = mel_spectrogram_to_device(stft, mel, x, batch, n, dtype, 2.0, dmel, mem);
    const double scale = kDecade, offset = scale * std::log(1.0);   // reference 1, amin 1e-10
    CK(smb::launch_mfcc(dmel, dtype, batch, (int)mel->n_mels, g.frames, (int)n_mfcc,
                        mel->dct_table(n_mfcc, has_lifter ? lifter : 0.0), d_max, max_known,
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
    const bool clamp = check_db_args("power_to_db", reference, amin, top_db);
    check_mem(mem);
    // the composition's first checks, in its wording
    require_same_fft("mel_spectrogram", stft, mel);
    check_signal("power_spectrum", batch, n);
    const size_t esz = dtype_size(dtype);
    const smb::FrameGeom g = stft->frame_geom(n);
    if (batch == 0 || g.frames == 0) return;
    stft->ensure_device();
    mel->ensure_device();
    cudaStream_t st = stft->dev->stream.use;
    unsigned long long* d_max = mel->dev->d_max.get();
    const int64_t count = batch * mel->n_mels * g.frames;
    // the result stays on the device until it is in decibels
    void* dmel = mem == SMB_MEM_HOST ? stft->cepstral.ensure((size_t)count * esz) : out;
    const bool max_known = mel_spectrogram_to_device(stft, mel, x, batch, n, dtype, power, dmel, mem);
    const double scale = kDecade;                                   // gain 10: powers
    const double offset = scale * std::log(std::max(amin, reference));
    if (max_known)
      CK(smb::launch_db_known_max(dmel, count, dtype, amin, scale, offset, clamp, clamp ? top_db : 0.0,
                                  d_max, st));
    else
      CK(smb::launch_to_db(dmel, count, dtype, 0, amin, scale, offset, clamp, clamp ? top_db : 0.0,
                           d_max, dmel, st));
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
  return guarded([&] { plan->ensure_device(); plan->dev->stream.set(s); });
}
int smb_resample_plan_sync(smb_resample_plan* plan) {
  return guarded([&] { if (plan->dev) CK(cudaStreamSynchronize(plan->dev->stream.use)); });
}
int smb_resample_plan_set_executor(smb_resample_plan* plan, int exec) {
  return guarded([&] {
    if (exec != SMB_EXEC_DIRECT && exec != SMB_EXEC_PLANNED)
      throw smb::invalid_argument("set_executor: SMB_EXEC_DIRECT or SMB_EXEC_PLANNED");
    plan->executor = exec;
  });
}
static const smb::ResampleStage& stage_of(const smb_resample_plan* plan, int stage, const char* op) {
  if (stage < 0 || stage >= (int)plan->plan.stages.size())
    throw smb::invalid_argument(smb::format("%s: no such stage", op));
  return plan->plan.stages[(size_t)stage];
}
int smb_resample_stage_layout(smb_resample_plan* plan, int stage, int group,
                              smb_resample_layout* out) {
  return guarded([&] {
    const smb::ResampleStage& s = stage_of(plan, stage, "stage_layout");
    plan->build_tables();
    const smb::GemmLayout& gl = plan->tables[(size_t)stage].gemm;
    smb_resample_layout r{};
    r.form = plan->form((size_t)stage);
    r.groups = r.form == SMB_FORM_ROW ? (int)gl.rows.size()
             : r.form == SMB_FORM_WINDOW ? (int)gl.windows.size() : 1;
    if (group < 0 || group >= r.groups) throw smb::invalid_argument("stage_layout: no such column group");
    if (r.form == SMB_FORM_ROW) {
      const smb::GemmRowsArgs& a = gl.rows[(size_t)group].a;
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
      const smb::GemmResampleArgs& a = gl.windows[(size_t)group].a;
      r.columns = a.l;
      r.col_begin = a.col_begin;
      r.chunks = a.chunks;
    } else {
      r.columns = (int)s.l;
    }
    *out = r;
  });
}
static void ols_geometry_of(const smb::OlsPlan& p, smb_ols_geometry* out) {
  smb_ols_geometry g{};
  g.kernel = ols_kernel_of(p);
  if (g.kernel != SMB_OLS_NONE) {
    g.n = p.n; g.b = p.b; g.delta = p.delta; g.w = p.w;
    g.l = p.l; g.m = p.m; g.k = p.k;
    g.polyphase = p.polyphase ? 1 : 0;
    g.full_inverse = p.full_inverse ? 1 : 0;
  }
  *out = g;
}
int smb_resample_stage_ols(const smb_resample_plan* plan, int stage, smb_ols_geometry* out) {
  return guarded([&] {
    ols_geometry_of(smb::ols_plan_for_stage(stage_of(plan, stage, "stage_ols")), out);
  });
}
int smb_fir_ols(const smb_fir_plan* plan, smb_ols_geometry* out) {
  return guarded([&] { ols_geometry_of(smb::ols_plan_for_fir(plan->h), out); });
}
int64_t smb_ols_blocks(const smb_ols_geometry* g, int64_t n_out) {
  int64_t r = -1;
  guarded([&] {
    if (g->kernel == SMB_OLS_NONE || g->b < 1 || g->l < 1 || g->m < 1 || (g->l > 1 && g->m != 1))
      throw smb::invalid_argument("ols_blocks: not an overlap-save geometry");
    smb::OlsPlan p;
    p.n = g->n; p.b = g->b; p.delta = g->delta; p.l = g->l; p.m = g->m; p.k = g->k;
    r = p.blocks_for(n_out);
  });
  return r;
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
    const smb::ResampleStage& s = stage_of(plan, stage, "stage_info");
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
    const smb::ResampleStage& s = stage_of(plan, stage, "stage_design");
    if (fc) *fc = s.fc;
    if (beta) *beta = s.beta;
  });
}
int smb_resample_stage_prototype(const smb_resample_plan* plan, int stage, double* out,
                                 int64_t* len) {
  return guarded([&] {
    const std::vector<double>& h = stage_of(plan, stage, "stage_prototype").proto;
    if (len) *len = (int64_t)h.size();
    if (out) std::memcpy(out, h.data(), h.size() * sizeof(double));
  });
}
int64_t smb_resample_output_frames(const smb_resample_plan* plan, int64_t n) {
  int64_t r = -1;
  guarded([&] { r = plan->plan.output_frames(n); });
  return r;
}

}  // extern "C"

// Resample.apply over a batch of independent signals: a copy for the identity, one stage, or
// a cascade through the plan's hand-off buffer; a host batch goes through in slices, the
// copies of one slice under the kernels of its neighbours (HostPipe).
// stage(i, x, nb, n, n_out, out, st) launches stage i over device buffers.
template <typename T, typename Stage>
static void resample_call(smb_resample_plan* plan, const T* x, int64_t batch, int64_t n, T* out,
                          int mem, Stage&& stage) {
  if (batch < 0) throw smb::invalid_argument("apply: negative batch");
  const smb::ResamplePlan& rp = plan->plan;
  const int64_t total = rp.output_frames(n);
  if (batch == 0 || n == 0 || total == 0) return;
  plan->ensure_device();
  cudaStream_t st = plan->dev->stream.use;
  auto run = [&](const void* din_v, void* dout_v, int64_t nb) {
    const T* din = (const T*)din_v;
    T* dout = (T*)dout_v;
    if (rp.identity()) {
      CK(cudaMemcpyAsync(dout, din, (size_t)nb * n * sizeof(T), cudaMemcpyDeviceToDevice, st));
    } else if (rp.stages.size() == 1) {
      stage(0, din, nb, n, total, dout, st);
    } else {
      // cascade (resample.ml:1819-1842): stage 1 emits its exact ceil tail,
      // stage 2 runs over it with zeros beyond and is cut to output_frames.
      const smb::ResampleStage& s1 = rp.stages[0];
      const int64_t n1 = (n * s1.l + s1.m - 1) / s1.m;
      T* mid = (T*)plan->mid.ensure((size_t)nb * n1 * sizeof(T));
      stage(0, din, nb, n, n1, mid, st);
      stage(1, mid, nb, n1, total, dout, st);
    }
  };
  dispatch(mem, plan->pipe, st, x, out, batch, (size_t)n * sizeof(T), (size_t)total * sizeof(T), run);
}

extern "C" {

int smb_resample_apply(smb_resample_plan* plan, const float* x, int64_t batch, int64_t n,
                       float* out, int mem) {
  return guarded([&] {
    resample_call(plan, x, batch, n, out, mem,
                  [&](size_t i, const float* src, int64_t nb, int64_t len, int64_t n_out, float* dst,
                      cudaStream_t st) { plan->run_stage(i, src, nb, len, n_out, dst, st); });
  });
}

// float64 audio: the reference's executor carries both dtypes (resample.ml:72-84);
// here double always takes the direct kernel, in double.
int smb_resample_apply_f64(smb_resample_plan* plan, const double* x, int64_t batch, int64_t n,
                           double* out, int mem) {
  return guarded([&] {
    resample_call(plan, x, batch, n, out, mem,
                  [&](size_t i, const double* src, int64_t nb, int64_t len, int64_t n_out, double* dst,
                      cudaStream_t st) {
                    const smb::ResampleStage& s = plan->plan.stages[i];
                    CK(smb::launch_polyphase_direct_f64(src, nb, len, plan->dev->stages[i].d_bank64.get(), (int)s.l,
                                                        (int)s.m, (int)s.k, n_out, dst, st));
                  });
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
      CK(cudaMemcpy2DAsync(next.ptr.get(), (size_t)grown * esz, carry[cur].ptr.get(), (size_t)cap * esz,
                           (size_t)(fed - base) * esz, (size_t)channels, cudaMemcpyDeviceToDevice, st));
    CK(cudaStreamSynchronize(st));
    carry[cur] = std::move(next);
    carry[1 - cur].ensure((size_t)channels * grown * esz);     // (larger than it was: reallocates)
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
    CK(cudaMemcpy2DAsync(w, (size_t)len * esz, (char*)carry[cur].ptr.get() + (size_t)(a0 - base) * esz,
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
        CK(cudaMemcpy2DAsync(carry[1 - cur].ptr.get(), (size_t)cap * esz,
                             (char*)carry[cur].ptr.get() + (size_t)(keep - base) * esz, (size_t)cap * esz,
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
int smb_resample_kernel_destroy(smb_resample_kernel* k) { return guarded([&] { delete k; }); }
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
    check_mem(mem);
    if (n == 0) return;
    k->plan->ensure_device();
    cudaStream_t st = k->plan->dev->stream.use;
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
    CK(cudaMemcpy2DAsync((char*)k->carry[k->cur].ptr.get() + (size_t)(k->fed - k->base) * k->esz,
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
    check_mem(mem);
    const int64_t total = k->fed ? k->plan->plan.output_frames(k->fed) : 0;
    if (total <= k->emitted) return;
    k->plan->ensure_device();
    cudaStream_t st = k->plan->dev->stream.use;
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
  return guarded([&] { plan->ensure_device(); plan->dev->stream.set(s); });
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
      method = plan->dev->ols_plan.ok && plan->k >= 8 ? SMB_EXEC_OLS : SMB_EXEC_DIRECT;
    if (method == SMB_EXEC_OLS && !plan->dev->ols_plan.ok)
      throw smb::invalid_argument(
          "fir: this filter is too long for the overlap-save kernel (use the direct method)");
    cudaStream_t st = plan->dev->stream.use;
    auto run = [&](const void* din, void* dout, int64_t nb) {
      if (method == SMB_EXEC_OLS)
        plan->dev->ols.run(plan->dev->ols_plan, (const float*)din, nb, n, n, (float*)dout, plan->dev->sm_count,
                           st);
      else
        CK(smb::launch_polyphase_direct((const float*)din, nb, n, plan->dev->d_bank.get(), 1, 1, (int)plan->k, n,
                                        (float*)dout, st));
    };
    dispatch(mem, plan->pipe, st, x, out, batch, (size_t)n * 4, (size_t)n * 4, run);
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
    check_mem(mem_in);
    check_mem(mem_out);
    if (frames == 0) return;
    require_device();
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const int64_t width = mode == SMB_INGEST_PLANAR ? channels : 1;
    // staging per thread and per device: kernels only ever see a buffer of the current device
    static thread_local std::vector<DeviceBuffer> stage_in, stage_out;
    int device = 0;
    CK(cudaGetDevice(&device));
    if ((size_t)device >= stage_in.size()) {
      stage_in.resize((size_t)device + 1);
      stage_out.resize((size_t)device + 1);
    }
    const void* din = interleaved;
    if (mem_in == SMB_MEM_HOST) {
      void* up = stage_in[(size_t)device].ensure((size_t)frames * channels * esz);
      CK(cudaMemcpyAsync(up, interleaved, (size_t)frames * channels * esz, cudaMemcpyHostToDevice, st));
      din = up;
    }
    if (mem_out == SMB_MEM_DEVICE) {
      CK(smb::launch_ingest_layout(din, dtype, frames, (int)channels, mode == SMB_INGEST_DOWNMIX,
                                   (char*)out + (size_t)out_off * esz, out_total, st));
      if (mem_in == SMB_MEM_HOST) CK(cudaStreamSynchronize(st));   // the host block may be reused
    } else {
      void* dn = stage_out[(size_t)device].ensure((size_t)frames * width * esz);
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
  // streams first: they outlive everything used on them
  stream_ptr own_compute;                       // native rate: the compute stream
  stream_ptr copy;
  std::unique_ptr<smb_resample_plan> plan;      // null: native rate
  std::unique_ptr<smb_resample_kernel> kernel;  // borrows the plan: declared after it, destroyed first
  cudaStream_t compute = nullptr;               // own_compute, or the plan's stream
  pinned_ptr staging[2];
  DeviceBuffer up[2], planar;
  event_ptr copied[2], consumed[2];
  bool in_flight[2] = {false, false};
  int cur = 0;
  bool finished = false;
  int64_t frames_in = 0, frames_out = 0;
  ~smb_ingest() {
    // an upload in flight may still read a pinned block: drain before anything is freed
    if (copy) cudaStreamSynchronize(copy.get());
    if (compute) cudaStreamSynchronize(compute);
  }
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
      smb_resample_plan* plan = nullptr;
      if (smb_resample_plan_create(&plan, sample_rate, target, quality, 0.0, 0.0) != SMB_OK)
        throw smb::invalid_argument(t_error);
      r->plan.reset(plan);
      smb_resample_kernel* kernel = nullptr;
      if (smb_resample_kernel_create(&kernel, plan, dtype, r->width, r->max_block) != SMB_OK)
        throw smb::invalid_argument(t_error);
      r->kernel.reset(kernel);
      plan->ensure_device();
      r->compute = plan->dev->stream.use;
    } else {
      r->own_compute = new_stream();
      r->compute = r->own_compute.get();
    }
    r->copy = new_stream();
    for (int i = 0; i < 2; ++i) {
      void* block = nullptr;
      CK(cudaMallocHost(&block, (size_t)r->max_block * channels * esz));
      r->staging[i].reset(block);
      r->up[i].ensure((size_t)r->max_block * channels * esz);
      r->copied[i] = new_event();
      r->consumed[i] = new_event();
    }
    r->planar.ensure((size_t)r->max_block * r->width * esz);
    *reader = r.release();
  });
}
int smb_ingest_destroy(smb_ingest* r) { return guarded([&] { delete r; }); }
int64_t smb_ingest_max_block(const smb_ingest* r) { return r->max_block; }
int smb_ingest_staging(smb_ingest* r, void** block) {
  return guarded([&] {
    same_device(r->bound_device);
    // the upload that last read this block (two submits ago) must have left the host
    if (r->in_flight[r->cur]) {
      CK(cudaEventSynchronize(r->copied[r->cur].get()));
      r->in_flight[r->cur] = false;
    }
    *block = r->staging[r->cur].get();
  });
}
int64_t smb_ingest_submit_frames(const smb_ingest* r, int64_t frames) {
  if (r->finished || frames <= 0) return 0;
  return r->kernel ? smb_resample_kernel_step_frames(r->kernel.get(), frames) : frames;
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
    cudaEvent_t copied = r->copied[b].get(), consumed = r->consumed[b].get();
    void* up = r->up[b].ptr.get();
    // the layout pass that last read up[b] must be done before the copy overwrites it
    CK(cudaStreamWaitEvent(r->copy.get(), consumed, 0));
    CK(cudaMemcpyAsync(up, r->staging[b].get(), (size_t)frames * r->channels * r->esz,
                       cudaMemcpyHostToDevice, r->copy.get()));
    CK(cudaEventRecord(copied, r->copy.get()));
    r->in_flight[b] = true;
    CK(cudaStreamWaitEvent(r->compute, copied, 0));
    const int64_t released = smb_ingest_submit_frames(r, frames);
    if (r->kernel) {
      CK(smb::launch_ingest_layout(up, r->dtype, frames, (int)r->channels,
                                   r->mode == SMB_INGEST_DOWNMIX, r->planar.ptr.get(), frames, r->compute));
      CK(cudaEventRecord(consumed, r->compute));
      if (smb_resample_kernel_step(r->kernel.get(), r->planar.ptr.get(), frames, out_device, SMB_MEM_DEVICE) != SMB_OK)
        throw cuda_failure(t_error);
    } else {
      CK(smb::launch_ingest_layout(up, r->dtype, frames, (int)r->channels,
                                   r->mode == SMB_INGEST_DOWNMIX, out_device, frames, r->compute));
      CK(cudaEventRecord(consumed, r->compute));
    }
    r->frames_in += frames;
    r->frames_out += released;
    r->cur = 1 - b;
  });
}
int64_t smb_ingest_finish_frames(const smb_ingest* r) {
  return (r->finished || !r->kernel) ? 0 : smb_resample_kernel_flush_frames(r->kernel.get());
}
int smb_ingest_finish(smb_ingest* r, void* out_device) {
  return guarded([&] {
    same_device(r->bound_device);
    if (r->finished) return;
    const int64_t tail = smb_ingest_finish_frames(r);
    r->finished = true;
    if (r->kernel && smb_resample_kernel_flush(r->kernel.get(), out_device, SMB_MEM_DEVICE) != SMB_OK)
      throw cuda_failure(t_error);
    r->frames_out += tail;
  });
}
int smb_ingest_sync(smb_ingest* r) {
  return guarded([&] {
    CK(cudaStreamSynchronize(r->copy.get()));
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
