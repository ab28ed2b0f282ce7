// Fused STFT + mel kernel for fft_size = 2048, float32 audio (sm_100a): the
// "frame-pair" kernel.
//
//   framing + boundary extension + window -> real FFT 2048 -> |X|^p
//   -> sparse mel projection -> [batch, n_mels, frames]
//
// replaces Stft.analyse / magnitude_pow / Mel.apply (stft.ml:356-364, 670-674;
// mel.ml:202-231) for Soundml.mel_spectrogram (soundml.ml:12-24) in one launch; the
// complex spectrum and the power spectrogram never reach HBM.
//
// What is different from stft2048.cu (which stays for the bin-major outputs and the
// zero-padded shorter frames): a warp transforms TWO consecutive frames of a clip at
// once, every value a float32x2 register pair (frame A, frame B).  Hop-adjacent frames
// use the same window, the same FFT twiddles and the same split twiddles, so
//   * every arithmetic instruction of the transform is a packed FADD2 / FMUL2 / FFMA2
//     with the constant as an immediate or broadcast operand: half the issue slots;
//   * window, inter-pass twiddle and split twiddle are fetched once per two frames:
//     half the shared-memory wavefronts of the tables;
//   * the transposition between the passes and the pass-2 loads move 16 bytes per lane
//     (LDS.128 / STS.128), half the instructions;
//   * the mel band product reads (bin, bin + 1) x (frame A, frame B) as one 16-byte
//     load and accumulates both frames with one FFMA2 per weight; a lane owns a whole
//     filter for one frame pair, so its result goes straight to global memory: no
//     partial sums, no second barrier.
// The float32 pipe does the same number of lane-operations as before; it is what
// bounds the kernel now (see DESIGN.md 4.1).
//
// Decomposition: one persistent CTA per SM, 8 warps in two independent groups of 4;
// a group owns a tile of 8 consecutive frames of one clip (staged once, by one bulk
// copy one tile ahead when the source run is aligned), warp w takes frames 2w, 2w+1.
// Real FFT 2048 = complex FFT 1024 on z[n] = x[2n] + i x[2n+1] as 32 x 32 register
// passes with a transposition through a warp-private padded buffer; the real-spectrum
// split pairs bin k with 1024 - k by warp shuffle.  The power rows of a warp's two
// frames overwrite its own transposition buffer, [bin][2 frames].
#include <algorithm>
#include <cstdint>

#include "fft32x2.cuh"
#include "kernels.h"
#include "max_key.cuh"
#include "stft_stage.cuh"

namespace smb {

namespace {

using namespace fft32x2;
using fft32impl::kW64C;
using fft32impl::kW64S;

constexpr int kTile = kPairTile;            // frames per group tile
constexpr int kGroupWarps = kTile / 2;      // a warp carries two frames
constexpr int kGroupThreads = 32 * kGroupWarps;
constexpr int kGroups = 16 / kTile;          // eight warps in all
constexpr int kF = kPairFilters;             // filters per mel round
constexpr int kExPitch = 33;                // 16-byte elements per transposition row (conflict-free both ways)
constexpr int kWarpBuf = 32 * kExPitch * 16;   // bytes: [32][33] x (re A, re B, im A, im B)
constexpr int kPowerBins = 1032;            // bins per power row incl. the zeroed tail the mel steps may read
static_assert(32 * (kGroupWarps - 1) + kPowerBins * 8 <= kWarpBuf, "power rows fit the transposition buffer");

enum Mode { kModeMel = 0, kModeCeiling = 1 };

struct Params {
  Stft2048PairArgs a;
  stage::BulkRule bulk;
  int span_bytes;            // bytes reserved per group for samples (multiple of 128)
  int tables_bytes;          // reserved bytes, split twiddles, mel tables (multiple of 128)
  int tiles_per_signal, total_tiles;
};

// ---- TMEM as a per-lane table store.  The window and the inter-pass twiddles are
// per-lane constants (lane = n2 needs w[64 n1 + 2 n2 + c] and W1024^(k1 n2) for every
// n1, k1): 128 floats per lane, too many for registers, and as shared-memory tables
// they cost 64 of the kernel's ~400 wavefronts per frame on the pipe that bounds it.
// Tensor memory is organised exactly that way -- 128 lanes x 512 32-bit columns, a
// warp reading "its" 32 lanes with tcgen05.ld.32x32b -- and has its own datapath, so
// the tables live there: columns [0, 64) window, [64, 128) twiddles, one copy per
// 32-lane quarter (warps w and w + 4 share quarter w % 4).
constexpr uint32_t kTmemCols = 128;
// tmem_ld16 (sm100.cuh) leaves the wait to this one: naming the registers orders their
// first use behind it
__device__ __forceinline__ void tmem_wait16(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]),
                 "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]),
                 "+r"(r[13]), "+r"(r[14]), "+r"(r[15]));
}

__device__ __forceinline__ pk_t shfl_pk(pk_t v, int src) {
  return __shfl_sync(0xffffffffu, v, src);
}

// |x|^p of both frames; SQUARE: p = 2
template <bool SQUARE>
__device__ __forceinline__ pk_t power_of(CP x, float power) {
  const pk_t sq = pfma(x.im, x.im, pmul(x.re, x.re));
  if (SQUARE) return sq;
  float a = pk_lo(sq), b = pk_hi(sq);
  if (power == 1.0f) { a = sqrtf(a); b = sqrtf(b); }
  else { a = powf(sqrtf(a), power); b = powf(sqrtf(b), power); }
  return pk(a, b);
}

// ROWS: hop / 64 when the hop is a multiple of 64 and at most 1024, else 0.  Frame B
// starts hop samples = ROWS rows of 32 complex points after frame A, so row n1 of B
// is row n1 + ROWS of A in the same lane: the pair needs 32 + ROWS sample loads
// instead of 64.
template <bool SQUARE, int MODE, int ROWS>
__global__ void __launch_bounds__(kGroups * kGroupThreads, 1)
stft2048p_kernel(const Params p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  // tables: [0, 16384) unused (see tables_bytes_needed); split twiddles [32] float2;
  // mel weights; mel items
  float2* sTwPost = reinterpret_cast<float2*>(smem_raw + 16384);
  float* sMelW = reinterpret_cast<float*>(smem_raw + 16640);
  PairMelItem* sItems = reinterpret_cast<PairMelItem*>(sMelW + p.a.mel_w_floats);
  __shared__ __align__(8) uint64_t sbars[kGroups];
  __shared__ __align__(8) uint64_t sfree[kGroups];     // a group's power rows have been read (4 warps arrive)
  __shared__ uint32_t tmem_slot;

  const int tid = threadIdx.x;
  const int group = tid / kGroupThreads;
  const int gtid = tid % kGroupThreads;
  const int warp = gtid >> 5;
  const int lane = tid & 31;
  unsigned char* gbase = smem_raw + p.tables_bytes + group * (p.span_bytes + kGroupWarps * kWarpBuf);
  float* sSamples = reinterpret_cast<float*>(gbase);
  unsigned char* sBufs = gbase + p.span_bytes;                 // kGroupWarps transposition buffers
  unsigned char* ex = sBufs + warp * kWarpBuf;                 // this warp's
  float* prow = reinterpret_cast<float*>(ex + 32 * warp);      // its power rows, [bin][2]

  if (tid < 32) tmem_alloc(&tmem_slot, kTmemCols);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  // tensor-memory address of this warp's table rows
  const uint32_t ttab = tmem_slot + ((uint32_t)(((tid >> 5) & 3) * 32) << 16);
  if (tid < 128) {                       // one warp per 32-lane quarter fills it
    uint32_t v[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
#pragma unroll
      for (int e = 0; e < 16; ++e)       // column 2 n1 + c: w[64 n1 + 2 lane + c] / 2
        v[e] = __float_as_uint(p.a.window[64 * (8 * q + (e >> 1)) + 2 * lane + (e & 1)] * 0.5f);
      tmem_st16(ttab + 16 * q, v);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
#pragma unroll
      for (int e = 0; e < 16; ++e) {     // column 64 + 2 k1 + c: W1024^(k1 lane)
        const float2 t = p.a.tw_pass[(8 * q + (e >> 1)) * 32 + lane];
        v[e] = __float_as_uint((e & 1) ? t.y : t.x);
      }
      tmem_st16(ttab + 64 + 16 * q, v);
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");   // ordered by the barrier below
  if (tid < 32) sTwPost[tid] = p.a.tw_post[tid];
  if (MODE == kModeMel) {
    for (int i = tid; i < p.a.mel_w_floats; i += blockDim.x) sMelW[i] = p.a.mel_w[i];
    for (int i = tid; i < kGroupWarps * p.a.mel_rounds * kF; i += blockDim.x) sItems[i] = p.a.mel_items[i];
  }
  if (tid == 0) {
    for (int gI = 0; gI < kGroups; ++gI) {
      mbar_init(smem_u32(&sbars[gI]), 1);
      mbar_init(smem_u32(&sfree[gI]), kGroupWarps);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t sbar = smem_u32(&sbars[group]);
  const uint32_t fbar = smem_u32(&sfree[group]);
  uint32_t sphase = 0, tiles_done = 0;

  const FrameGeom g = p.a.g;
  const int mel_rounds = p.a.mel_rounds;
  const int slot = blockIdx.x * kGroups + group;
  const int stride = gridDim.x * kGroups;
  const int total_tiles = p.total_tiles, tiles_per_signal = p.tiles_per_signal;
  // (clip, tile of the clip) walk the round-robin deal without a division per tile
  const int step_b = stride / tiles_per_signal, step_t = stride - step_b * tiles_per_signal;
  int nb = slot / tiles_per_signal, nt = slot - nb * tiles_per_signal;
  float vmax = 0.0f;                       // maximum of what this thread writes (mel values are >= 0)
  bool bulk = false;
  if (slot < total_tiles)
    bulk = stage::stage_tile<kTile, kGroupThreads>(g, p.a.x, p.bulk, nb, nt, sSamples, gtid, sbar);

  for (int tile = slot; tile < total_tiles; tile += stride) {
    const int b = nb;
    const long long p0 = (long long)nt * kTile;
    nb += step_b;
    nt += step_t;
    if (nt >= tiles_per_signal) { nt -= tiles_per_signal; ++nb; }
    const int nf = (int)min((long long)kTile, g.frames - p0);

    // ---- the tile's samples were requested one iteration ago
    // no group barrier here when the tile came by bulk copy: every thread sees the
    // samples through the mbarrier, and the only other thing the barrier ordered -- the
    // previous tile's mel reads of the power rows against this tile's transposition
    // stores -- is waited for where it matters, just before those stores (sfree)
    if (bulk) {
      mbar_wait(sbar, sphase & 1);
      ++sphase;
    } else {
      asm volatile("cp.async.wait_all;" ::: "memory");
      named_sync(group + 1, kGroupThreads);
    }

    {
      // ---- pass 1: lane = n2, registers = n1; z[n] = x[2n] + i x[2n+1], n = 32 n1 + n2.
      // Frames past the end of a tail tile read stale (in-bounds) samples; their
      // results are never written.  (No branch around the transform: the shuffles of
      // the split then sit in code the compiler knows to be convergent.)
      CP a[32];
      if (ROWS > 0) {
        const float2* sA = reinterpret_cast<const float2*>(sSamples + 2 * warp * g.hop) + lane;
        float2 raw[32 + ROWS];
#pragma unroll
        for (int r = 0; r < 32 + ROWS; ++r) raw[r] = sA[32 * r];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint32_t wv[16];
          tmem_ld16(ttab + 16 * q, wv);
          tmem_wait16(wv);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int n1 = 8 * q + e;
            const float wx = __uint_as_float(wv[2 * e]), wy = __uint_as_float(wv[2 * e + 1]);
            a[n1] = CP{pk(raw[n1].x * wx, raw[n1 + ROWS].x * wx), pk(raw[n1].y * wy, raw[n1 + ROWS].y * wy)};
          }
        }
      } else {
        const float2* sA = reinterpret_cast<const float2*>(sSamples + 2 * warp * g.hop) + lane;
        const float2* sB = reinterpret_cast<const float2*>(sSamples + (2 * warp + 1) * g.hop) + lane;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint32_t wv[16];
          tmem_ld16(ttab + 16 * q, wv);
          tmem_wait16(wv);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int n1 = 8 * q + e;
            const float2 a0 = sA[32 * n1], b0 = sB[32 * n1];
            const float wx = __uint_as_float(wv[2 * e]), wy = __uint_as_float(wv[2 * e + 1]);
            a[n1] = CP{pk(a0.x * wx, b0.x * wx), pk(a0.y * wy, b0.y * wy)};
          }
        }
      }
      fft32(a);                                   // a[k1] = Y[n2 = lane][k1]
      // ---- the previous tile's power rows (this buffer) have been read by all four warps
      if (tiles_done > 0) mbar_wait(fbar, (tiles_done - 1) & 1);
      // ---- twiddle W1024^(k1 n2), transpose through the warp's padded buffer
      {
        ulonglong2* st = reinterpret_cast<ulonglong2*>(ex) + lane;
        uint32_t tv[16];
#pragma unroll
        for (int k1 = 0; k1 < 32; k1 += 2) {
          if ((k1 & 7) == 0) {
            tmem_ld16(ttab + 64 + 2 * k1, tv);
            tmem_wait16(tv);
          }
          const float4 t = make_float4(__uint_as_float(tv[2 * (k1 & 7)]), __uint_as_float(tv[2 * (k1 & 7) + 1]),
                                       __uint_as_float(tv[2 * (k1 & 7) + 2]), __uint_as_float(tv[2 * (k1 & 7) + 3]));
          const CP v0 = k1 == 0 ? a[0]
                                : CP{pfmas(a[k1].im, -t.y, pmuls(a[k1].re, t.x)),
                                     pfmas(a[k1].im, t.x, pmuls(a[k1].re, t.y))};
          const CP v1 = CP{pfmas(a[k1 + 1].im, -t.w, pmuls(a[k1 + 1].re, t.z)),
                           pfmas(a[k1 + 1].im, t.z, pmuls(a[k1 + 1].re, t.w))};
          st[k1 * kExPitch] = make_ulonglong2(v0.re, v0.im);
          st[(k1 + 1) * kExPitch] = make_ulonglong2(v1.re, v1.im);
        }
      }
      __syncwarp();
      // ---- pass 2: lane = k1, registers = n2  ->  a[k2] = Z'[k1 + 32 k2]
      {
        const ulonglong2* ld = reinterpret_cast<const ulonglong2*>(ex) + lane * kExPitch;
#pragma unroll
        for (int n2 = 0; n2 < 32; ++n2) {
          const ulonglong2 v = ld[n2];
          a[n2] = CP{v.x, v.y};
        }
      }
      __syncwarp();                               // the buffer becomes the power rows
      fft32(a);

      if (MODE != kModeMel) {
        // the measurement floor: no split, no |X|^2, no mel -- one store per value
#pragma unroll
        for (int k2 = 0; k2 < 32; ++k2)
          *reinterpret_cast<pk_t*>(prow + 2 * (lane + 32 * k2)) = padd(a[k2].re, a[k2].im);
      } else {
        // ---- real-spectrum split.  With Z' = Z/2 (window pre-scaled):
        //   S = Z'[k] + conj Z'[N-k],  D = Z'[k] - conj Z'[N-k],  W = W2048^k
        //   X[k] = S + W (-i D),   X[N-k] = conj(S - W (-i D))
        const int partner = (32 - lane) & 31;
        const float2 wl = sTwPost[lane];
        const bool first = lane == 0;
#pragma unroll
        for (int k2 = 0; k2 < 16; ++k2) {
          // lanes != 0 need the partner's register 31-k2; lane 0 pairs with itself
          // through register (32-k2) mod 32
          const CP own = a[31 - k2], alt = a[(32 - k2) & 31];
          const CP r = CP{shfl_pk(first ? alt.re : own.re, partner),
                          shfl_pk(first ? alt.im : own.im, partner)};
          const CP A = a[k2];
          const CP S = CP{padd(A.re, r.re), psub(A.im, r.im)};
          const CP D = CP{psub(A.re, r.re), padd(A.im, r.im)};
          const float wx = k2 == 0 ? wl.x : wl.x * kW64C[k2] - wl.y * kW64S[k2];
          const float wy = k2 == 0 ? wl.y : wl.x * kW64S[k2] + wl.y * kW64C[k2];
          const pk_t tr = pfmas(D.re, wy, pmuls(D.im, wx));      // w.x D.im + w.y D.re
          const pk_t ti = pfmas(D.re, -wx, pmuls(D.im, wy));     // w.y D.im - w.x D.re
          const CP xk = CP{padd(S.re, tr), padd(S.im, ti)};
          const CP xn = CP{psub(S.re, tr), psub(ti, S.im)};
          const int k = lane + 32 * k2;
          *reinterpret_cast<pk_t*>(prow + 2 * k) = power_of<SQUARE>(xk, p.a.power);
          *reinterpret_cast<pk_t*>(prow + 2 * (1024 - k)) = power_of<SQUARE>(xn, p.a.power);
        }
        if (first) {                              // k = 512 pairs with itself
          const CP xm = CP{padd(a[16].re, a[16].re), padd(a[16].im, a[16].im)};   // |.| ignores the conjugate
          *reinterpret_cast<pk_t*>(prow + 2 * 512) = power_of<SQUARE>(xm, p.a.power);
        } else if (lane < kPowerBins - 1024) {
          *reinterpret_cast<pk_t*>(prow + 2 * (1024 + lane)) = 0ull;   // tail read by the mel steps
        }
      }
    }
    named_sync(group + 1, kGroupThreads);
    // ---- the sample buffer is free: fetch the next tile under the mel phase
    if (tile + stride < total_tiles)
      bulk = stage::stage_tile<kTile, kGroupThreads>(g, p.a.x, p.bulk, nb, nt, sSamples, gtid, sbar);

    if (MODE == kModeMel) {
      // ---- mel projection.  lane = (filter i of the round's eight, frame pair j): one
      // 16-byte load brings bins (k, k+1) of frames (2j, 2j+1) from warp j's power rows
      // (row bases 32 j bytes apart and filter starts of alternating parity keep a
      // quarter-warp's loads in distinct bank groups); one FFMA2 per weight.  Bin
      // k = b0 + u of the band goes to accumulator u mod 4, in ascending order; the
      // four are added pairwise at the end -- a fixed summation tree.
      const int i = lane / kGroupWarps, j = lane % kGroupWarps;
      const ulonglong2* pj = reinterpret_cast<const ulonglong2*>(sBufs + j * kWarpBuf + 32 * j);
      const int2* mine = reinterpret_cast<const int2*>(sItems + warp * p.a.mel_rounds * kF + i);
      const bool okA = 2 * j < nf, okB = 2 * j + 1 < nf;
      float* ob = p.a.out + (long long)b * p.a.n_mels * g.frames + p0 + 2 * j;
      const int frames = (int)g.frames;                     // n_mels * frames < 2^31 (launcher)
      for (int r = 0; r < mel_rounds; ++r) {
        const int2 it = mine[r * kF];                       // {weights | iterations << 24, h0 | m << 16}
        const int iters = (int)((unsigned)it.x >> 24);      // two 4-bin steps each; the same for the whole warp
        if (iters == 0) break;                              // idle rounds come last
        const float4* wq = reinterpret_cast<const float4*>(sMelW) + (it.x & 0xFFFFFF);
        const ulonglong2* pp = pj + (it.y & 0xFFFF);
        // four independent accumulator chains; every step's loads are in flight under
        // the FMAs of the step before (the last iteration reads one step past the
        // band -- inside the tables, never used)
        pk_t acc0 = 0ull, acc1 = 0ull, acc2 = 0ull, acc3 = 0ull;
        float4 wa = wq[0];
        ulonglong2 a01 = pp[0], a23 = pp[1];
#pragma unroll 1
        for (int t = 0; t < iters; ++t) {
          const float4 wb = wq[kF];
          const ulonglong2 b01 = pp[2], b23 = pp[3];
          acc0 = pfmas(a01.x, wa.x, acc0);
          acc1 = pfmas(a01.y, wa.y, acc1);
          acc2 = pfmas(a23.x, wa.z, acc2);
          acc3 = pfmas(a23.y, wa.w, acc3);
          wq += 2 * kF;
          pp += 4;
          if (t + 1 < iters) {            // (warp-uniform) nothing is fetched past the band
            wa = wq[0];
            a01 = pp[0];
            a23 = pp[1];
          }
          acc0 = pfmas(b01.x, wb.x, acc0);
          acc1 = pfmas(b01.y, wb.y, acc1);
          acc2 = pfmas(b23.x, wb.z, acc2);
          acc3 = pfmas(b23.y, wb.w, acc3);
        }
        const pk_t acc = padd(padd(acc0, acc1), padd(acc2, acc3));
        const int m = it.y >> 16;
        float* o = ob + m * frames;
        if (m >= 0 && okA) { o[0] = pk_lo(acc); vmax = fmaxf(vmax, pk_lo(acc)); }
        if (m >= 0 && okB) { o[1] = pk_hi(acc); vmax = fmaxf(vmax, pk_hi(acc)); }
      }
    } else {
      // ceiling mode: one value per thread and tile keeps the rows alive
      if (p.a.out) p.a.out[(long long)tile * kGroupThreads + gtid] = prow[2 * gtid];
    }
    // this warp has read the power rows it needs: count off (the next tile's
    // transposition stores wait for all four warps, see above)
    __syncwarp();
    if (lane == 0) mbar_arrive(fbar);
    ++tiles_done;
  }
  if (MODE == kModeMel && p.a.max_slot) warp_max_to((double)vmax, p.a.max_slot);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (tid < 32) tmem_dealloc(tmem_slot, kTmemCols);
}

}  // namespace

static const size_t kSmemLimit = 232448;   // 227 KB opt-in maximum per CTA

static int span_bytes_needed(const FrameGeom& g) {
  return ((((kTile - 1) * g.hop + 2048) * 4) + 127) & ~127;
}
// The first 16384 bytes are not read: the window and the inter-pass twiddles live in
// tensor memory.  They stay reserved because this size decides, through
// stft2048p_supports, which geometries SMB_PATH_AUTO sends to this kernel; reclaiming
// them would move geometries between kernels.
static int tables_bytes_needed(int mel_w_floats, int mel_rounds) {
  return (16640 + mel_w_floats * 4 + kGroupWarps * mel_rounds * kF * (int)sizeof(PairMelItem) + 127) & ~127;
}
static size_t smem_needed(const FrameGeom& g, int mel_w_floats, int mel_rounds) {
  return (size_t)tables_bytes_needed(mel_w_floats, mel_rounds) +
         (size_t)kGroups * (span_bytes_needed(g) + kGroupWarps * kWarpBuf);
}

bool stft2048p_supports(const FrameGeom& g, int n_mels, int mel_w_floats, int mel_rounds) {
  if (g.fft != 2048 || g.hop < 2 || (g.hop & 1) != 0) return false;   // 8-byte sample loads per frame
  if (n_mels < 1 || n_mels > 32767 || mel_w_floats < 0 || (mel_w_floats & 3) != 0 ||
      mel_w_floats >= (1 << 24) || mel_rounds < 0)
    return false;
  if ((long long)n_mels * g.frames >= (1LL << 31)) return false;     // 32-bit row offsets inside a clip
  return smem_needed(g, mel_w_floats, mel_rounds) + 64 <= kSmemLimit;
}

cudaError_t launch_stft2048p(const Stft2048PairArgs& a, bool ceiling, int sm_count, cudaStream_t st) {
  if (a.batch == 0 || a.g.frames == 0) return cudaSuccess;
  const long long tiles_per_signal = (a.g.frames + kTile - 1) / kTile;
  if (tiles_per_signal * a.batch >= (1LL << 31)) {
    // tile indices are 32-bit inside the kernel: split the batch
    const long long half = a.batch / 2;
    Stft2048PairArgs lo = a, hi = a;
    lo.batch = half;
    hi.batch = a.batch - half;
    hi.x = a.x + half * a.g.n;
    if (!ceiling) hi.out = a.out + half * a.n_mels * a.g.frames;
    cudaError_t e1 = launch_stft2048p(lo, ceiling, sm_count, st);
    return e1 != cudaSuccess ? e1 : launch_stft2048p(hi, ceiling, sm_count, st);
  }
  Params p;
  p.a = a;
  if (ceiling) { p.a.mel_w_floats = 0; p.a.mel_rounds = 0; }
  p.bulk = stage::bulk_rule(a.x, a.g, kTile);
  p.span_bytes = span_bytes_needed(a.g);
  p.tables_bytes = tables_bytes_needed(p.a.mel_w_floats, p.a.mel_rounds);
  p.tiles_per_signal = (int)tiles_per_signal;
  p.total_tiles = (int)(tiles_per_signal * a.batch);
  const size_t smem = smem_needed(a.g, p.a.mel_w_floats, p.a.mel_rounds);
  if (smem + 64 > kSmemLimit) return cudaErrorInvalidConfiguration;
  const long long want = (p.total_tiles + kGroups - 1) / kGroups;
  const int grid = (int)(want < sm_count ? want : sm_count);
  cudaError_t e;
#define SMB_LAUNCH2048P_R(SQ, MODE, R)                                                         \
  e = cudaFuncSetAttribute(stft2048p_kernel<SQ, MODE, R>,                                      \
                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);            \
  if (e != cudaSuccess) return e;                                                              \
  stft2048p_kernel<SQ, MODE, R><<<grid, kGroups * kGroupThreads, smem, st>>>(p);
  // hop 512 (fft / 4) and 256 (fft / 8) share sample rows between the frames of a pair
#define SMB_LAUNCH2048P(SQ, MODE)                                                              \
  if (a.g.hop == 512) { SMB_LAUNCH2048P_R(SQ, MODE, 8) }                                       \
  else if (a.g.hop == 256) { SMB_LAUNCH2048P_R(SQ, MODE, 4) }                                  \
  else { SMB_LAUNCH2048P_R(SQ, MODE, 0) }
  if (ceiling) { SMB_LAUNCH2048P(true, kModeCeiling) }
  else if (a.power == 2.0f) { SMB_LAUNCH2048P(true, kModeMel) }
  else { SMB_LAUNCH2048P(false, kModeMel) }
#undef SMB_LAUNCH2048P
#undef SMB_LAUNCH2048P_R
  ++g_launch_count;
  return cudaGetLastError();
}

}  // namespace smb
