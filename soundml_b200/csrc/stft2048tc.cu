// Fused STFT kernel for fft_size = 2048, float32 audio, with the two 32-point
// DFT passes on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
//   framing + boundary extension + window -> real FFT 2048 -> |X|^p
//   -> (optionally) sparse mel projection -> [batch, bins | n_mels, frames]
//
// Same contract as stft2048.cu (Stft.analyse / magnitude_pow / Mel.apply,
// stft.ml:356-364, 670-674; mel.ml:202-231); what changes is where the
// butterflies run.  Real FFT 2048 = complex FFT 1024 on z[n] = x[2n] + i x[2n+1],
// n = 32 n1 + n2, k = k1 + 32 k2:
//
//   pass 1   Y[n2][k1]  = sum_n1 z[32 n1 + n2] W32^(n1 k1)
//   twiddle  Y'[n2][k1] = Y[n2][k1] W1024^(k1 n2)
//   pass 2   Z[k1+32k2] = sum_n2 Y'[n2][k1] W32^(n2 k2)
//
// Each pass is a real matrix product  D[128 x 64] = A[128 x 64] . F[64 x 64]:
// the 128 rows are (frame, n2) -- resp. (frame, k1) -- of a tile of 4 frames, the
// 64 columns the interleaved (re, im) of the 32 complex points, F the 32-point DFT
// written out in real arithmetic (the same matrix for both passes).  kind::f16
// operands with fp32 accumulation in TMEM; float32 accuracy is kept by operand
// splitting, a = a_hi + a_lo and F = F_hi + F_lo in fp16 (11 + 11 significant
// bits), D = a_hi F_hi + a_lo F_hi + a_hi F_lo (the dropped term is 2^-22).
// fp16 has 5 exponent bits: the tile's samples are scaled by a power of two
// chosen from their largest magnitude (|a| < 512, so |Y| < 2^15), undone in the
// real split; products and sums are exact powers of two away from the unscaled
// ones.
//
//   * One persistent CTA per SM, groups of 4 warps.  A group owns a tile of 4
//     consecutive frames of one signal: it stages the tile's 3 hop + 2048 samples
//     (cp.async, one tile ahead), builds A1 = window x samples (hi, lo) in the
//     canonical K-major SWIZZLE_128B layout, one thread issues the 12 MMAs of
//     pass 1 and commits to the group's mbarrier, every thread reads its row of
//     D1 back (tcgen05.ld; thread = (frame, n2)), applies the twiddle, splits and
//     scatters into A2 (rows (frame, k1)), 12 MMAs again, reads D2 (thread =
//     (frame, k1), registers = k2) and finishes like stft2048.cu: real split by
//     warp shuffles, |X|^p into the frame's row, band mel, write-out.  The mel
//     step is laid out for 4-frame tiles: every filter's band is cut into pieces
//     of at most 4 float4 steps, a lane carries one piece for all four frames
//     (one weight load feeds 16 FMAs), partial sums are added up at write-out.
//   * The groups of a CTA run out of phase, so one group's MMAs overlap the
//     CUDA-core phases of the others; operand buffers, the power rows and the
//     accumulators are private to a group (TMEM columns 128 g .. 128 g + 127).
#include "fft32.cuh"
#include "kernels.h"
#include "stft_stage.cuh"

#include <cstdint>
#include <cuda_fp16.h>

namespace smb {

namespace {

using fft32impl::pk_add;
using fft32impl::pk_mul;
using fft32impl::pk_sub;

constexpr int kFft = 2048;
constexpr int kHalf = 1024;
constexpr int kTile = kTcTile;            // frames per tile = 128 MMA rows
constexpr int kGroupThreads = 32 * kTile;
static_assert(kTile == 4, "one warp per frame, 128 TMEM lanes per tile");
constexpr int kRowReal = 1032;            // floats per power row (mel partial sums follow it)
constexpr int kRowComplex = 2056;         // floats per complex row, = 8 mod 32
constexpr int kABytes = 128 * 128;        // one split of a pass's A operand
constexpr int kBBytes = 64 * 128;         // one split of F
constexpr int kMaxGroups = 4;

// tcgen05.mma, K-major SWIZZLE_128B operands (8-row groups 1024 B apart), the descriptors given by their low words (start address field) over the
// common high word: the K-steps of a batch only move the start address
__device__ __forceinline__ void umma_f16_lo(uint32_t tmem_d, uint32_t alo, uint32_t blo, uint32_t idesc,
                                            bool accumulate) {
  constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);   // SBO, version, SWIZZLE_128B
  if (accumulate)
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "setp.eq.b32 p, 0, 0;\n\t"
        "mov.b64 da, {%1, %3};\n\tmov.b64 db, {%2, %3};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}"
        ::"r"(tmem_d), "r"(alo), "r"(blo), "r"(kDescHi), "r"(idesc)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, 0, 0;\n\t"
        "mov.b64 da, {%1, %3};\n\tmov.b64 db, {%2, %3};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}"
        ::"r"(tmem_d), "r"(alo), "r"(blo), "r"(kDescHi), "r"(idesc)
        : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c,
                                             uint32_t d) {
  // no "memory" clobber: these bytes are only read by the tensor core, after the
  // proxy fence + barrier that follow; ordinary loads may move across the store
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d));
}
__device__ __forceinline__ void st_shared_b32(uint32_t addr, uint32_t a) {
  asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(a));
}
// fp16 pair (lo half = a, hi half = b), round to nearest
__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
// the two halves of an fp16 pair back in float32
__device__ __forceinline__ float2 unpack_half2(uint32_t h) {
  return __half22float2(*reinterpret_cast<const __half2*>(&h));
}

struct Params {
  Stft2048Args a;
  int span_cap;              // floats reserved per group for samples (multiple of 4)
  int region_bytes;          // operand / row region per group (multiple of 1024)
  int row_stride;            // floats per output row of a frame
  long long tiles_per_signal, total_tiles;
};

// Tile geometry shared by the staging call and the consumer.
struct TileRef {
  int b, p0;                 // signal, first frame
};
// An interior tile whose source run is 16-byte aligned is brought in by one bulk
// copy (TMA); everything else goes through cp.async and the boundary rule.
__device__ __forceinline__ bool tile_is_bulk(const Params& p, TileRef t) {
  const FrameGeom& g = p.a.g;
  const int nf = (int)min((long long)kTile, g.frames - t.p0);
  const int span = (nf - 1) * g.hop + kFft;
  const long long s0 = (long long)t.p0 * g.hop - g.left;
  const size_t addr = reinterpret_cast<size_t>(p.a.x + (long long)t.b * g.n + s0);
  return s0 >= 0 && s0 + span <= g.n && (addr & 15) == 0 && (span & 3) == 0;
}
// Brings one tile's samples (padded stream positions p0*hop .. + span) into the
// group's sample buffer; the tail up to span_cap is zeroed (the scale scan reads
// the whole buffer).  Run by ONE warp of the group.  Bulk tiles: lane 0 issues the
// copy, which lands on `bar`.  Otherwise the rules of stft2048.cu::stage_tile
// apply (cp.async for the real samples, the reference's boundary rule
// stft.ml:300-338 for the border) and this warp waits for its cp.async group
// before the group's barrier.
__device__ __forceinline__ void stage_tile(const Params& p, TileRef t, bool bulk, float* sSamples,
                                           int lane, uint32_t bar) {
  const FrameGeom& g = p.a.g;
  const int nf = (int)min((long long)kTile, g.frames - t.p0);
  const int span = (nf - 1) * g.hop + kFft;
  const long long q0 = (long long)t.p0 * g.hop;
  const long long s0 = q0 - g.left;
  const float* xs = p.a.x + (long long)t.b * g.n;
  const float* src = xs + s0;                       // src + i is valid for i in [lo, hi)
  const unsigned base = (unsigned)__cvta_generic_to_shared(sSamples);
  for (int i = span + lane; i < p.span_cap; i += 32) sSamples[i] = 0.0f;
  if (bulk) {
    if (lane == 0) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_expect_tx(bar, 4u * (uint32_t)span);
      bulk_g2s(base, src, 4u * (uint32_t)span, bar);
    }
    return;
  }
  const int lo = (int)max(0LL, min((long long)span, -s0));
  const int hi = (int)max((long long)lo, min((long long)span, g.n - s0));
  for (int i = lane; i < lo; i += 32) {
    const long long s = stage::src_index(g, q0 + i);
    sSamples[i] = s >= 0 ? __ldg(xs + s) : (float)g.pad_value;
  }
  for (int i = hi + lane; i < span; i += 32) {
    const long long s = stage::src_index(g, q0 + i);
    sSamples[i] = s >= 0 ? __ldg(xs + s) : (float)g.pad_value;
  }
  stage::copy_real_samples<32>(base, src, lo, hi, lane);
}

// STEP1: bin_step == 1 (fft 2048 proper): every bin is kept.
template <int OUT, bool SQUARE, int kGroups, bool STEP1>
__global__ void __launch_bounds__(kGroups * kGroupThreads, 1)
stft2048tc_kernel(const Params p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[2 * kMaxGroups];
  __shared__ uint32_t tmem_base_slot;
  __shared__ __align__(16) float sMax[kMaxGroups * kTile];

  // SWIZZLE_128B operands need 1024-byte aligned tiles: work with shared-window
  // addresses and keep every pointer derived from smem_raw by an integer offset.
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t pad = (1024u - (raw_addr & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;
  const uint32_t smem_addr = raw_addr + pad;
  // [F hi | F lo] [regions x groups] [tw_pass] [tw_post] [samples x groups] [mel vals] [pieces] [pcnt]
  const uint32_t regions_off = 2 * kBBytes;
  const uint32_t tables_off = regions_off + kGroups * p.region_bytes;
  float2* sTwPass = reinterpret_cast<float2*>(smem + tables_off);           // [16][32][2] W_1024^(k1 n2)
  float2* sTwPost = sTwPass + 1024;                                          // [16][32] W_2048^(l + 32 k2)
  float* sSamplesAll = reinterpret_cast<float*>(sTwPost + 512);
  float* sMelVals = sSamplesAll + kGroups * p.span_cap;
  const int nnz_pad = (p.a.nnz + 3) & ~3;
  MelPiece* sPieces = reinterpret_cast<MelPiece*>(sMelVals + nnz_pad);       // [warps][rounds][32]
  unsigned char* sPcnt = reinterpret_cast<unsigned char*>(sPieces + kTile * p.a.mel_rounds * 32);

  const int tid = threadIdx.x;
  const int group = tid / kGroupThreads;
  const int gtid = tid % kGroupThreads;
  const int warp = gtid >> 5;
  const int lane = tid & 31;

  {
    const uint4* src = reinterpret_cast<const uint4*>(p.a.dft_images);
    uint4* dst = reinterpret_cast<uint4*>(smem);
    for (int i = tid; i < 2 * kBBytes / 16; i += blockDim.x) dst[i] = src[i];
  }
  for (int i = tid; i < 1024; i += blockDim.x) {
    const int l = i & 31, k1 = i >> 5;
    sTwPass[(((k1 >> 1) * 32 + l) << 1) + (k1 & 1)] = p.a.tw_pass[i];
  }
  for (int i = tid; i < 512; i += blockDim.x) sTwPost[i] = p.a.tw_post[i];
  if (OUT == kFastMel) {
    for (int i = tid; i < p.a.nnz; i += blockDim.x) sMelVals[i] = p.a.vals[i];
    for (int i = tid; i < kTile * p.a.mel_rounds * 32; i += blockDim.x) sPieces[i] = p.a.mel_pieces[i];
    for (int i = tid; i < p.a.n_mels; i += blockDim.x) sPcnt[i] = p.a.mel_pcnt[i];
  }
  if (tid == 0) {
    for (int gI = 0; gI < 2 * kMaxGroups; ++gI) mbar_init(smem_u32(&bars[gI]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  constexpr int kTmemCols = kGroups > 2 ? 512 : 256;
  if (tid < 32) tmem_alloc(&tmem_base_slot, kTmemCols);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // F images -> async proxy
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tmem_base_slot;
  const uint32_t acc1 = tmem + 128 * group, acc2 = acc1 + 64;
  const uint32_t lane_base = ((uint32_t)(warp * 32)) << 16;
  const uint32_t bar = smem_u32(&bars[group]);               // MMAs of this group done
  const uint32_t sbar = smem_u32(&bars[kMaxGroups + group]);  // bulk copy of the samples landed
  uint32_t phase = 0, sphase = 0;

  const FrameGeom g = p.a.g;
  const int bin_shift = STEP1 ? 0 : 31 - __clz(p.a.bin_step), bin_mask = STEP1 ? 0 : p.a.bin_step - 1;
  const int slot = blockIdx.x * kGroups + group;
  const int stride = gridDim.x * kGroups;
  const int total_tiles = (int)p.total_tiles, tiles_per_signal = (int)p.tiles_per_signal;
  // tile -> (signal, first frame) is kept incrementally: one division here only
  const int stride_b = stride / tiles_per_signal, stride_t = stride - stride_b * tiles_per_signal;
  TileRef cur;
  cur.b = slot / tiles_per_signal;
  int cur_t = slot - cur.b * tiles_per_signal;
  cur.p0 = cur_t * kTile;

  float* sSamples = sSamplesAll + group * p.span_cap;
  const uint32_t region_addr = smem_addr + regions_off + group * p.region_bytes;
  float* sRows = reinterpret_cast<float*>(smem + regions_off + group * p.region_bytes);
  const uint32_t a_hi = region_addr, a_lo = region_addr + kABytes;
  const uint32_t f_hi = smem_addr, f_lo = smem_addr + kBBytes;
  // low words of the operand descriptors (start address in 16-byte units, LBO = 1);
  // a K-step of 16 halves moves the start by 32 bytes = 2 units
  const uint32_t dl_a_hi = ((a_hi >> 4) & 0x3FFF) | (1u << 16), dl_a_lo = ((a_lo >> 4) & 0x3FFF) | (1u << 16);
  const uint32_t dl_f_hi = ((f_hi >> 4) & 0x3FFF) | (1u << 16), dl_f_lo = ((f_lo >> 4) & 0x3FFF) | (1u << 16);
  // instruction descriptor: D f32, A/B f16, both K-major, N = 64, M = 128
  constexpr uint32_t kIdesc = (1u << 4) | ((64u >> 3) << 17) | ((128u >> 4) << 24);

  // This thread's window values never change: pass-1 operand element (n1, c) of
  // row n2 = lane is x[64 n1 + 2 n2 + c]; warp w builds n1 = 8 w .. 8 w + 7 for
  // all frames of the tile.  The 1/2 of the real split rides on the window.
  float2 wreg[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int j = 64 * (8 * warp + i) + 2 * lane;
    wreg[i] = make_float2(0.5f * __ldg(p.a.window + j), 0.5f * __ldg(p.a.window + j + 1));
  }
  // pass 2's operand: element (n2 = lane, c) of row k1 sits in 16-byte chunk
  // (lane / 4) ^ (k1 mod 8), at byte 4 (lane mod 4)
  const uint32_t lane_chunk = (((uint32_t)lane >> 2) << 4) | (((uint32_t)lane & 3u) << 2);

  float* row = sRows + warp * p.row_stride;

  bool bulk = false;
  if (slot < total_tiles) {
    bulk = tile_is_bulk(p, cur);
    if (warp == 0) stage_tile(p, cur, bulk, sSamples, lane, sbar);
  }
  for (int tile = slot; tile < total_tiles; tile += stride) {
    const int b = cur.b, p0 = cur.p0;
    const int nf = (int)min((long long)kTile, g.frames - p0);
    TileRef nxt;                                    // the tile after this one
    {
      int t = cur_t + stride_t;
      nxt.b = cur.b + stride_b;
      if (t >= tiles_per_signal) { t -= tiles_per_signal; ++nxt.b; }
      cur_t = t;
      nxt.p0 = t * kTile;
    }
    cur = nxt;

    if (bulk) {
      mbar_wait(sbar, sphase & 1);
      ++sphase;
    } else if (warp == 0) {
      asm volatile("cp.async.wait_all;" ::: "memory");
    }
    named_sync(group + 1, kGroupThreads);

    // ---- scale: largest sample magnitude of the tile -> power of two
    float scale, unscale;
    {
      float m = 0.0f;
      const float4* s4 = reinterpret_cast<const float4*>(sSamples);
      for (int i = gtid; i < (p.span_cap >> 2); i += kGroupThreads) {
        const float4 v = s4[i];
        m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
      }
      // non-negative floats order like their bit patterns: one REDUX per warp
      m = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(m)));
      if (lane == 0) sMax[group * kTile + warp] = m;
      named_sync(group + 1, kGroupThreads);
      const float4 mm = *reinterpret_cast<const float4*>(sMax + group * kTile);
      m = fmaxf(fmaxf(mm.x, mm.y), fmaxf(mm.z, mm.w));
      // m in [2^e, 2^(e+1))  ->  scale = 2^(9 - e): |x| scale < 1024, window/2 <= 1/2
      int sb = 263 - (int)(__float_as_uint(m) >> 23);
      sb = max(1, min(254, sb));
      scale = __uint_as_float((uint32_t)sb << 23);
      unscale = __uint_as_float((uint32_t)(254 - sb) << 23);
    }

    // ---- pass-1 operand: rows (f, n2 = lane), this warp's 16 K-columns
    {
      float2 ws[8];
      const float2 sc2 = make_float2(scale, scale);
#pragma unroll
      for (int i = 0; i < 8; ++i) ws[i] = pk_mul(wreg[i], sc2);
      const uint32_t sw = (uint32_t)lane & 7u;
      const uint32_t c0 = (((uint32_t)(2 * warp) ^ sw) << 4), c1 = (((uint32_t)(2 * warp + 1) ^ sw) << 4);
      const bool even = (g.hop & 1) == 0;
      const float* fs0 = sSamples + 64 * (8 * warp) + 2 * lane;
      // software pipeline: the samples of frame f + 1 are requested before frame f
      // is converted, so the shared-memory latency hides under the arithmetic
      auto load_frame = [&](int f, float2 (&v)[8]) {
        const float* fs = fs0 + f * g.hop;
        if (even || (f & 1) == 0) {
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = *reinterpret_cast<const float2*>(fs + 64 * i);
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = make_float2(fs[64 * i], fs[64 * i + 1]);
        }
      };
      auto convert_frame = [&](int f, const float2 (&v)[8]) {
        uint32_t hw[8], lw[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float2 u = pk_mul(v[i], ws[i]);
          hw[i] = pack_half2(u.x, u.y);
          const float2 l = pk_sub(u, unpack_half2(hw[i]));
          lw[i] = pack_half2(l.x, l.y);
        }
        const uint32_t rowoff = (uint32_t)(32 * f + lane) * 128u;
        st_shared_v4(a_hi + rowoff + c0, hw[0], hw[1], hw[2], hw[3]);
        st_shared_v4(a_hi + rowoff + c1, hw[4], hw[5], hw[6], hw[7]);
        st_shared_v4(a_lo + rowoff + c0, lw[0], lw[1], lw[2], lw[3]);
        st_shared_v4(a_lo + rowoff + c1, lw[4], lw[5], lw[6], lw[7]);
      };
      float2 va[8], vb[8];
      load_frame(0, va);
      if (nf > 1) load_frame(1, vb);
      convert_frame(0, va);
      if (nf > 2) load_frame(2, va);
      if (nf > 1) convert_frame(1, vb);
      if (nf > 3) load_frame(3, vb);
      if (nf > 2) convert_frame(2, va);
      if (nf > 3) convert_frame(3, vb);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    named_sync(group + 1, kGroupThreads);

    if (gtid == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        umma_f16_lo(acc1, dl_a_hi + 2 * ks, dl_f_hi + 2 * ks, kIdesc, ks > 0);
        umma_f16_lo(acc1, dl_a_lo + 2 * ks, dl_f_hi + 2 * ks, kIdesc, true);
        umma_f16_lo(acc1, dl_a_hi + 2 * ks, dl_f_lo + 2 * ks, kIdesc, true);
      }
      umma_commit(bar);
    }
    // ---- the sample buffer is free: fetch the next tile under the rest of this one
    const bool more = tile + stride < total_tiles;
    if (more) {
      bulk = tile_is_bulk(p, nxt);
      if (warp == 1) stage_tile(p, nxt, bulk, sSamples, lane, sbar);
    }

    mbar_wait(bar, phase & 1);
    ++phase;
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // ---- D1 row (f = warp, n2 = lane): twiddle, split, scatter into pass 2's
    // operand, rows (f, k1), K-column (n2, c)
    {
      const float4* t4 = reinterpret_cast<const float4*>(sTwPass) + lane;
      const uint32_t base_hi = a_hi + (uint32_t)(32 * warp) * 128u + lane_chunk;
      // chunk q = columns 16 q .. 16 q + 15 = k1 8 q .. 8 q + 7, four float4 of twiddles.
      // TMEM loads and twiddle loads run one chunk ahead of the arithmetic.
      auto load_tw = [&](int q, float4 (&t)[4]) {
#pragma unroll
        for (int j = 0; j < 4; ++j) t[j] = t4[(4 * q + j) * 32];
      };
      auto convert_chunk = [&](int q, const uint32_t (&d)[16], const float4 (&t)[4]) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int k1 = 8 * q + 2 * j;             // (k1 mod 8) = 2 j
          const float yr0 = __uint_as_float(d[4 * j]), yi0 = __uint_as_float(d[4 * j + 1]);
          const float yr1 = __uint_as_float(d[4 * j + 2]), yi1 = __uint_as_float(d[4 * j + 3]);
          const float2 z0 = make_float2(yr0 * t[j].x - yi0 * t[j].y, yr0 * t[j].y + yi0 * t[j].x);
          const float2 z1 = make_float2(yr1 * t[j].z - yi1 * t[j].w, yr1 * t[j].w + yi1 * t[j].z);
          const uint32_t h0 = pack_half2(z0.x, z0.y), h1 = pack_half2(z1.x, z1.y);
          const float2 l0 = pk_sub(z0, unpack_half2(h0)), l1 = pk_sub(z1, unpack_half2(h1));
          const uint32_t o0 = (base_hi ^ ((uint32_t)(2 * j) << 4)) + (uint32_t)k1 * 128u;
          const uint32_t o1 = (base_hi ^ ((uint32_t)(2 * j + 1) << 4)) + (uint32_t)(k1 + 1) * 128u;
          st_shared_b32(o0, h0);
          st_shared_b32(o0 + kABytes, pack_half2(l0.x, l0.y));
          st_shared_b32(o1, h1);
          st_shared_b32(o1 + kABytes, pack_half2(l1.x, l1.y));
        }
      };
      uint32_t da[16], db[16];
      float4 ta[4], tb[4];
      tmem_ld16(acc1 + lane_base, da);
      tmem_ld16(acc1 + lane_base + 16, db);
      load_tw(0, ta);
      tmem_ld_wait();
      load_tw(1, tb);
      convert_chunk(0, da, ta);
      tmem_ld16(acc1 + lane_base + 32, da);
      load_tw(2, ta);
      convert_chunk(1, db, tb);
      tmem_ld16(acc1 + lane_base + 48, db);
      tmem_ld_wait();
      load_tw(3, tb);
      convert_chunk(2, da, ta);
      convert_chunk(3, db, tb);
    }
    if (more && warp == 1 && !bulk) asm volatile("cp.async.wait_all;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    named_sync(group + 1, kGroupThreads);

    if (gtid == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        umma_f16_lo(acc2, dl_a_hi + 2 * ks, dl_f_hi + 2 * ks, kIdesc, ks > 0);
        umma_f16_lo(acc2, dl_a_lo + 2 * ks, dl_f_hi + 2 * ks, kIdesc, true);
        umma_f16_lo(acc2, dl_a_hi + 2 * ks, dl_f_lo + 2 * ks, kIdesc, true);
      }
      umma_commit(bar);
    }
    mbar_wait(bar, phase & 1);
    ++phase;
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // ---- D2 row (f = warp, k1 = lane): a[k2] = s Z'[k1 + 32 k2]; real split as in
    // stft2048.cu.  For the complex spectrum the tile's scale is undone here (it
    // rides on S and on the twiddle); |X|^p is taken on the scaled values (no
    // underflow of the squares for faint signals) and the scale comes off as one
    // multiply per value at write-out (the mel projection is linear).
    const bool late_unscale = OUT != kFastComplex;
    {
      float2 a[32];
      {
        uint32_t d0[32], d1[32];
        tmem_ld32(acc2 + lane_base, d0);
        tmem_ld32(acc2 + lane_base + 32, d1);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          a[i] = make_float2(__uint_as_float(d0[2 * i]), __uint_as_float(d0[2 * i + 1]));
          a[16 + i] = make_float2(__uint_as_float(d1[2 * i]), __uint_as_float(d1[2 * i + 1]));
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      if (warp < nf) {
        const int partner = (32 - lane) & 31;
        const float us = late_unscale ? 1.0f : unscale;
        const float2 us2 = make_float2(us, us);
        float2 r[16];
#pragma unroll
        for (int k2 = 0; k2 < 16; ++k2) {
          // lanes != 0 need the partner's register 31-k2; lane 0 pairs with itself
          // through register (32-k2) mod 32.  The conjugate is taken on the way.
          const float2 own = a[31 - k2];
          const float2 alt = a[(32 - k2) & 31];
          const float sx = lane == 0 ? alt.x : own.x;
          const float sy = lane == 0 ? alt.y : own.y;
          r[k2].x = __shfl_sync(0xffffffffu, sx, partner);
          r[k2].y = -__shfl_sync(0xffffffffu, sy, partner);
        }
        float2* rowc = reinterpret_cast<float2*>(row);
        // results first (the twiddle loads can all run ahead: no store in between),
        // stores after: xk -> a[k2], conj X[N-k] -> r[k2] (or the two powers in a[k2])
#pragma unroll
        for (int k2 = 0; k2 < 16; ++k2) {
          //   S = Z'[k] + conj Z'[N-k],  D = Z'[k] - conj Z'[N-k],  W = W2048^k
          //   X[k] = S + W (-i D),   X[N-k] = conj(S - W (-i D))
          float2 w = sTwPost[k2 * 32 + lane];
          if (!late_unscale) w = pk_mul(w, us2);
          float2 S = pk_add(a[k2], r[k2]);
          const float2 D = pk_sub(a[k2], r[k2]);
          if (!late_unscale) S = pk_mul(S, us2);
          const float2 T = make_float2(w.x * D.y + w.y * D.x, w.y * D.y - w.x * D.x);
          const float2 xk = pk_add(S, T);
          const float2 xm = pk_sub(S, T);                     // conj of X[N-k]
          if (OUT == kFastComplex) {
            a[k2] = xk;
            r[k2] = make_float2(xm.x, -xm.y);
          } else {
            float pk = xk.x * xk.x + xk.y * xk.y;
            float pn = xm.x * xm.x + xm.y * xm.y;
            if (!SQUARE) {
              if (p.a.power == 1.0f) { pk = sqrtf(pk); pn = sqrtf(pn); }
              else { pk = powf(sqrtf(pk), p.a.power); pn = powf(sqrtf(pn), p.a.power); }
            }
            a[k2] = make_float2(pk, pn);
          }
        }
#pragma unroll
        for (int k2 = 0; k2 < 16; ++k2) {
          const int k = lane + 32 * k2, nk = kHalf - k;
          const bool keep_k = STEP1 || (k & bin_mask) == 0, keep_n = STEP1 || (nk & bin_mask) == 0;
          if (OUT == kFastComplex) {
            if (keep_k) rowc[k >> bin_shift] = a[k2];
            if (keep_n) rowc[nk >> bin_shift] = r[k2];
          } else {
            if (keep_k) row[k >> bin_shift] = a[k2].x;
            if (keep_n) row[nk >> bin_shift] = a[k2].y;
          }
        }
        if (lane == 0) {                            // k = 512 pairs with itself
          const float2 xm = make_float2(2.0f * a[16].x * us, -2.0f * a[16].y * us);
          if (OUT == kFastComplex) rowc[512 >> bin_shift] = xm;
          else {
            float pm = xm.x * xm.x + xm.y * xm.y;
            if (!SQUARE) pm = p.a.power == 1.0f ? sqrtf(pm) : powf(sqrtf(pm), p.a.power);
            row[512 >> bin_shift] = pm;
            const int bins = (kHalf >> bin_shift) + 1;
            row[bins] = row[bins + 1] = row[bins + 2] = 0.0f;   // float4 padding read by the mel bands
          }
        }
      }
    }
    named_sync(group + 1, kGroupThreads);

    if (OUT == kFastMel) {
      // ---- mel projection over the tile's power rows.  A lane carries one piece
      // (at most 4 float4 steps of one filter's band) for the four frames: the
      // weight load is one contiguous run per warp, every power value is read
      // once per filter it feeds; a warp's pieces in a round have one step count.
      const MelPiece* mine = sPieces + warp * p.a.mel_rounds * 32 + lane;
      float* part = sRows + kRowReal;
      for (int r = 0; r < p.a.mel_rounds; ++r) {
        const MelPiece q = mine[r * 32];
        const int steps = (int)((unsigned)q.off >> 24);
        const float4* wq = reinterpret_cast<const float4*>(sMelVals + (q.off & 0xFFFFFF));
        const float4* v0 = reinterpret_cast<const float4*>(sRows + q.lo);
        const float4* v1 = reinterpret_cast<const float4*>(sRows + p.row_stride + q.lo);
        const float4* v2 = reinterpret_cast<const float4*>(sRows + 2 * p.row_stride + q.lo);
        const float4* v3 = reinterpret_cast<const float4*>(sRows + 3 * p.row_stride + q.lo);
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        // the step count is uniform over the warp; two steps at a time keeps ten
        // 16-byte loads in flight ahead of the 32 FMAs that consume them
        int i = 0;
        for (; i + 2 <= steps; i += 2) {
          const float4 ww = wq[32 * i], wz = wq[32 * i + 32];
          const float4 x0 = v0[i], x1 = v1[i], x2 = v2[i], x3 = v3[i];
          const float4 y0 = v0[i + 1], y1 = v1[i + 1], y2 = v2[i + 1], y3 = v3[i + 1];
          a0 = fmaf(ww.x, x0.x, a0); a1 = fmaf(ww.x, x1.x, a1);
          a2 = fmaf(ww.x, x2.x, a2); a3 = fmaf(ww.x, x3.x, a3);
          a0 = fmaf(ww.y, x0.y, a0); a1 = fmaf(ww.y, x1.y, a1);
          a2 = fmaf(ww.y, x2.y, a2); a3 = fmaf(ww.y, x3.y, a3);
          a0 = fmaf(ww.z, x0.z, a0); a1 = fmaf(ww.z, x1.z, a1);
          a2 = fmaf(ww.z, x2.z, a2); a3 = fmaf(ww.z, x3.z, a3);
          a0 = fmaf(ww.w, x0.w, a0); a1 = fmaf(ww.w, x1.w, a1);
          a2 = fmaf(ww.w, x2.w, a2); a3 = fmaf(ww.w, x3.w, a3);
          a0 = fmaf(wz.x, y0.x, a0); a1 = fmaf(wz.x, y1.x, a1);
          a2 = fmaf(wz.x, y2.x, a2); a3 = fmaf(wz.x, y3.x, a3);
          a0 = fmaf(wz.y, y0.y, a0); a1 = fmaf(wz.y, y1.y, a1);
          a2 = fmaf(wz.y, y2.y, a2); a3 = fmaf(wz.y, y3.y, a3);
          a0 = fmaf(wz.z, y0.z, a0); a1 = fmaf(wz.z, y1.z, a1);
          a2 = fmaf(wz.z, y2.z, a2); a3 = fmaf(wz.z, y3.z, a3);
          a0 = fmaf(wz.w, y0.w, a0); a1 = fmaf(wz.w, y1.w, a1);
          a2 = fmaf(wz.w, y2.w, a2); a3 = fmaf(wz.w, y3.w, a3);
        }
        if (i < steps) {
          const float4 ww = wq[32 * i];
          const float4 x0 = v0[i], x1 = v1[i], x2 = v2[i], x3 = v3[i];
          a0 = fmaf(ww.x, x0.x, a0); a1 = fmaf(ww.x, x1.x, a1);
          a2 = fmaf(ww.x, x2.x, a2); a3 = fmaf(ww.x, x3.x, a3);
          a0 = fmaf(ww.y, x0.y, a0); a1 = fmaf(ww.y, x1.y, a1);
          a2 = fmaf(ww.y, x2.y, a2); a3 = fmaf(ww.y, x3.y, a3);
          a0 = fmaf(ww.z, x0.z, a0); a1 = fmaf(ww.z, x1.z, a1);
          a2 = fmaf(ww.z, x2.z, a2); a3 = fmaf(ww.z, x3.z, a3);
          a0 = fmaf(ww.w, x0.w, a0); a1 = fmaf(ww.w, x1.w, a1);
          a2 = fmaf(ww.w, x2.w, a2); a3 = fmaf(ww.w, x3.w, a3);
        }
        part[q.pid] = a0;
        part[p.row_stride + q.pid] = a1;
        part[2 * p.row_stride + q.pid] = a2;
        part[3 * p.row_stride + q.pid] = a3;
      }
      named_sync(group + 1, kGroupThreads);
    }

    // ---- write the tile along the frame axis: [batch, rows, frames]
    {
      const int f = gtid & (kTile - 1), r0 = gtid / kTile;
      // |s X|^p = s^p |X|^p
      const float post = SQUARE ? unscale * unscale
                                : (p.a.power == 1.0f ? unscale : powf(unscale, p.a.power));
      if (f < nf) {
        if (OUT == kFastMel) {
          float* ob = p.a.out + ((long long)b * p.a.n_mels + r0) * g.frames + p0 + f;
          const long long step = (long long)(kGroupThreads / kTile) * g.frames;
          const float* src = sRows + f * p.row_stride + kRowReal;
          // the j-th partial sum of filter m sits at j * mpad + m (up to four; slots a
          // filter does not use hold stale bits and are masked out, never added)
          const int mpad = p.a.mel_mpad;
          for (int m = r0; m < p.a.n_mels; m += kGroupThreads / kTile, ob += step) {
            const int cnt = sPcnt[m];
            const float s0 = src[m], s1 = src[mpad + m], s2 = src[2 * mpad + m], s3 = src[3 * mpad + m];
            *ob = ((s0 + (cnt > 1 ? s1 : 0.0f)) + ((cnt > 2 ? s2 : 0.0f) + (cnt > 3 ? s3 : 0.0f))) * post;
          }
        } else if (OUT == kFastPower) {
          const int out_bins = kHalf / p.a.bin_step + 1;
          float* ob = p.a.out + ((long long)b * out_bins + r0) * g.frames + p0 + f;
          const long long step = (long long)(kGroupThreads / kTile) * g.frames;
          const float* src = sRows + f * p.row_stride;
          for (int r = r0; r < out_bins; r += kGroupThreads / kTile, ob += step)
            *ob = src[r] * post;
        } else {
          const int out_bins = kHalf / p.a.bin_step + 1;
          float2* ob = reinterpret_cast<float2*>(p.a.out) + ((long long)b * out_bins + r0) * g.frames +
                       p0 + f;
          const long long step = (long long)(kGroupThreads / kTile) * g.frames;
          const float2* src = reinterpret_cast<const float2*>(sRows + f * p.row_stride);
          for (int r = r0; r < out_bins; r += kGroupThreads / kTile, ob += step)
            *ob = src[r];
        }
      }
    }
    named_sync(group + 1, kGroupThreads);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (tid < 32) tmem_dealloc(tmem, kTmemCols);
}

}  // namespace

static const size_t kSmemLimit = 232448;   // 227 KB opt-in maximum per CTA

static int span_needed(const FrameGeom& g) {
  return (((kTile - 1) * g.hop + kFft) + 3) & ~3;
}
static int row_floats(int out_kind, int mpad) {
  if (out_kind == kFastComplex) return kRowComplex;
  if (out_kind == kFastPower) return kRowReal;
  return kRowReal + ((4 * mpad + 1 + 3) & ~3);          // partial sums [4][mpad] + one scratch slot
}
static int region_needed(int out_kind, int mpad) {
  const int rows = kTile * row_floats(out_kind, mpad) * 4;
  const int need = rows > 2 * kABytes ? rows : 2 * kABytes;
  return (need + 1023) & ~1023;
}
static size_t smem_layout(int out_kind, int n_mels, int nnz, int mel_rounds, int mpad, int span_cap,
                          int groups) {
  const int nnz_pad = (nnz + 3) & ~3;
  size_t bytes = 1024;                                             // alignment slack
  bytes += 2 * kBBytes;
  bytes += (size_t)groups * region_needed(out_kind, mpad);
  bytes += (size_t)(2 * 1024 + 2 * 512) * 4;                       // tw_pass, tw_post
  bytes += (size_t)groups * span_cap * 4;
  bytes += (size_t)nnz_pad * 4;
  bytes += (size_t)kTile * mel_rounds * 32 * sizeof(MelPiece);
  bytes += (size_t)((n_mels + 3) & ~3);
  return bytes;
}

bool stft2048tc_supports(const FrameGeom& g, int out_kind, int n_mels, int nnz, int mel_rounds,
                         int mpad) {
  if (g.fft != kFft || g.hop < 1 || g.hop > 4096) return false;
  if (out_kind == kFastMel && (n_mels < 1 || n_mels > 255 || nnz >= (1 << 24) || mpad > 256))
    return false;
  const bool mel = out_kind == kFastMel;
  return smem_layout(out_kind, mel ? n_mels : 0, mel ? nnz : 0, mel ? mel_rounds : 0,
                     mel ? mpad : 0, span_needed(g), 2) <= kSmemLimit;
}

cudaError_t launch_stft2048tc(const Stft2048Args& a, int out_kind, int sm_count, cudaStream_t st) {
  if (a.batch == 0 || a.g.frames == 0) return cudaSuccess;
  if ((a.g.frames + kTile - 1) / kTile * a.batch >= (1LL << 31)) {
    const long long half = a.batch / 2;
    Stft2048Args lo = a, hi = a;
    lo.batch = half;
    hi.batch = a.batch - half;
    hi.x = a.x + half * a.g.n;
    const long long rows = out_kind == kFastMel ? a.n_mels : kHalf / a.bin_step + 1;
    hi.out = a.out + half * rows * a.g.frames * (out_kind == kFastComplex ? 2 : 1);
    cudaError_t e1 = launch_stft2048tc(lo, out_kind, sm_count, st);
    return e1 != cudaSuccess ? e1 : launch_stft2048tc(hi, out_kind, sm_count, st);
  }
  Params p;
  p.a = a;
  if (out_kind != kFastMel) { p.a.nnz = 0; p.a.n_mels = 0; p.a.mel_rounds = 0; p.a.mel_mpad = 0; }
  p.span_cap = span_needed(a.g);
  p.region_bytes = region_needed(out_kind, p.a.mel_mpad);
  p.row_stride = row_floats(out_kind, p.a.mel_mpad);
  p.tiles_per_signal = (a.g.frames + kTile - 1) / kTile;
  p.total_tiles = p.tiles_per_signal * a.batch;
  int groups = 4;
  auto layout = [&](int gr) {
    return smem_layout(out_kind, p.a.n_mels, p.a.nnz, p.a.mel_rounds, p.a.mel_mpad, p.span_cap, gr);
  };
  while (groups > 2 && layout(groups) > kSmemLimit) --groups;
  const size_t smem = layout(groups);
  if (smem > kSmemLimit) return cudaErrorInvalidConfiguration;
  long long want = (p.total_tiles + groups - 1) / groups;
  const int grid = (int)(want < sm_count ? want : sm_count);
  cudaError_t e;
#define SMB_LAUNCHTC_GS(OUT, SQ, G, S1)                                                      \
  e = cudaFuncSetAttribute(stft2048tc_kernel<OUT, SQ, G, S1>,                                \
                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);          \
  if (e != cudaSuccess) return e;                                                            \
  stft2048tc_kernel<OUT, SQ, G, S1><<<grid, G * kGroupThreads, smem, st>>>(p);
#define SMB_LAUNCHTC_G(OUT, SQ, G)                                                           \
  if (a.bin_step == 1) { SMB_LAUNCHTC_GS(OUT, SQ, G, true) } else { SMB_LAUNCHTC_GS(OUT, SQ, G, false) }
#define SMB_LAUNCHTC(OUT, SQ)                                                                \
  if (groups == 4) { SMB_LAUNCHTC_G(OUT, SQ, 4) }                                           \
  else if (groups == 3) { SMB_LAUNCHTC_G(OUT, SQ, 3) }                                      \
  else { SMB_LAUNCHTC_G(OUT, SQ, 2) }
  const bool sq = a.power == 2.0f;
  if (out_kind == kFastMel) { if (sq) { SMB_LAUNCHTC(kFastMel, true) } else { SMB_LAUNCHTC(kFastMel, false) } }
  else if (out_kind == kFastPower) { if (sq) { SMB_LAUNCHTC(kFastPower, true) } else { SMB_LAUNCHTC(kFastPower, false) } }
  else { SMB_LAUNCHTC(kFastComplex, true) }
#undef SMB_LAUNCHTC
#undef SMB_LAUNCHTC_G
#undef SMB_LAUNCHTC_GS
  ++g_launch_count;
  return cudaGetLastError();
}

}  // namespace smb
