// Fused STFT kernel for fft_size = 2048, float32 audio (sm_100a).
//
//   framing + boundary extension + window -> real FFT 2048 -> |X|^p
//   -> (optionally) sparse mel projection -> [batch, bins | n_mels, frames]
//
// replaces, for this geometry, Stft.analyse / magnitude_pow / Mel.apply
// (stft.ml:356-364, 670-674; mel.ml:202-231) in one pass: the complex spectrum
// and the power spectrogram never reach HBM on the mel path.
//
// Frame sizes 1024, 512, 256 and 128 ride on the same kernel: a frame zero-padded
// to 2048 has the shorter transform's bin k at bin k * (2048 / fft), so the host
// hands over a window whose tail is zero and `bin_step` = 2048 / fft; the real
// split keeps every bin_step-th bin in the frame's row, and everything after it
// (mel bands, write-out) sees a row of fft / 2 + 1 bins.
//
// Decomposition
//   * One persistent CTA per SM, 16 warps in independent groups.  A group of
//     kFastTile warps owns a tile of kFastTile consecutive frames of one signal:
//     it stages the tile's (kFastTile-1)*hop + 2048 samples once (each sample is
//     shared by up to four overlapping frames), then every warp transforms one
//     frame.  Two shapes are written out -- two groups of 8 warps (the default)
//     and four groups of 4 (one warp of every group on each scheduler); on the
//     headline workload they measure 1.44 ms and 1.48 ms per 1024-clip launch:
//     the longer tile amortises the mel weights and the halo over more frames.
//   * Real FFT 2048 = complex FFT 1024 on z[n] = x[2n] + i x[2n+1], done as
//     32 x 32: pass 1 (lane = n2) is a 32-point FFT held entirely in
//     registers over the stride-32 samples, the twiddled result is transposed
//     through a padded, warp-private shared buffer, pass 2 (lane = k1) is the
//     second register FFT (both in the packed float32x2 form of fft32.cuh: FADD2 /
//     FMUL2 / FFMA2 halve their issue slots; measured 1.58 -> 1.47 ms on the headline
//     workload).  The even/odd split that turns Z into the real
//     spectrum pairs bin k with 1024-k, which live in lanes l and 32-l: the
//     partner values move by warp shuffle, each lane finishing 16 pairs.
//   * Mel: the filterbank is >98 % zeros (each bin feeds at most two
//     triangles), so the projection runs as a band product over the tile's power
//     rows in shared memory, in float32 FMAs: every filter's band is cut into
//     pieces of a few float4 steps, a lane carries one piece for all the frames of
//     the tile (one 16-byte weight load feeds 4 FMAs per frame), partial sums are
//     added at write-out.
//   * Interior tiles are brought in by one bulk copy (TMA) per tile, issued by
//     one thread and awaited on the group's mbarrier; boundary tiles go through
//     cp.async and the reference's index rule.
//   * Outputs are staged per tile so global writes run along the contiguous
//     frame axis.
#include <algorithm>
#include <cstdint>
#include <cstdlib>

#include "fft32.cuh"
#include "kernels.h"
#include "stft_stage.cuh"

namespace smb {

namespace {

constexpr int kFft = 2048;
constexpr int kHalf = 1024;              // complex points
constexpr int kTile = kFastTile;         // frames per group tile, one warp each
constexpr int kGroupThreads = 32 * kTile;
constexpr int kGroupWarps = kTile;
constexpr int kMaxGroups = kTile == 8 ? 2 : 4;
static_assert(kTile == 8 || kTile == 4, "tile shapes the lane maps are written for");
// floats per warp region: holds [32][34] complex; 16-byte rows; the frames of a
// tile land 4 banks apart (8 frames) or 8 banks apart (4 frames)
constexpr int kRowStride = kTile == 8 ? 2180 : 2184;
constexpr int kMelOutOff = 1032;         // the mel partial sums of a frame sit behind its power row
constexpr int kExStride = 34;            // padded transpose row (complex): 16-byte rows, conflict-free

using namespace fft32impl;

struct Params {
  Stft2048Args a;
  // interior tiles by one bulk copy: tiles t in
  // [bulk_t_lo, bulk_t_hi] of a clip b with (b * bulk_nmod + bulk_c0) % 4 == 0
  int bulk_t_lo, bulk_t_hi;
  unsigned bulk_nmod, bulk_c0;
  int span_cap;              // floats reserved per group for samples
  long long tiles_per_signal, total_tiles;
  // bin-major outputs (power / complex): a group walks a contiguous run of tiles and
  // keeps the frames that do not fill a 32-byte sector of an output row until the
  // next tile completes it (see the write-out); carry_cap = floats per group, 0 = off
  int carry_cap;
  int carry_period;              // carried elements per S consecutive rows
  unsigned long long carry_prefix;   // byte i: carried elements of the rows before row i of a period
};

// Brings one tile's samples (padded stream positions p0*hop .. + span) into the
// group's sample buffer.  Positions that map to real samples are fetched with
// cp.async (16 bytes per request when source and destination are both 16-byte
// aligned, else 8 or 4); border positions are resolved by the reference's
// boundary rule (stft.ml:300-338) and stored directly.  Completion is awaited
// by the caller (cp.async.wait_all + group barrier).  An interior tile whose source
// run is 16-byte aligned is one bulk copy (TMA) issued by the group's first thread
// onto `bar`: returns true and the caller waits on the mbarrier instead.
__device__ __forceinline__ bool stage_tile(const Params& p, int b, int t, float* sSamples, int gtid,
                                           uint32_t bar) {
  const FrameGeom& g = p.a.g;
  // interior full tile with a 16-byte aligned source run: the launcher worked the
  // tile range and the clip-phase rule out once (a handful of 32-bit operations
  // here instead of the 64-bit bounds and address tests in every thread)
  if (t >= p.bulk_t_lo && t <= p.bulk_t_hi && (((unsigned)b * p.bulk_nmod + p.bulk_c0) & 3u) == 0) {
    if (gtid == 0) {
      const uint32_t span = (uint32_t)((kTile - 1) * g.hop + kFft);
      const float* src = p.a.x + (long long)b * g.n + ((long long)t * kTile * g.hop - g.left);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_expect_tx(bar, 4u * span);
      bulk_g2s(smem_u32(sSamples), src, 4u * span, bar);
    }
    return true;
  }
  const long long p0 = (long long)t * kTile;              // tile t of clip b
  const int nf = (int)min((long long)kTile, g.frames - p0);
  const int span = (nf - 1) * g.hop + kFft;
  const long long q0 = p0 * g.hop;
  const long long s0 = q0 - g.left;
  const float* xs = p.a.x + (long long)b * g.n;
  // [lo, hi): positions of the span that are real samples
  const int lo = (int)max(0LL, min((long long)span, -s0));
  const int hi = (int)max((long long)lo, min((long long)span, g.n - s0));
  for (int i = gtid; i < lo; i += kGroupThreads) {
    const long long s = stage::src_index(g, q0 + i);
    sSamples[i] = s >= 0 ? __ldg(xs + s) : (float)g.pad_value;
  }
  for (int i = hi + gtid; i < span; i += kGroupThreads) {
    const long long s = stage::src_index(g, q0 + i);
    sSamples[i] = s >= 0 ? __ldg(xs + s) : (float)g.pad_value;
  }
  stage::copy_real_samples<kGroupThreads>(smem_u32(sSamples), xs + s0, lo, hi, gtid);
  return false;
}

// STEP1: bin_step == 1 (fft 2048 proper): every bin is kept, no per-bin tests.
template <int OUT, bool SQUARE, int kGroups, bool STEP1>
__global__ void __launch_bounds__(kGroups * kGroupThreads, 1)
stft2048_kernel(const Params p) {
  extern __shared__ __align__(16) float smem[];
  // Constant tables are laid out so a lane fetches two of its values per
  // 16-byte load: [pair][lane][2] (half the shared-memory instructions).
  float* sWindow = smem;                                        // [16][32] x {w(n1), w(n1+1)} float2 pairs, x 1/2
  float2* sTwPass = reinterpret_cast<float2*>(sWindow + kFft);  // [16][32][2]  W_1024^(k1 n2), k1 = 2 pair + {0,1}
  float2* sTwPost = sTwPass + 1024;                             // [32]         W_2048^l
  float* sMelVals = reinterpret_cast<float*>(sTwPost + 32);     // band weights [round][step][lane] x float4
  const int nnz_pad = (p.a.nnz + 3) & ~3;
  MelPiece* sPieces = reinterpret_cast<MelPiece*>(sMelVals + nnz_pad);   // [warps][rounds][32]
  unsigned char* sPcnt = reinterpret_cast<unsigned char*>(sPieces + kGroupWarps * p.a.mel_rounds * 32);
  __shared__ __align__(8) uint64_t sbars[kMaxGroups];          // bulk copy of a group's samples landed
  __shared__ unsigned char sCarryMap[32];                       // carry slot within a period -> row phase | k << 4
  // offsets stay integers so every pointer keeps its shared-memory provenance
  // (generic LD/ST would go through the slower generic path)
  const int tables_bytes = (kFft + 2 * 1024 + 2 * 32 + nnz_pad) * 4 +
                           kGroupWarps * p.a.mel_rounds * 32 * (int)sizeof(MelPiece) +
                           ((p.a.n_mels + 3) & ~3);
  float* groups_base = smem + (((tables_bytes + 15) & ~15) >> 2);
  const int group_floats = p.span_cap + kTile * kRowStride + p.carry_cap;

  const int tid = threadIdx.x;
  const int group = tid / kGroupThreads;
  const int gtid = tid % kGroupThreads;
  const int warp = gtid >> 5;
  const int lane = tid & 31;
  float* sSamples = groups_base + group * group_floats;
  float* sRows = sSamples + p.span_cap;
  float* sCarry = sRows + kTile * kRowStride;

  for (int i = tid; i < kFft; i += blockDim.x) {
    // source index j = 2 (32 n1 + l) + c  ->  ((n1/2) * 32 + l) * 4 + (n1 & 1) * 2 + c
    const int c = i & 1, l = (i >> 1) & 31, n1 = i >> 6;
    sWindow[(((n1 >> 1) * 32 + l) << 2) + ((n1 & 1) << 1) + c] = p.a.window[i] * 0.5f;
  }
  for (int i = tid; i < 1024; i += blockDim.x) {
    const int l = i & 31, k1 = i >> 5;
    sTwPass[(((k1 >> 1) * 32 + l) << 1) + (k1 & 1)] = p.a.tw_pass[i];
  }
  if (tid < 32) sTwPost[tid] = p.a.tw_post[tid];
  if (OUT == kFastMel) {
    for (int i = tid; i < p.a.nnz; i += blockDim.x) sMelVals[i] = p.a.vals[i];
    for (int i = tid; i < kGroupWarps * p.a.mel_rounds * 32; i += blockDim.x) sPieces[i] = p.a.mel_pieces[i];
    for (int i = tid; i < p.a.n_mels; i += blockDim.x) sPcnt[i] = p.a.mel_pcnt[i];
  }
  if (OUT != kFastMel && p.carry_cap) {
    const int S = OUT == kFastComplex ? 4 : 8;
    if (tid < S) {
      const int q = (tid * (int)(p.a.g.frames & (S - 1))) & (S - 1);
      const int at = (int)((p.carry_prefix >> (8 * tid)) & 0xff);
      for (int k = 0; k < q; ++k) sCarryMap[at + k] = (unsigned char)(tid | (k << 4));
    }
  }
  if (tid == 0) {
    for (int gI = 0; gI < kMaxGroups; ++gI) mbar_init(smem_u32(&sbars[gI]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const uint32_t sbar = smem_u32(&sbars[group]);
  uint32_t sphase = 0;

  const FrameGeom g = p.a.g;
  const int bin_shift = STEP1 ? 0 : 31 - __clz(p.a.bin_step), bin_mask = STEP1 ? 0 : p.a.bin_step - 1;
  // tile indices fit 32 bits (checked by the launcher): cheap decode
  const int slot = blockIdx.x * kGroups + group;
  const int stride = gridDim.x * kGroups;
  const int total_tiles = (int)p.total_tiles, tiles_per_signal = (int)p.tiles_per_signal;
  float* row = sRows + warp * kRowStride;
  float2* ex = reinterpret_cast<float2*>(row);

  // where a thread starts in the carry slots, and how a step of kGroupThreads moves it
  const int cper = OUT != kFastMel && p.carry_cap ? p.carry_period : 1;
  const int park_g4 = gtid / cper, park_idx = gtid % cper;
  const int park_dq = kGroupThreads / cper, park_dr = kGroupThreads % cper;
  // mel: tiles dealt round-robin; bin-major outputs with a carry: contiguous runs
  int first = slot, last = total_tiles, tstep = stride;
  if (OUT != kFastMel && p.carry_cap) {
    const int run = (total_tiles + stride - 1) / stride;
    first = min(slot * run, total_tiles);
    last = min(first + run, total_tiles);
    tstep = 1;
  }
  // (clip, tile of the clip) walk the deal without a division per tile
  const int step_b = tstep / tiles_per_signal, step_t = tstep - step_b * tiles_per_signal;
  int nb = first / tiles_per_signal, nt = first - nb * tiles_per_signal;
  bool bulk = false;
  if (first < last) bulk = stage_tile(p, nb, nt, sSamples, gtid, sbar);
  for (int tile = first; tile < last; tile += tstep) {
    const int b = nb;
    const long long p0 = (long long)nt * kTile;
    nb += step_b;
    nt += step_t;
    if (nt >= tiles_per_signal) { nt -= tiles_per_signal; ++nb; }
    const int nf = (int)min((long long)kTile, g.frames - p0);

    // ---- the tile's samples were requested one iteration ago (or just above
    // the loop): wait for this thread's copies, then for the group's.
    if (bulk) {
      mbar_wait(sbar, sphase & 1);
      ++sphase;
    } else {
      asm volatile("cp.async.wait_all;" ::: "memory");
    }
    named_sync(group + 1, kGroupThreads);

    if (warp < nf) {
      // ---- pass 1: lane = n2, registers = n1; z[n] = x[2n] + i x[2n+1], n = 32 n1 + n2
      float2 a[32];
      const float* fs = sSamples + warp * g.hop;
      const float4* w4 = reinterpret_cast<const float4*>(sWindow);
      if (((warp * g.hop) & 1) == 0) {
        const float2* f2 = reinterpret_cast<const float2*>(fs);
#pragma unroll
        for (int n1 = 0; n1 < 32; n1 += 2) {
          const float2 v0 = f2[32 * n1 + lane], v1 = f2[32 * (n1 + 1) + lane];
          const float4 w = w4[(n1 >> 1) * 32 + lane];
          a[n1] = make_float2(v0.x * w.x, v0.y * w.y);
          a[n1 + 1] = make_float2(v1.x * w.z, v1.y * w.w);
        }
      } else {
#pragma unroll
        for (int n1 = 0; n1 < 32; n1 += 2) {
          const float4 w = w4[(n1 >> 1) * 32 + lane];
          a[n1] = make_float2(fs[64 * n1 + 2 * lane] * w.x, fs[64 * n1 + 2 * lane + 1] * w.y);
          a[n1 + 1] = make_float2(fs[64 * (n1 + 1) + 2 * lane] * w.z,
                                  fs[64 * (n1 + 1) + 2 * lane + 1] * w.w);
        }
      }
      fft32_packed(a);                            // a[k1] = Y[n2 = lane][k1]
      // twiddle W1024^(k1 n2) and transpose through the padded buffer
      {
        const float4* t4 = reinterpret_cast<const float4*>(sTwPass);
#pragma unroll
        for (int k1 = 0; k1 < 32; k1 += 2) {
          const float4 t = t4[(k1 >> 1) * 32 + lane];
          ex[k1 * kExStride + lane] =
              k1 == 0 ? a[0]
                      : make_float2(a[k1].x * t.x - a[k1].y * t.y, a[k1].x * t.y + a[k1].y * t.x);
          ex[(k1 + 1) * kExStride + lane] = make_float2(a[k1 + 1].x * t.z - a[k1 + 1].y * t.w,
                                                        a[k1 + 1].x * t.w + a[k1 + 1].y * t.z);
        }
      }
      __syncwarp();
      // ---- pass 2: lane = k1, registers = n2  ->  a[k2] = Z'[k1 + 32 k2]
      {
        const float4* e4 = reinterpret_cast<const float4*>(ex + lane * kExStride);
#pragma unroll
        for (int n2 = 0; n2 < 32; n2 += 2) {
          const float4 v = e4[n2 >> 1];
          a[n2] = make_float2(v.x, v.y);
          a[n2 + 1] = make_float2(v.z, v.w);
        }
      }
      __syncwarp();                               // the buffer becomes the output row
      fft32_packed(a);

      // ---- real-spectrum split.  With Z' = Z/2 (window pre-scaled):
      //   S = Z'[k] + conj Z'[N-k],  D = Z'[k] - conj Z'[N-k],  W = W2048^k
      //   X[k] = S + W (-i D),   X[N-k] = conj(S - W (-i D))
      const int partner = (32 - lane) & 31;
      float2 r[16];
#pragma unroll
      for (int k2 = 0; k2 < 16; ++k2) {
        // lanes != 0 need the partner's register 31-k2; lane 0 pairs with itself
        // through register (32-k2) mod 32.
        const float2 own = a[31 - k2];
        const float2 alt = a[(32 - k2) & 31];
        const float sx = lane == 0 ? alt.x : own.x;
        const float sy = lane == 0 ? alt.y : own.y;
        r[k2].x = __shfl_sync(0xffffffffu, sx, partner);
        r[k2].y = __shfl_sync(0xffffffffu, sy, partner);
      }
      float2* rowc = reinterpret_cast<float2*>(row);
      const float2 wl = sTwPost[lane];
#pragma unroll
      for (int k2 = 0; k2 < 16; ++k2) {
        const float2 A = a[k2];
        const float2 S = make_float2(A.x + r[k2].x, A.y - r[k2].y);
        const float2 D = make_float2(A.x - r[k2].x, A.y + r[k2].y);
        const float2 w = k2 == 0 ? wl
                                 : make_float2(wl.x * kW64C[k2] - wl.y * kW64S[k2],
                                               wl.x * kW64S[k2] + wl.y * kW64C[k2]);
        const float tr = w.x * D.y + w.y * D.x;
        const float ti = w.y * D.y - w.x * D.x;
        const float2 xk = make_float2(S.x + tr, S.y + ti);
        const float2 xn = make_float2(S.x - tr, ti - S.y);
        const int k = lane + 32 * k2, nk = kHalf - k;
        const bool keep_k = STEP1 || (k & bin_mask) == 0, keep_n = STEP1 || (nk & bin_mask) == 0;
        if (OUT == kFastComplex) {
          if (keep_k) rowc[k >> bin_shift] = xk;
          if (keep_n) rowc[nk >> bin_shift] = xn;
        } else {
          float pk = xk.x * xk.x + xk.y * xk.y;
          float pn = xn.x * xn.x + xn.y * xn.y;
          if (!SQUARE) {
            if (p.a.power == 1.0f) { pk = sqrtf(pk); pn = sqrtf(pn); }
            else { pk = powf(sqrtf(pk), p.a.power); pn = powf(sqrtf(pn), p.a.power); }
          }
          if (keep_k) row[k >> bin_shift] = pk;
          if (keep_n) row[nk >> bin_shift] = pn;
        }
      }
      if (lane == 0) {                            // k = 512 pairs with itself
        const float2 xm = make_float2(2.0f * a[16].x, -2.0f * a[16].y);
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
    named_sync(group + 1, kGroupThreads);

    // ---- the sample buffer is free: start fetching the next tile's samples
    // under the mel / write-out phases.
    if (tile + tstep < last) bulk = stage_tile(p, nb, nt, sSamples, gtid, sbar);

    if (OUT == kFastMel) {
      // ---- mel projection over the tile's power rows.  A lane carries one piece
      // (a few float4 steps of one filter's band) for all the frames of the tile:
      // the weight load is one contiguous run per warp, the rows' loads fall in
      // distinct bank groups across a quarter-warp (host schedule); a warp's
      // pieces in a round share one step count, so there is no divergence.
      const MelPiece* mine = sPieces + warp * p.a.mel_rounds * 32 + lane;
      float* part = sRows + kMelOutOff;
      for (int r = 0; r < p.a.mel_rounds; ++r) {
        const MelPiece q = mine[r * 32];
        const int steps = (int)((unsigned)q.off >> 24);
        const float4* wq = reinterpret_cast<const float4*>(sMelVals + (q.off & 0xFFFFFF));
        const float4* v = reinterpret_cast<const float4*>(sRows + q.lo);
        float acc[kTile];
#pragma unroll
        for (int f = 0; f < kTile; ++f) acc[f] = 0.0f;
        for (int i = 0; i < steps; ++i) {
          const float4 ww = wq[32 * i];
          float4 x[kTile];
#pragma unroll
          for (int f = 0; f < kTile; ++f) x[f] = v[f * (kRowStride / 4) + i];
#pragma unroll
          for (int f = 0; f < kTile; ++f) {
            acc[f] = fmaf(ww.x, x[f].x, acc[f]);
            acc[f] = fmaf(ww.y, x[f].y, acc[f]);
            acc[f] = fmaf(ww.z, x[f].z, acc[f]);
            acc[f] = fmaf(ww.w, x[f].w, acc[f]);
          }
        }
#pragma unroll
        for (int f = 0; f < kTile; ++f) part[f * kRowStride + q.pid] = acc[f];
      }
      named_sync(group + 1, kGroupThreads);
    }

    // ---- write the tile along the frame axis: [batch, rows, frames].  kTile
    // consecutive lanes carry the tile's frames of one output row.
    {
      const int f = gtid & (kTile - 1), r0 = gtid / kTile;
      if (OUT == kFastMel) {
        if (f < nf) {
          float* ob = p.a.out + ((long long)b * p.a.n_mels + r0) * g.frames + p0 + f;
          const long long step = (long long)(kGroupThreads / kTile) * g.frames;
          const float* src = sRows + f * kRowStride + kMelOutOff;
          // the j-th partial sum of filter m sits at j * mpad + m (up to four; slots a
          // filter does not use hold stale bits and are masked out, never added)
          const int mpad = p.a.mel_mpad;
#pragma unroll 4
          for (int m = r0; m < p.a.n_mels; m += kGroupThreads / kTile, ob += step) {
            const int cnt = sPcnt[m];
            const float s0 = src[m], s1 = src[mpad + m], s2 = src[2 * mpad + m], s3 = src[3 * mpad + m];
            *ob = (s0 + (cnt > 1 ? s1 : 0.0f)) + ((cnt > 2 ? s2 : 0.0f) + (cnt > 3 ? s3 : 0.0f));
          }
        }
      }
      if (OUT != kFastMel) {
        // Rows are frames-contiguous and a tile's 8 frames start anywhere inside a
        // 32-byte sector of the row (row length is odd at the headline shape), so a
        // plain write leaves a partial sector at both ends of every run; L2 writes
        // those back before the neighbouring tile fills them (ncu: +1.5 GB DRAM read,
        // +0.9 GB write at 1024 clips).  Instead every row writes the 8 elements that
        // start q = (row offset mod sector) before the tile: q carried over from the
        // previous tile of the same clip (kept by the same thread, no barrier) plus
        // its own first 8-q, and parks its last q.  First / last tiles of a clip or
        // of the group's run write what they have.
        typedef typename std::conditional<OUT == kFastComplex, float2, float>::type T;
        constexpr int S = 32 / (int)sizeof(T);               // elements per sector
        const int out_bins = kHalf / p.a.bin_step + 1;
        const long long R0 = (long long)b * out_bins;
        const int fm = (int)(g.frames & (S - 1));
        const bool carrying = p.carry_cap != 0;
        const bool has_carry = carrying && tile != first && p0 != 0;
        const bool park = carrying && tile + tstep < last && p0 + kTile < g.frames;   // then nf == kTile
        T* carry = reinterpret_cast<T*>(sCarry);
        const T* src = reinterpret_cast<const T*>(sRows);
        constexpr int kRowT = kRowStride * 4 / (int)sizeof(T);
        T* out = reinterpret_cast<T*>(p.a.out);
        // a thread's rows are kGroupThreads / kTile apart, a multiple of S: its phase
        // in the sector period, hence q and its side of the split, never change
        constexpr int kRows = kGroupThreads / kTile;
        static_assert(kRows % S == 0, "row step keeps the sector phase");
        const int ph = (int)((R0 + r0) & (S - 1));
        const int q = carrying ? (ph * fm) & (S - 1) : 0;
        const bool own = f >= q;
        const int j0 = f - q, j1 = kTile - q + f;             // first-store frame / parked frame
        const bool w = own ? j0 < nf : has_carry;
        const bool tail = !own && j1 < nf;
        const int cs = p.carry_period * (int)(((R0 + r0) / S) - (R0 / S)) + (int)((p.carry_prefix >> (8 * ph)) & 0xff) + f;
        const int cstep = p.carry_period * (kRows / S);
        T* orow = out + (R0 + r0) * g.frames + p0;
        const long long ostep = (long long)kRows * g.frames;
        // one load per row position whichever side the thread is on
        const T* ld = own ? src + j0 * kRowT + r0 : carry + cs;
        const int ldstep = own ? kRows : cstep;
        if (park) {
          if (w)
            for (int r = r0; r < out_bins; r += kRows, orow += ostep, ld += ldstep) orow[j0] = *ld;
          named_sync(group + 1, kGroupThreads);                                  // the old carry has been read
          // park the tile's last q frames of every row: carry slot e <-> (row, frame)
          // through the per-period map, dense over the group's threads
          const int r_off = (int)(R0 & (S - 1));
          const int total = ((int)((R0 + out_bins - 1) / S - R0 / S) + 1) * p.carry_period;
          int g4 = park_g4, idx = park_idx;
          for (int e = gtid; e < total; e += kGroupThreads) {
            const int m = sCarryMap[idx];
            const int mph = m & 15, k = m >> 4;
            const int r = g4 * S + mph - r_off;
            const int mq = (mph * fm) & (S - 1);
            if (r >= 0 && r < out_bins) carry[e] = src[(kTile - mq + k) * kRowT + r];
            idx += park_dr;
            g4 += park_dq;
            if (idx >= p.carry_period) { idx -= p.carry_period; ++g4; }
          }
        } else {
          const T* s1 = src + (tail ? j1 : 0) * kRowT;
          for (int r = r0; r < out_bins; r += kRows, orow += ostep, ld += ldstep) {
            if (w) orow[j0] = *ld;
            if (tail) orow[j1] = s1[r];
          }
        }
      }
    }
    // no barrier here: nothing writes the rows before the group barrier at the top
    // of the next iteration, which orders these row reads before the next tile's
    // transposes (and the parked carry before its readers)
  }
}

}  // namespace

static size_t smem_layout(int n_mels, int nnz, int mel_rounds, int span_cap, int groups) {
  const int nnz_pad = (nnz + 3) & ~3;
  size_t bytes = (size_t)(kFft + 2 * 1024 + 2 * 32) * 4;         // window, tw_pass, tw_post
  bytes += (size_t)nnz_pad * 4;                                    // band weights
  bytes += (size_t)kGroupWarps * mel_rounds * 32 * sizeof(MelPiece);          // warp schedule
  bytes += (size_t)((n_mels + 3) & ~3);                            // partial sums per filter
  bytes = (bytes + 15) & ~(size_t)15;
  bytes += (size_t)groups * (span_cap + kTile * kRowStride) * 4;
  return bytes;
}

static const size_t kSmemLimit = 232448;   // 227 KB opt-in maximum per CTA

static int span_needed(const FrameGeom& g) {
  return (((kTile - 1) * g.hop + kFft) + 3) & ~3;
}

bool stft2048_supports(const FrameGeom& g, int out_kind, int n_mels, int nnz, int mel_rounds,
                       int mpad) {
  if (g.fft != kFft || g.hop < 1 || g.hop > 4096) return false;   // g: the kernel's geometry
  // the partial sums of a frame live behind its power row, inside the row stride
  if (out_kind == kFastMel && (n_mels < 1 || n_mels > 255 || nnz >= (1 << 24) ||
                               kMelOutOff + 4 * mpad + 1 > kRowStride))
    return false;
  const bool mel = out_kind == kFastMel;
  return smem_layout(mel ? n_mels : 0, mel ? nnz : 0, mel ? mel_rounds : 0, span_needed(g),
                     kMaxGroups / 2) <= kSmemLimit;
}

cudaError_t launch_stft2048(const Stft2048Args& a, int out_kind, int sm_count, cudaStream_t st) {
  if (a.batch == 0 || a.g.frames == 0) return cudaSuccess;
  if ((a.g.frames + kTile - 1) / kTile * a.batch >= (1LL << 31)) {
    // tile indices are 32-bit inside the kernel: split the batch
    const long long half = a.batch / 2;
    Stft2048Args lo = a, hi = a;
    lo.batch = half;
    hi.batch = a.batch - half;
    hi.x = a.x + half * a.g.n;
    const long long rows = out_kind == kFastMel ? a.n_mels : kHalf / a.bin_step + 1;
    hi.out = a.out + half * rows * a.g.frames * (out_kind == kFastComplex ? 2 : 1);
    cudaError_t e1 = launch_stft2048(lo, out_kind, sm_count, st);
    return e1 != cudaSuccess ? e1 : launch_stft2048(hi, out_kind, sm_count, st);
  }
  Params p;
  p.a = a;
  p.bulk_t_lo = 0;
  p.bulk_t_hi = -1;
  p.bulk_nmod = p.bulk_c0 = 0;
  if ((a.g.hop & 3) == 0 && (reinterpret_cast<size_t>(a.x) & 3) == 0) {
    // full tile t reads source samples [t*T*hop - left, ... + span): inside the clip, and
    // 16-byte aligned when (x/4 + b*n - left) % 4 == 0 (T*hop is a multiple of 4)
    const long long th = (long long)kTile * a.g.hop, span = (long long)(kTile - 1) * a.g.hop + kFft;
    const long long lo = (a.g.left + th - 1) / th;
    const long long hi = std::min<long long>((a.g.n + a.g.left - span >= 0 ? (a.g.n + a.g.left - span) / th : -1),
                                  a.g.frames / kTile - 1);
    if (lo <= hi) {
      p.bulk_t_lo = (int)lo;
      p.bulk_t_hi = (int)hi;
      p.bulk_nmod = (unsigned)(a.g.n & 3);
      p.bulk_c0 = (unsigned)(((reinterpret_cast<size_t>(a.x) >> 2) + 4 - (size_t)(a.g.left & 3)) & 3);
    }
  }
  if (out_kind != kFastMel) { p.a.nnz = 0; p.a.n_mels = 0; p.a.mel_rounds = 0; p.a.mel_mpad = 0; }
  p.span_cap = span_needed(a.g);
  p.tiles_per_signal = (a.g.frames + kTile - 1) / kTile;
  p.total_tiles = p.tiles_per_signal * a.batch;
  // the full complement of groups per SM when their tiles fit shared memory, else half
  const int groups = smem_layout(p.a.n_mels, p.a.nnz, p.a.mel_rounds, p.span_cap, kMaxGroups) <= kSmemLimit
                         ? kMaxGroups : kMaxGroups / 2;
  size_t smem = smem_layout(p.a.n_mels, p.a.nnz, p.a.mel_rounds, p.span_cap, groups);
  if (smem > kSmemLimit) return cudaErrorInvalidConfiguration;
  p.carry_cap = p.carry_period = 0;
  p.carry_prefix = 0;
  if (out_kind != kFastMel && !getenv("SMB_NO_CARRY")) {
    // sector carry of the bin-major write-out: q(row) = (row * frames) mod S elements
    const int S = out_kind == kFastComplex ? 4 : 8;
    const int fm = (int)(a.g.frames & (S - 1));
    int period = 0;
    for (int i = 0; i < S; ++i) {
      p.carry_prefix |= (unsigned long long)period << (8 * i);
      period += (i * fm) & (S - 1);
    }
    const int out_bins = kHalf / a.bin_step + 1;
    const int cap = ((period * (out_bins / S + 2) * (out_kind == kFastComplex ? 2 : 1)) + 3) & ~3;
    if (period > 0 && smem + (size_t)groups * cap * 4 + 64 <= kSmemLimit) {   // 64: the static tables
      p.carry_cap = cap;
      p.carry_period = period;
      smem += (size_t)groups * cap * 4;
    }
  }
  long long want = (p.total_tiles + groups - 1) / groups;
  const int grid = (int)(want < sm_count ? want : sm_count);
  cudaError_t e;
#define SMB_LAUNCH2048_GS(OUT, SQ, G, S1)                                                    \
  e = cudaFuncSetAttribute(stft2048_kernel<OUT, SQ, G, S1>,                                  \
                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);          \
  if (e != cudaSuccess) return e;                                                            \
  stft2048_kernel<OUT, SQ, G, S1><<<grid, G * kGroupThreads, smem, st>>>(p);
#define SMB_LAUNCH2048_G(OUT, SQ, G)                                                         \
  if (a.bin_step == 1) { SMB_LAUNCH2048_GS(OUT, SQ, G, true) } else { SMB_LAUNCH2048_GS(OUT, SQ, G, false) }
#define SMB_LAUNCH2048(OUT, SQ)                                                              \
  if (groups == kMaxGroups) { SMB_LAUNCH2048_G(OUT, SQ, kMaxGroups) }                       \
  else { SMB_LAUNCH2048_G(OUT, SQ, kMaxGroups / 2) }
  const bool sq = a.power == 2.0f;
  if (out_kind == kFastMel) { if (sq) { SMB_LAUNCH2048(kFastMel, true) } else { SMB_LAUNCH2048(kFastMel, false) } }
  else if (out_kind == kFastPower) { if (sq) { SMB_LAUNCH2048(kFastPower, true) } else { SMB_LAUNCH2048(kFastPower, false) } }
  else { SMB_LAUNCH2048(kFastComplex, true) }
#undef SMB_LAUNCH2048
#undef SMB_LAUNCH2048_G
#undef SMB_LAUNCH2048_GS
  ++g_launch_count;
  return cudaGetLastError();
}

}  // namespace smb
