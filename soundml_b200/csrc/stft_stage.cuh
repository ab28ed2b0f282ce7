// Device helpers shared by the STFT kernels: the reference's boundary rule, the
// cp.async fetch of a tile's real samples and the frame-pair kernel's tile staging that
// brings a run of overlapping frames into shared memory once.
#pragma once
#include <cstdint>

#include "kernels.h"
#include "sm100.cuh"

namespace smb {
namespace stage {

// padded stream position q -> source index, or -1 for the constant fill
// (stft.ml:300-338: reflect_index / edge clamp / constant).  kOneReflectionFirst tries
// the single reflection (every border of a signal longer than the extension) before
// the division.
template <bool kOneReflectionFirst = false>
__device__ __forceinline__ long long src_index(const FrameGeom& g, long long q) {
  long long s = q - g.left;
  if (s >= 0 && s < g.n) return s;
  if (g.pad == 0) {
    if (g.n == 1) return 0;
    const long long period = 2 * (g.n - 1);
    if (kOneReflectionFirst) {
      const long long once = s < 0 ? -s : period - s;
      if (once >= 0 && once < g.n) return once;
    }
    long long r = s % period;
    if (r < 0) r += period;
    return r < g.n ? r : period - r;
  }
  if (g.pad == 2) return s < 0 ? 0 : g.n - 1;
  return -1;
}

// cp.async of a tile's real samples, src[i] -> shared address base + 4 i for i in
// [lo, hi), over THREADS threads of which this is tid: 16-byte requests when src is
// 16-byte aligned (8 when 8-byte aligned; base is 16-byte aligned), single floats for
// the unaligned head and tail.  The caller waits with cp.async.wait_all.
template <int THREADS>
__device__ __forceinline__ void copy_real_samples(unsigned base, const float* src, int lo, int hi, int tid) {
  const size_t addr = reinterpret_cast<size_t>(src);
  if ((addr & 15) == 0) {
    const int head = min(hi, (lo + 3) & ~3), tail = max(head, hi & ~3);
    for (int i = lo + tid; i < head; i += THREADS)
      asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(base + 4u * i), "l"(src + i) : "memory");
    for (int i = head + 4 * tid; i < tail; i += 4 * THREADS)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(base + 4u * i), "l"(src + i) : "memory");
    for (int i = tail + tid; i < hi; i += THREADS)
      asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(base + 4u * i), "l"(src + i) : "memory");
  } else if ((addr & 7) == 0) {
    const int head = min(hi, (lo + 1) & ~1), tail = max(head, hi & ~1);
    for (int i = lo + tid; i < head; i += THREADS)
      asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(base + 4u * i), "l"(src + i) : "memory");
    for (int i = head + 2 * tid; i < tail; i += 2 * THREADS)
      asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(base + 4u * i), "l"(src + i) : "memory");
    for (int i = tail + tid; i < hi; i += THREADS)
      asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(base + 4u * i), "l"(src + i) : "memory");
  } else {
    for (int i = lo + tid; i < hi; i += THREADS)
      asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(base + 4u * i), "l"(src + i) : "memory");
  }
}

// Which tiles of which clips are one aligned bulk copy: tiles t in [t_lo, t_hi] of a
// clip b with (b * nmod + c0) % 4 == 0.  Worked out once by the launcher.
struct BulkRule {
  int t_lo, t_hi;
  unsigned nmod, c0;
  unsigned chunk;      // floats per bulk copy (multiple of 4), 0 = one copy per tile
};

// Brings the samples of tile t of clip b (padded stream positions t*TILE*hop .. + span)
// into `dst`.  An interior tile whose source run is 16-byte aligned is one bulk copy
// issued by the group's first thread onto `bar` (returns true: the caller waits on the
// mbarrier); any other tile fetches its real samples with cp.async (16 / 8 / 4 bytes
// as the alignment allows) and resolves border positions through the reference's
// boundary rule (returns false: the caller waits with cp.async.wait_all).
template <int TILE, int THREADS>
__device__ __forceinline__ bool stage_tile(const FrameGeom& g, const float* x, const BulkRule& rule,
                                           int b, int t, float* dst, int gtid, uint32_t bar) {
  if (t >= rule.t_lo && t <= rule.t_hi && (((unsigned)b * rule.nmod + rule.c0) & 3u) == 0) {
    if (gtid == 0) {
      const uint32_t span = (uint32_t)((TILE - 1) * g.hop + 2048);
      const float* src = x + (long long)b * g.n + ((long long)t * TILE * g.hop - g.left);
      // (no proxy fence: the buffer was only READ through the generic proxy, and those
      // reads have returned -- the readers counted off or passed a barrier after using
      // the values; a consumer release needs no more than that, as in every TMA pipeline)
      mbar_expect_tx(bar, 4u * span);
      // several copies instead of one: each keeps its own lines in flight (rule.chunk
      // floats apiece, a multiple of 4; 0 = the whole span at once)
      const uint32_t chunk = rule.chunk ? rule.chunk : span;
      for (uint32_t at = 0; at < span; at += chunk)
        bulk_g2s(smem_u32(dst + at), src + at, 4u * min(chunk, span - at), bar);
    }
    return true;
  }
  const long long p0 = (long long)t * TILE;
  const int nf = (int)min((long long)TILE, g.frames - p0);
  const int span = (nf - 1) * g.hop + 2048;
  const long long q0 = p0 * g.hop;
  const long long s0 = q0 - g.left;
  const float* xs = x + (long long)b * g.n;
  // [lo, hi): positions of the span that are real samples
  const int lo = (int)max(0LL, min((long long)span, -s0));
  const int hi = (int)max((long long)lo, min((long long)span, g.n - s0));
  // border positions, four per thread and round so that their loads are in flight together
  for (int side = 0; side < 2; ++side) {
    const int from = side == 0 ? 0 : hi, to = side == 0 ? lo : span;
    for (int i0 = from + gtid; i0 < to; i0 += 4 * THREADS) {
      float v[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int i = i0 + k * THREADS;
        const long long s = i < to ? src_index<true>(g, q0 + i) : -1;
        v[k] = s >= 0 ? __ldg(xs + s) : (float)g.pad_value;
      }
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (i0 + k * THREADS < to) dst[i0 + k * THREADS] = v[k];
    }
  }
  copy_real_samples<THREADS>(smem_u32(dst), xs + s0, lo, hi, gtid);
  return false;
}

// The launcher's side of BulkRule: full tile t reads source samples
// [t*TILE*hop - left, ... + span): inside the clip, and 16-byte aligned when
// (x/4 + b*n - left) % 4 == 0 (TILE*hop is a multiple of 4).
inline BulkRule bulk_rule(const float* x, const FrameGeom& g, int tile) {
  BulkRule r{0, -1, 0u, 0u, 0u};
  if ((g.hop & 3) != 0 || (reinterpret_cast<size_t>(x) & 3) != 0) return r;
  const long long th = (long long)tile * g.hop, span = (long long)(tile - 1) * g.hop + 2048;
  const long long lo = (g.left + th - 1) / th;
  long long hi = g.n + g.left - span >= 0 ? (g.n + g.left - span) / th : -1;
  if (g.frames / tile - 1 < hi) hi = g.frames / tile - 1;
  if (lo <= hi) {
    r.t_lo = (int)lo;
    r.t_hi = (int)hi;
    r.nmod = (unsigned)(g.n & 3);
    r.c0 = (unsigned)(((reinterpret_cast<size_t>(x) >> 2) + 4 - (size_t)(g.left & 3)) & 3);
  }
  return r;
}

}  // namespace stage
}  // namespace smb
