// Phase-rich polyphase stage as a banded matrix product on the 5th-generation
// tensor cores (tcgen05 + TMEM), sm_100a.
//
// The reference runs such stages (L >= 64 phases, e.g. 44.1 -> 16 kHz: L/M =
// 160/441, 523 taps) as [R; P] x [P; L] through Nx.matmul
// (resample.ml:430-476, 1608-1698, gemm_bank :207-226): block-row rho holds the
// L outputs of one phase cycle and reads the P = 2K + 1 + floor((L-1) M / L)
// consecutive inputs starting at rho*M - K; column r of G is the phase-(r M mod L)
// bank row shifted down by floor(r M / L).  This is a true dense contraction
// (3.8 TFLOP for BASELINE config 4), so it belongs on the tensor pipe:
//
//   D[128 rows x L] (TMEM, fp32)  +=  A[128 x 32] (smem)  *  B[L x 32]^T (smem)
//
// per K-chunk of 32 inputs, kind::tf32.  float32 accuracy (1e-5 of peak) is kept
// by operand splitting: a = a_hi + a_lo, g = g_hi + g_lo with 11-bit pieces and
// D += a_hi g_hi + a_hi g_lo + a_lo g_hi  (the dropped term is 2^-22).  The two
// small terms go to their own accumulator and the main term alternates between
// two accumulators per chunk, which keeps each accumulation chain short.
//
//   A: gathered by four producer warps (a warp takes 32 block-rows, lane = sample
//      within the chunk: one coalesced 128-byte request per row), split, written
//      in the canonical K-major SWIZZLE_128B layout (16-byte chunk index XOR row
//      mod 8); loads run two chunks ahead in registers.
//   B: pre-split, pre-swizzled images of G built once per plan on the host; one
//      cp.async.bulk (TMA) per chunk lands hi+lo with an mbarrier.
//   MMA: a fifth warp's elected lane issues 4 K-steps x 3 products per chunk;
//      tcgen05.commit releases the stage; three stages, mbarriers only.
//   Epilogue: tcgen05.ld (32 lanes x 16 columns per warp), sum of the three
//      accumulators, transposed through shared memory so global stores are
//      row-contiguous (a block-row is L consecutive outputs).
#include "kernels.h"
#include "sm100.cuh"

#include <algorithm>
#include <cstdint>

namespace smb {

namespace {

constexpr int kRows = 128;            // block-rows per CTA (UMMA M)
constexpr int kChunk = 32;            // tf32 elements per 128-byte swizzle row
constexpr int kStages = 3;
constexpr int kABytes = kRows * 128;  // one split of the A chunk
constexpr int kProducerWarps = 8;      // warps 0-3 double as the epilogue
constexpr int kProducers = kProducerWarps * 32;
constexpr int kRowsPerWarp = kRows / kProducerWarps;
constexpr int kMmaWarp = kProducerWarps;
constexpr int kThreads = kProducers + 32;  // producer warps + 1 TMA/MMA warp

// K-major, SWIZZLE_128B shared-memory matrix descriptor (8-row groups 1024 B apart).
__device__ __forceinline__ uint64_t umma_desc(uint32_t addr) {
  uint64_t d = 0;
  d |= (uint64_t)((addr >> 4) & 0x3FFF);         // start address, 16-byte units
  d |= (uint64_t)1 << 16;                         // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;               // stride byte offset between 8-row groups
  d |= (uint64_t)1 << 46;                         // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                         // SWIZZLE_128B
  return d;
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// loads and waits: the values are ready on return
__device__ __forceinline__ void tmem_ld16_waited(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// Warps 0-3: producers (gather + split + swizzled store of A) and, at the end,
// the epilogue (a warp may only read its own 32 TMEM lanes).  Warp 4: loads the
// B images by TMA and issues the MMAs.  Stages hand over through mbarriers only:
//   a_full[s] (128 arrivals)  b_full[s] (TMA bytes)  ->  MMA  ->  empty[s] (commit)
__global__ void __launch_bounds__(kThreads, 1)
resample_gemm_kernel(const GemmResampleArgs a) {
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B operands need 1024-byte aligned tiles
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~(uintptr_t)1023);
  const int b_bytes = a.n_pad * 128;                      // one split of the B chunk
  const int stage_bytes = 2 * kABytes + 2 * b_bytes;
  __shared__ __align__(8) uint64_t bars[3 * kStages + 1];
  __shared__ uint32_t tmem_base_slot;

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int lane = tid & 31;
  const long long c = blockIdx.y;
  const long long row0 = (long long)blockIdx.x * kRows;
  const float* xs = a.x + c * a.n;
  float* out = a.out + c * a.n_out;

  const uint32_t bar_a = smem_u32(&bars[0]);                // [stage]: A tile written
  const uint32_t bar_b = smem_u32(&bars[kStages]);          // [stage]: B bytes landed
  const uint32_t bar_empty = smem_u32(&bars[2 * kStages]);  // [stage]: MMAs reading the stage done
  const uint32_t bar_done = smem_u32(&bars[3 * kStages]);   // all MMAs done
  if (tid == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(bar_a + 8 * s, kProducers);
      mbar_init(bar_b + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    mbar_init(bar_done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp) tmem_alloc(&tmem_base_slot, a.tmem_cols);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tmem_base_slot;
  const uint32_t acc_main0 = tmem, acc_main1 = tmem + a.n_pad;
  const uint32_t acc_corr = tmem + 2 * a.n_pad;

  if (warp == kMmaWarp) {
    // ===== B loader + MMA issuer (one elected lane) =====
    if (lane == 0) {
      // instruction descriptor: D f32, A/B tf32, both K-major, M = 128; N per chunk
      const uint32_t idesc0 = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kRows >> 4) << 24);
      uint32_t used_main0 = 0, used_main1 = 0, used_corr = 0;
      const uint8_t* images = reinterpret_cast<const uint8_t*>(a.b_images);
      // G is banded: chunk ch only touches columns [col0, col0 + ncols) of the
      // accumulators, and only that slice of the image exists (chunk_meta).
      auto load_b = [&](int ch) {
        const int s = ch % kStages;
        const int4 meta = __ldg(a.chunk_meta + ch);
        const uint32_t bytes = 2u * (uint32_t)meta.z * 128u;
        mbar_expect_tx(bar_b + 8 * s, bytes);
        bulk_g2s(smem_u32(smem + s * stage_bytes + 2 * kABytes), images + meta.x, bytes,
                 bar_b + 8 * s);
      };
      for (int ch = 0; ch < kStages && ch < a.chunks; ++ch) load_b(ch);
      for (int ch = 0; ch < a.chunks; ++ch) {
        const int s = ch % kStages;
        const uint32_t parity = (ch / kStages) & 1;
        mbar_wait(bar_a + 8 * s, parity);
        mbar_wait(bar_b + 8 * s, parity);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int4 meta = __ldg(a.chunk_meta + ch);
        const uint32_t idesc = idesc0 | ((uint32_t)(meta.z >> 3) << 17);
        const uint32_t a_hi = smem_u32(smem + s * stage_bytes), a_lo = a_hi + kABytes;
        const uint32_t b_hi = a_hi + 2 * kABytes, b_lo = b_hi + (uint32_t)meta.z * 128u;
        const uint32_t acc = ((ch & 1) ? acc_main1 : acc_main0) + (uint32_t)meta.y;
        const uint32_t acc_c = acc_corr + (uint32_t)meta.y;
        uint32_t& used = (ch & 1) ? used_main1 : used_main0;
#pragma unroll
        for (int ks = 0; ks < kChunk / 8; ++ks) {
          const uint32_t off = ks * 32;                             // 8 tf32 = 32 bytes along K
          umma_tf32(acc, umma_desc(a_hi + off), umma_desc(b_hi + off), idesc, used);
          used = 1;
          umma_tf32(acc_c, umma_desc(a_hi + off), umma_desc(b_lo + off), idesc, used_corr);
          used_corr = 1;
          umma_tf32(acc_c, umma_desc(a_lo + off), umma_desc(b_hi + off), idesc, 1);
        }
        umma_commit(bar_empty + 8 * s);
        if (ch == a.chunks - 1) umma_commit(bar_done);
        // refill this stage's B as soon as its MMAs have drained
        if (ch + kStages < a.chunks) {
          mbar_wait(bar_empty + 8 * s, parity);
          load_b(ch + kStages);
        }
      }
    }
    __syncwarp();
  } else {
    // ===== producers: a warp gathers 32 block-rows, lane = sample within the
    // chunk, so every row is one coalesced 128-byte request.  Loads run two
    // chunks ahead of the stores (registers), stores one to three chunks ahead
    // of the tensor core (stages).
    float v0[kRowsPerWarp], v1[kRowsPerWarp];
    const long long first_row = row0 + warp * kRowsPerWarp;
    // x index of (row rr of this warp, this lane) in chunk 0; chunk ch adds 32 ch
    const long long base0 = first_row * a.m + lane - a.k;
    // the warp's whole footprint over all chunks is interior for most tiles:
    // no per-element bounds checks then
    const bool interior = first_row * a.m - a.k >= 0 &&
                          (first_row + kRowsPerWarp - 1) * a.m - a.k + (long long)a.chunks * kChunk <= a.n;
    auto load_chunk = [&](int ch, float (&v)[kRowsPerWarp]) {
      if (ch >= a.chunks) return;
      const long long b0 = base0 + (long long)ch * kChunk;
      if (interior) {
        const float* p = xs + b0;
#pragma unroll
        for (int rr = 0; rr < kRowsPerWarp; ++rr) v[rr] = __ldg(p + rr * a.m);
      } else {
#pragma unroll
        for (int rr = 0; rr < kRowsPerWarp; ++rr) {
          const long long si = b0 + (long long)rr * a.m;
          v[rr] = (si >= 0 && si < a.n) ? __ldg(xs + si) : 0.0f;
        }
      }
    };
    auto store_chunk = [&](int ch, const float (&v)[kRowsPerWarp]) {
      const int s = ch % kStages;
      if (ch >= kStages) mbar_wait(bar_empty + 8 * s, ((ch / kStages) - 1) & 1);
      // element (row, k) lands at 16-byte chunk (k/4) XOR (row mod 8) of its
      // 128-byte row (K-major SWIZZLE_128B)
      float* ahi = reinterpret_cast<float*>(smem + s * stage_bytes) + warp * kRowsPerWarp * 32;
      float* alo = ahi + kABytes / 4;
#pragma unroll
      for (int rr = 0; rr < kRowsPerWarp; ++rr) {
        const float h = __uint_as_float(__float_as_uint(v[rr]) & 0xFFFFE000u);
        const int cell = rr * 32 + ((((lane >> 2) ^ (rr & 7)) << 2) | (lane & 3));
        ahi[cell] = h;
        alo[cell] = v[rr] - h;
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // st.shared -> async proxy
      mbar_arrive(bar_a + 8 * s);
    };
    load_chunk(0, v0);
    load_chunk(1, v1);
    for (int ch = 0; ch < a.chunks; ch += 2) {
      store_chunk(ch, v0);
      load_chunk(ch + 2, v0);
      if (ch + 1 < a.chunks) {
        store_chunk(ch + 1, v1);
        load_chunk(ch + 3, v1);
      }
    }
    if (warp >= 4) goto teardown;             // warps 0-3 own the TMEM lanes

    // ===== epilogue: TMEM -> registers (thread = block-row) -> shared tile ->
    // row-contiguous global stores (a block-row is L consecutive outputs)
    mbar_wait(bar_done, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    float* tile = reinterpret_cast<float*>(smem);            // the stages are drained
    const int pitch = a.n_pad + 4;
    const uint32_t lane_base = ((uint32_t)(warp * 32)) << 16;
    const bool two_main = a.chunks > 1;
    for (int col = 0; col < a.n_pad; col += 16) {
      float d0[16], d1[16], dc[16];
      tmem_ld16_waited(acc_main0 + lane_base + col, d0);
      tmem_ld16_waited(acc_corr + lane_base + col, dc);
      if (two_main) tmem_ld16_waited(acc_main1 + lane_base + col, d1);
      float4* dst = reinterpret_cast<float4*>(tile + tid * pitch + col);
#pragma unroll
      for (int e = 0; e < 16; e += 4) {
        float4 o;
        o.x = (two_main ? d0[e] + d1[e] : d0[e]) + dc[e];
        o.y = (two_main ? d0[e + 1] + d1[e + 1] : d0[e + 1]) + dc[e + 1];
        o.z = (two_main ? d0[e + 2] + d1[e + 2] : d0[e + 2]) + dc[e + 2];
        o.w = (two_main ? d0[e + 3] + d1[e + 3] : d0[e + 3]) + dc[e + 3];
        dst[e >> 2] = o;
      }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(kRows) : "memory");   // producers/epilogue warps only
    // block-row r is the L_total consecutive outputs of one phase cycle; this
    // launch owns columns [col_begin, col_begin + l) of it
    const long long rows_total = (a.n_out + a.l_total - 1) / a.l_total;
    const int rows_here = (int)min((long long)kRows, rows_total - row0);
    const bool vec = ((a.l | a.l_total | a.col_begin) & 3) == 0 &&
                     (reinterpret_cast<size_t>(out) & 15) == 0;
    if (vec) {
      const int per_row = a.l >> 2;
      for (int j = tid; j < rows_here * per_row; j += kRows) {
        const int row = j / per_row, c4 = j - row * per_row;
        const long long g = (row0 + row) * a.l_total + a.col_begin + 4 * c4;
        const float4 val = *reinterpret_cast<const float4*>(tile + row * pitch + 4 * c4);
        if (g + 3 < a.n_out) {
          *reinterpret_cast<float4*>(out + g) = val;
        } else {                                              // the signal ends inside this float4
          const float e[4] = {val.x, val.y, val.z, val.w};
          for (int t = 0; t < 4 && g + t < a.n_out; ++t) out[g + t] = e[t];
        }
      }
    } else {
      for (int j = tid; j < rows_here * a.l; j += kRows) {
        const int row = j / a.l, cc = j - row * a.l;
        const long long g = (row0 + row) * a.l_total + a.col_begin + cc;
        if (g < a.n_out) out[g] = tile[row * pitch + cc];
      }
    }
  }
teardown:
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem, a.tmem_cols);
}


// ---------------------------------------------------------------------------------------
// Row form of the same product (GemmRowsArgs, kernels.h).  The window form above gathers
// row rho of A as the P consecutive inputs from rho M - K: consecutive rows overlap, so
// every input sample is fetched, split and stored P / M times (2.18 x for 44.1 -> 16 kHz),
// a tile walks ceil(P / 32) K-chunks, and each chunk is 12 small products.  Here A is
// the input cut into NON-overlapping rows X[i][j'] = xz[i M + j' - K], j' < M; with
// G_q = rows [q M, (q + 1) M) of G
//
//     out[rho][r] = sum_q  ( X[rho + q] . G_q[:, r] )
//
// so the CTA keeps one accumulator D_q = X G_q per shift q (q < ceil(P / M) <= 4; the later
// ones only hold the few columns whose taps reach that far) and the epilogue adds
// D_q[i + q] into output row i.  The accumulators sit side by side in tensor memory in
// DESCENDING q: the band of G makes the active columns of D_q a suffix and those of
// D_(q-1) a prefix, so a chunk's nonzeros are one contiguous run of TMEM columns -- ONE
// product of N ~ 200 per K-step and split term where the window form issues several of
// N ~ 16 .. 160 (the tensor core retires a small product faster than one thread can issue
// the next: measured ~ 94 cycles per tcgen05.mma).
//
// A tile is 128 rows of A = four groups of 32 X-rows, one per epilogue warp (a warp can
// only read its own 32 TMEM lanes); consecutive groups overlap by shifts - 1 X-rows, so
// that every warp finds D_q[i + q] in its own lanes (a warp shuffle) and finishes
// 32 - (shifts - 1) output rows on its own: no exchange, no barrier in the epilogue.
//
// One persistent CTA per SM, warp-specialised, every hand-over an mbarrier:
//   warps 0-7   producers: gather, split and store the A chunks, running ahead of the
//               tensor core by the two A stages (and two more chunks in registers), across tiles;
//   warp  8     one lane issues the MMAs and nothing else (a chunk is 12 products; whatever
//               else that thread does is time the tensor core's queue runs dry); after a
//               tile's last chunk it commits acc_full and waits for acc_free;
//   warp  9     one lane streams the B images (cp.async.bulk), stage by stage as they drain;
//   warp  18    a second MMA issuer for plans that deal their slices to two owners;
//   warps 10-17 epilogue (two per TMEM lane quarter, alternate 16-column groups): drain the accumulators, shift,
//               turn 32 x 16 blocks through shared memory (a drained B stage) and write whole
//               64-byte runs to global memory, zero the accumulators with tcgen05.st (every
//               product accumulates) and arrive on acc_free.  Meanwhile the producers and
//               the B loader are already filling the next tile's stages.
constexpr int kMaxStages = 4;                       // A / B stages: shared-memory A (2, 3) or (3, 2); tensor-memory A (2, up to 4)
constexpr int kLoadWarp = kMmaWarp + 1;             // streams the B images
constexpr int kEpiWarp0 = kMmaWarp + 2;
constexpr int kEpiWarps = 8;                        // two per TMEM lane quarter, alternate 16-column groups (four cost the
                                                    // five-chunk stages 15 %: 0.84 -> 0.96 ms)
constexpr int kEpiPerQuarter = kEpiWarps / 4;
constexpr int kIssue2Warp = kEpiWarp0 + kEpiWarps;    // the second MMA issuer (plans with two owners)
constexpr int kRowsThreads = kThreads + 32 + 32 * kEpiWarps + 32;
constexpr int kMaxRowsChunks = 32, kMaxRowsSlices = 80;
constexpr int kRowsTurnBytes = kProducerWarps * 32 * 17 * 4;   // the producers' transposition tiles (A in tensor memory)

__device__ __forceinline__ void tmem_st16_zero(uint32_t taddr) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};"
      ::"r"(taddr), "r"(0u) : "memory");
}
// load without the wait: several are put in flight, then one tcgen05.wait::ld
__device__ __forceinline__ void tmem_ld16_async(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// A operand from tensor memory (lane = row, consecutive columns = consecutive K)
__device__ __forceinline__ void umma_tf32_ta(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.eq.b32 p, 0, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc)
      : "memory");
}

__global__ void __launch_bounds__(kRowsThreads, 1)
resample_rows_kernel(const GemmRowsArgs a, const int tiles_per_clip, const int total_tiles) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~(uintptr_t)1023);
  const int kAStages = a.a_stages, kBStages = a.b_stages;
  const bool a_in_tmem = a.a_tmem != 0;                     // A tiles in tensor memory: 64 columns per stage
  uint8_t* b_smem = smem + (a_in_tmem ? 0 : kAStages * 2 * kABytes);
  __shared__ __align__(8) uint64_t bars[4 * kMaxStages + 3];
  __shared__ uint32_t tmem_base_slot;
  __shared__ int4 s_chunk[kMaxRowsChunks], s_slice[kMaxRowsSlices];

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int lane = tid & 31;
  const int group_rows = 32 - (a.shifts - 1);               // finished output rows per epilogue warp
  const int rows_out = 4 * group_rows;                      // ... per tile

  const uint32_t bar_a = smem_u32(&bars[0]);                         // [A stage]: tile written
  const uint32_t bar_a_empty = smem_u32(&bars[kMaxStages]);          // [A stage]: its MMAs done
  const uint32_t bar_b = smem_u32(&bars[2 * kMaxStages]);            // [B stage]: bytes landed
  const uint32_t bar_b_empty = smem_u32(&bars[3 * kMaxStages]);
  const uint32_t bar_acc_full = smem_u32(&bars[4 * kMaxStages]);     // a tile's MMAs done
  const uint32_t bar_acc_free = smem_u32(&bars[4 * kMaxStages + 1]); // accumulators drained and zeroed
  const uint32_t bar_scratch = smem_u32(&bars[4 * kMaxStages + 2]);  // the epilogue is done with the B stage it borrowed
  if (tid == 0) {
    for (int s = 0; s < kAStages; ++s) {
      mbar_init(bar_a + 8 * s, kProducers);
      mbar_init(bar_a_empty + 8 * s, 1 + a.two_issuers);
    }
    for (int s = 0; s < kBStages; ++s) {
      mbar_init(bar_b + 8 * s, 1);
      mbar_init(bar_b_empty + 8 * s, 1 + a.two_issuers);
    }
    mbar_init(bar_acc_full, 1 + a.two_issuers);
    mbar_init(bar_acc_free, 32 * kEpiWarps);
    mbar_init(bar_scratch, kEpiWarps);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = tid; i < a.chunks; i += kRowsThreads) s_chunk[i] = a.chunk_meta[i];
  for (int i = tid; i < a.slices; i += kRowsThreads) s_slice[i] = a.slice_meta[i];
  if (warp == kMmaWarp) tmem_alloc(&tmem_base_slot, a.tmem_cols);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tmem_base_slot;

  // this CTA's tiles: blockIdx.x, + gridDim.x, ...
  const int my_tiles = total_tiles > (int)blockIdx.x ? (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int my_chunks = my_tiles * a.chunks;                 // (the launcher keeps this below 2^31)

  if (warp == kMmaWarp || (warp == kIssue2Warp && a.two_issuers)) {
    // ===== MMA issuer (one elected lane).  A plan may deal its slices to two issuers: one
    // thread issues a tcgen05.mma every ~80 cycles whatever its size, so the separated small
    // terms (twice the pieces) go through two threads side by side -- each accumulator is
    // only ever touched by one of them, which keeps the summation order fixed.
    const int owner = warp == kIssue2Warp ? 1 : 0;
    if (lane == 0) {
      const uint32_t idesc0 = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kRows >> 4) << 24);
      int sa = 0, sb = 0;
      uint32_t pa = 0, pb = 0;                               // parities of the stages' current use
      for (int it = 0; it < my_tiles; ++it) {
        mbar_wait(bar_acc_free, (uint32_t)(it & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        for (int ch = 0; ch < a.chunks; ++ch) {
          mbar_wait(bar_a + 8 * sa, pa);
          mbar_wait(bar_b + 8 * sb, pb);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const int4 meta = s_chunk[ch];
          // descriptors differ from their base only in the start-address field
          const uint64_t a_hi = umma_desc(smem_u32(smem + sa * 2 * kABytes));
          const uint64_t a_lo = a_hi + (uint64_t)(kABytes >> 4);
          const uint32_t b_base = smem_u32(b_smem + (size_t)sb * a.b_stage_bytes);
          for (int sl = meta.z; sl < meta.z + meta.w; ++sl) {
            const int4 sm = s_slice[sl];
            if (((sm.w >> 2) & 1) != owner) continue;
            const uint32_t idesc = idesc0 | ((uint32_t)(sm.z >> 3) << 17);
            const uint64_t b_hi = umma_desc(b_base + (uint32_t)sm.x);
            const uint64_t b_lo = b_hi + (uint64_t)((sm.w >> 3) >> 4);
            const int kind = sm.w & 3;                                   // 0 all, 1 hi x hi, 2 the small terms
            const uint32_t acc = tmem + (uint32_t)sm.y;
            if (a_in_tmem) {
              const uint32_t ta_hi = tmem + (uint32_t)(a.a_tmem_col + 64 * sa), ta_lo = ta_hi + 32;
#pragma unroll
              for (int ks = 0; ks < kChunk / 8; ++ks) {
                const uint64_t off = (uint64_t)(ks * 2);               // 8 tf32 = 32 bytes = 2 units along K
                if (kind != 2) umma_tf32_ta(acc, ta_hi + 8 * ks, b_hi + off, idesc);
                if (kind != 1) {
                  umma_tf32_ta(acc, ta_hi + 8 * ks, b_lo + off, idesc);
                  umma_tf32_ta(acc, ta_lo + 8 * ks, b_hi + off, idesc);
                }
              }
            } else {
#pragma unroll
              for (int ks = 0; ks < kChunk / 8; ++ks) {
                const uint64_t off = (uint64_t)(ks * 2);               // 8 tf32 = 32 bytes = 2 units along K
                if (kind != 2) umma_tf32(acc, a_hi + off, b_hi + off, idesc, 1);
                if (kind != 1) {
                  umma_tf32(acc, a_hi + off, b_lo + off, idesc, 1);
                  umma_tf32(acc, a_lo + off, b_hi + off, idesc, 1);
                }
              }
            }
          }
          umma_commit(bar_a_empty + 8 * sa);
          umma_commit(bar_b_empty + 8 * sb);
          if (ch == a.chunks - 1) umma_commit(bar_acc_full);
          if (++sa == kAStages) { sa = 0; pa ^= 1; }
          if (++sb == kBStages) { sb = 0; pb ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == kLoadWarp) {
    // ===== B loader: the chunk images in order, round and round, as stages drain
    if (lane == 0) {
      const uint8_t* images = reinterpret_cast<const uint8_t*>(a.b_images);
      int stage = 0, ch = 0;
      uint32_t parity = 1;                                   // (first use of a stage: nothing to wait for)
      for (int g = 0; g < my_chunks; ++g) {
        if (g >= kBStages) mbar_wait(bar_b_empty + 8 * stage, parity);
        // the stage of a tile's last chunk is lent to the epilogue as its transposition
        // scratch; it comes round again for chunk kBStages - 1 of the next tile
        if (ch == kBStages - 1 && g >= a.chunks) mbar_wait(bar_scratch, (uint32_t)((g / a.chunks - 1) & 1));
        const int4 meta = s_chunk[ch];
        mbar_expect_tx(bar_b + 8 * stage, (uint32_t)meta.y);
        bulk_g2s(smem_u32(b_smem + (size_t)stage * a.b_stage_bytes), images + meta.x, (uint32_t)meta.y,
                 bar_b + 8 * stage);
        if (++stage == kBStages) { stage = 0; parity ^= 1; }
        if (++ch == a.chunks) ch = 0;
      }
    }
    __syncwarp();
  } else if (warp < kProducerWarps && a_in_tmem) {
    // ===== producers, A in tensor memory.  A warp may only write its own TMEM lane quarter
    // (w4 = warp % 4: rows 32 w4 .. + 31 of the tile) and a thread writes a row, so warp
    // (w4, kh) owns the block [32 rows] x [16 samples: half kh of the chunk].  It is loaded
    // coalesced -- a load instruction reads two 64-byte row segments, lane = (row parity,
    // sample) -- two chunks ahead in registers, turned through a [32][17] shared-memory
    // tile so that lane = row, split, and written with two tcgen05.st (hi | lo).
    const int w4 = warp & 3, kh = warp >> 2;
    const uint32_t lane_base = ((uint32_t)(w4 * 32)) << 16;
    float* turn = reinterpret_cast<float*>(b_smem + (size_t)kBStages * a.b_stage_bytes) + warp * (32 * 17);
    const int sub = lane >> 4, cc = lane & 15;               // row parity and sample of the loads
    float v0[16] = {}, v1[16] = {};
    int ld_it = 0, ld_ch = 0;
    auto load_chunk = [&](float (&v)[16]) {
      if (ld_it >= my_tiles) return;
      const int tile = (int)blockIdx.x + ld_it * (int)gridDim.x;
      const int c = tile / tiles_per_clip;
      const long long row = (long long)(tile - c * tiles_per_clip) * rows_out + group_rows * w4 + sub;
      const float* xs = a.x + (long long)c * a.n;
      const long long b0 = row * a.m - a.k + (long long)ld_ch * kChunk + 16 * kh + cc;   // row `sub` of the block
      const long long first = b0 - cc - (long long)sub * a.m;                          // the block's first sample
      if (first >= 0 && first + 31LL * a.m + 16 <= a.n) {
        const float* p = xs + b0;
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = __ldg(p + 2 * i * a.m);
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const long long si = b0 + 2LL * i * a.m;
          v[i] = (si >= 0 && si < a.n) ? __ldg(xs + si) : 0.0f;
        }
      }
      if (++ld_ch == a.chunks) { ld_ch = 0; ++ld_it; }
    };
    int st_stage = 0;
    uint32_t st_parity = 1;
    int stored = 0;
    auto store_chunk = [&](const float (&v)[16]) {
      // v[i] = (row 2 i + sub, sample cc)  ->  lane = row, 16 samples
#pragma unroll
      for (int i = 0; i < 16; ++i) turn[(2 * i + sub) * 17 + cc] = v[i];
      __syncwarp();
      uint32_t hi[16], lo[16];
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        const float x = turn[lane * 17 + e];
        hi[e] = __float_as_uint(x) & 0xFFFFE000u;
        lo[e] = __float_as_uint(x - __uint_as_float(hi[e]));
      }
      __syncwarp();                                          // the tile may be overwritten
      if (stored >= kAStages) {
        mbar_wait(bar_a_empty + 8 * st_stage, st_parity);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      }
      const uint32_t col = tmem + lane_base + (uint32_t)(a.a_tmem_col + 64 * st_stage + 16 * kh);
      tmem_st16(col, hi);
      tmem_st16(col + 32, lo);
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      mbar_arrive(bar_a + 8 * st_stage);
      ++stored;
      if (++st_stage == kAStages) { st_stage = 0; st_parity ^= 1; }
    };
    load_chunk(v0);
    load_chunk(v1);
    for (int g = 0; g < my_chunks; g += 2) {
      store_chunk(v0);
      load_chunk(v0);
      if (g + 1 < my_chunks) {
        store_chunk(v1);
        load_chunk(v1);
      }
    }
  } else if (warp < kProducerWarps) {
    // ===== producers: a warp gathers 16 rows of the tile, lane = sample within the chunk
    // (one 128-byte request per row); loads run two chunks ahead of the stores in registers.
    // Tile row i is X-row  row0 + group_rows (i / 32) + i % 32  (the groups overlap).
    // (the loads run TWO chunks ahead in registers whatever the number of A stages)
    float v0[kRowsPerWarp] = {}, v1[kRowsPerWarp] = {};
    const int row_in_tile = group_rows * (warp >> 1) + kRowsPerWarp * (warp & 1);
    int ld_it = 0, ld_ch = 0;                                // next chunk to load: tile iteration, chunk
    auto load_chunk = [&](float (&v)[kRowsPerWarp]) {
      if (ld_it >= my_tiles) return;
      const int tile = (int)blockIdx.x + ld_it * (int)gridDim.x;
      const int c = tile / tiles_per_clip;
      const long long first_row = (long long)(tile - c * tiles_per_clip) * rows_out + row_in_tile;
      const float* xs = a.x + (long long)c * a.n;
      const long long b0 = first_row * a.m + lane - a.k + (long long)ld_ch * kChunk;
      // the warp's rows of this chunk are interior for most tiles: no bounds checks then
      if (b0 - lane >= 0 && b0 - lane + (long long)(kRowsPerWarp - 1) * a.m + kChunk <= a.n) {
        const float* p = xs + b0;
#pragma unroll
        for (int rr = 0; rr < kRowsPerWarp; ++rr) v[rr] = __ldg(p + rr * a.m);
      } else {
#pragma unroll
        for (int rr = 0; rr < kRowsPerWarp; ++rr) {
          const long long si = b0 + (long long)rr * a.m;
          v[rr] = (si >= 0 && si < a.n) ? __ldg(xs + si) : 0.0f;
        }
      }
      if (++ld_ch == a.chunks) { ld_ch = 0; ++ld_it; }
    };
    int st_stage = 0;
    uint32_t st_parity = 1;                                  // (first use of a stage: nothing to wait for)
    int stored = 0;
    auto store_chunk = [&](const float (&v)[kRowsPerWarp]) {
      if (stored >= kAStages) mbar_wait(bar_a_empty + 8 * st_stage, st_parity);
      // element (row, k) lands at 16-byte chunk (k/4) XOR (row mod 8) of its 128-byte row
      float* ahi = reinterpret_cast<float*>(smem + st_stage * 2 * kABytes) + warp * kRowsPerWarp * 32;
      float* alo = ahi + kABytes / 4;
#pragma unroll
      for (int rr = 0; rr < kRowsPerWarp; ++rr) {
        const float h = __uint_as_float(__float_as_uint(v[rr]) & 0xFFFFE000u);
        const int cell = rr * 32 + ((((lane >> 2) ^ (rr & 7)) << 2) | (lane & 3));
        ahi[cell] = h;
        alo[cell] = v[rr] - h;
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // st.shared -> async proxy
      mbar_arrive(bar_a + 8 * st_stage);
      ++stored;
      if (++st_stage == kAStages) { st_stage = 0; st_parity ^= 1; }
    };
    // loads run THREE chunks ahead of the stores in registers: a chunk's rows come from HBM
    // (the input is read once), and two chunk-times do not cover that latency (four deep
    // spills at this block size)
    float v2[kRowsPerWarp] = {};
    load_chunk(v0);
    load_chunk(v1);
    load_chunk(v2);
    for (int g = 0; g < my_chunks; g += 3) {
      store_chunk(v0);
      load_chunk(v0);
      if (g + 1 < my_chunks) { store_chunk(v1); load_chunk(v1); }
      if (g + 2 < my_chunks) { store_chunk(v2); load_chunk(v2); }
    }
  } else if (warp >= kEpiWarp0 && warp < kEpiWarp0 + kEpiWarps) {
    // ===== epilogue warps: w4 = the TMEM lane quarter this warp may read = its row group
    const int w4 = warp & 3;
    const int half = (warp - kEpiWarp0) >> 2;                 // which 16-column groups: even or odd
    const uint32_t lane_base = ((uint32_t)(w4 * 32)) << 16;
    int total_cols = 0;
    for (int q = 0; q < a.n_acc; ++q) total_cols += a.acc_w[q];
    // the accumulators start every tile at zero.  A warp zeroes exactly the columns it
    // drained (right after reading them): the other warp of its lane quarter may still be
    // reading its own.
    auto release_accumulators = [&]() {
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      mbar_arrive(bar_acc_free);
    };
    for (int col = 16 * half; col < total_cols; col += 16 * kEpiPerQuarter) tmem_st16_zero(tmem + lane_base + col);
    release_accumulators();
    const long long rows_total = (a.n_out + a.l_total - 1) / a.l_total;
    for (int it = 0; it < my_tiles; ++it) {
      const int tile = (int)blockIdx.x + it * (int)gridDim.x;
      const int c = tile / tiles_per_clip;
      const long long out_row = (long long)(tile - c * tiles_per_clip) * rows_out + group_rows * w4 + lane;
      mbar_wait(bar_acc_full, (uint32_t)(it & 1));
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      // out[row] = (D_0[row] + D_1[row + 1]) + D_2[row + 2] ..., 16 columns at a time.
      // When L is not a multiple of 4 (no aligned 16-byte stores) the block is turned
      // through a [32][17] tile so that a store instruction writes two whole 64-byte
      // runs instead of 32 words of 32 different rows (48 -> 44.1 kHz: 1.22 -> 0.97 ms).
      // The tile lives in the B stage of the tile's last chunk (drained: acc_full has
      // completed).
      float* obase = a.out + (long long)c * a.n_out;
      const long long base_row = out_row - lane;              // the warp's first output row
      const bool vec = ((a.l | a.l_total | a.col_begin) & 3) == 0 && (reinterpret_cast<size_t>(obase) & 15) == 0;
      const int last_stage = (int)(((long long)it * a.chunks + a.chunks - 1) % kBStages);
      float* tr = reinterpret_cast<float*>(b_smem + (size_t)last_stage * a.b_stage_bytes) +
                  (warp - kEpiWarp0) * (32 * 17);
      for (int col = 16 * half; col < a.n_pad; col += 16 * kEpiPerQuarter) {
        // every accumulator that holds these 16 columns, in a fixed order
        // ((acc0 + acc1) + acc2) + ..., three loads in flight at a time (registers)
        float o[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) o[e] = 0.0f;
#pragma unroll
        for (int q0 = 0; q0 < 6; q0 += 3) {
          if (q0 >= a.n_acc) break;
          uint32_t d[3][16];
          bool have[3];
#pragma unroll
          for (int u = 0; u < 3; ++u) {
            const int q = q0 + u;
            have[u] = q < a.n_acc && col >= a.acc_lo[q < 5 ? q : 4] && col < a.acc_lo[q < 5 ? q : 4] + a.acc_w[q < 5 ? q : 4];
            if (have[u]) tmem_ld16_async(tmem + lane_base + (uint32_t)(a.acc_col[q < 5 ? q : 4] + col - a.acc_lo[q < 5 ? q : 4]), d[u]);
          }
          tmem_ld_wait();
#pragma unroll
          for (int u = 0; u < 3; ++u) {
            const int q = q0 + u < 5 ? q0 + u : 4;
            if (have[u]) {                                       // (uniform)
              tmem_st16_zero(tmem + lane_base + (uint32_t)(a.acc_col[q] + col - a.acc_lo[q]));
              const int sh = a.acc_shift[q];
#pragma unroll
              for (int e = 0; e < 16; ++e) o[e] += __shfl_down_sync(0xffffffffu, __uint_as_float(d[u][e]), sh);
            }
          }
        }
        __syncwarp();                                            // the previous group has been read out
        const long long idx0 = base_row * a.l_total + a.col_begin + col;   // index of (the warp's row 0, col) in the clip
        const int rows_ok = (int)min((long long)group_rows, rows_total - base_row);
        if (vec && col + 16 <= a.l) {
          // L a multiple of 4: a lane writes its row's 64 bytes itself, four 16-byte
          // stores (measured faster than turning the block through shared memory:
          // 1.97 against 2.14 ms on the 44.1 -> 16 kHz workload -- the tensor core waits
          // for the epilogue, so its latency counts more than its sector efficiency)
          const long long idx = idx0 + lane * a.l_total;
          if (lane < rows_ok) {
            if (idx + 16 <= a.n_out) {
              float4* dst = reinterpret_cast<float4*>(obase + idx);
#pragma unroll
              for (int e = 0; e < 16; e += 4) dst[e >> 2] = make_float4(o[e], o[e + 1], o[e + 2], o[e + 3]);
            } else {
#pragma unroll
              for (int e = 0; e < 16; ++e)
                if (idx + e < a.n_out) obase[idx + e] = o[e];
            }
          }
        } else {
#pragma unroll
          for (int e = 0; e < 16; ++e) tr[lane * 17 + e] = o[e];
          __syncwarp();
          const int cc = lane & 15;
          if (col + cc < a.l) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int r = 2 * i + (lane >> 4);
              const long long idx = idx0 + r * a.l_total + cc;
              if (r < rows_ok && idx < a.n_out) obase[idx] = tr[r * 17 + cc];
            }
          }
        }
      }
      __syncwarp();
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic accesses before the next bulk copy
      if (lane == 0) mbar_arrive(bar_scratch);
      release_accumulators();
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  // tmem_dealloc written out: through the wrapper, nvcc 12.9 allocates this kernel's
  // registers differently (same instructions, other register numbers)
  if (warp == kMmaWarp)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem),
                 "r"(a.tmem_cols) : "memory");
}

}  // namespace

// (a_stages = 0 when the A tiles live in tensor memory)
size_t resample_rows_smem_bytes(int a_stages, int b_stages, int b_stage_bytes) {
  return (size_t)a_stages * 2 * kABytes + (size_t)b_stages * b_stage_bytes + 1024;
}

cudaError_t launch_resample_rows(const GemmRowsArgs& a, long long batch, int sm_count, cudaStream_t st) {
  if (batch == 0 || a.n_out == 0) return cudaSuccess;
  const size_t smem = resample_rows_smem_bytes(a.a_tmem ? 0 : a.a_stages, a.b_stages, a.b_stage_bytes) +
                      (a.a_tmem ? kRowsTurnBytes : 0);
  if (a.a_stages < 2 || a.a_stages > kMaxStages || a.b_stages < 2 || a.b_stages > kMaxStages) return cudaErrorInvalidConfiguration;
  if (smem > 227 * 1024 || a.shifts < 1 || a.shifts > 4 || a.n_acc < a.shifts || a.n_acc > 5 || a.chunks > kMaxRowsChunks || a.slices > kMaxRowsSlices)
    return cudaErrorInvalidConfiguration;
  cudaError_t e = cudaFuncSetAttribute(resample_rows_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const long long rows = (a.n_out + a.l_total - 1) / a.l_total;
  const int rows_out = 4 * (32 - (a.shifts - 1));
  const long long tiles = (rows + rows_out - 1) / rows_out;
  // tile and chunk counters are 32-bit inside the kernel: split the batch
  const long long max_clips = std::max<long long>(1, ((1LL << 31) - 1) / (tiles * a.chunks) - 1);
  if (tiles * a.chunks >= (1LL << 30)) return cudaErrorInvalidConfiguration;
  for (long long b0 = 0; b0 < batch; b0 += max_clips) {
    const long long nb = std::min(max_clips, batch - b0);
    GemmRowsArgs s = a;
    s.x = a.x + b0 * a.n;
    s.out = a.out + b0 * a.n_out;
    const long long total = tiles * nb;
    const int grid = (int)(total < sm_count ? total : sm_count);
    resample_rows_kernel<<<grid, kRowsThreads, smem, st>>>(s, (int)tiles, (int)total);
    ++g_launch_count;
  }
  return cudaGetLastError();
}

size_t resample_gemm_smem_bytes(int n_pad) {
  return (size_t)kStages * (2 * kABytes + 2 * (size_t)n_pad * 128) + 1024;
}

cudaError_t launch_resample_gemm(const GemmResampleArgs& a, long long batch, cudaStream_t st) {
  if (batch == 0 || a.n_out == 0) return cudaSuccess;
  const size_t smem = resample_gemm_smem_bytes(a.n_pad);
  if (smem > 227 * 1024) return cudaErrorInvalidConfiguration;
  cudaError_t e = cudaFuncSetAttribute(resample_gemm_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const long long rows = (a.n_out + a.l_total - 1) / a.l_total;
  const long long tiles = (rows + kRows - 1) / kRows;
  for (long long b0 = 0; b0 < batch; b0 += 65535) {
    const long long nb = batch - b0 < 65535 ? batch - b0 : 65535;
    GemmResampleArgs s = a;
    s.x = a.x + b0 * a.n;
    s.out = a.out + b0 * a.n_out;
    dim3 grid((unsigned)tiles, (unsigned)nb);
    resample_gemm_kernel<<<grid, kThreads, smem, st>>>(s);
    ++g_launch_count;
  }
  return cudaGetLastError();
}

}  // namespace smb
