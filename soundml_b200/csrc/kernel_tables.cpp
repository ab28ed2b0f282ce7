// Host-side builders of the kernels' tables.  See kernel_tables.h.
#include "kernel_tables.h"

#include <algorithm>
#include <cstdlib>
#include <cstring>

namespace smb {

namespace {

// Puts weight g at (row r, element k < 32) of a tensor-core resampler B slice that starts
// at float `base` and holds `rows` rows per split: its tf32 piece hi (the float's leading
// 10 fraction bits, exact) in the first split and lo = g - hi in the second, each at the
// K-major SWIZZLE_128B cell (128-byte rows, 16-byte chunk index XOR row mod 8).
void put_tf32_split(std::vector<float>& img, size_t base, int64_t rows, int64_t r, int64_t k, double g) {
  const float gf = (float)g;
  uint32_t bits;
  std::memcpy(&bits, &gf, 4);
  bits &= 0xFFFFE000u;
  float hi;
  std::memcpy(&hi, &bits, 4);
  const float lo = (float)(g - (double)hi);
  const size_t cell = (size_t)(r * 32 + ((((k >> 2) ^ (r & 7)) << 2) | (k & 3)));
  img[base + cell] = hi;
  img[base + (size_t)rows * 32 + cell] = lo;
}

// Each warp's rounds: longest first onto the warp with the least load, a round costing
// steps * per_step + per_round; `rounds` is set to the longest list.
template <typename Round>
std::vector<std::vector<int>> deal_longest_first(const std::vector<Round>& built, int warps, int per_step,
                                                 int per_round, int& rounds) {
  std::vector<int> by_len(built.size());
  for (size_t q = 0; q < built.size(); ++q) by_len[q] = (int)q;
  std::stable_sort(by_len.begin(), by_len.end(),
                   [&](int a, int b) { return built[(size_t)a].steps > built[(size_t)b].steps; });
  std::vector<std::vector<int>> lists((size_t)warps);
  std::vector<long long> load((size_t)warps, 0);
  for (int q : by_len) {
    const size_t w = (size_t)(std::min_element(load.begin(), load.end()) - load.begin());
    lists[w].push_back(q);
    load[w] += built[(size_t)q].steps * per_step + per_round;
  }
  rounds = 0;
  for (const auto& l : lists) rounds = std::max(rounds, (int)l.size());
  return lists;
}

// Width of the equal column groups of <= 160 (rounded up to 16) that l columns are cut into.
int64_t group_width(int64_t l) {
  const int64_t n_groups = (l + 159) / 160;
  return ((l + n_groups - 1) / n_groups + 15) / 16 * 16;
}

// Appends the row-form group of columns [c0, c0 + l) of L (l_total); false if it does not fit.
// split_main: the row grid is shifted so that every column's filter centre falls into the
// same shift (qc), and that shift's two small split terms get an accumulator of their own:
// its main accumulator then is a chain of exact hi x hi products only (4 per chunk).  With
// everything in one accumulator per shift, a 14-chunk stage (44.1 -> 16 kHz) measured
// -121.9 dB THD+N in float32 against the reference's -125 dB gate (resample_quality.ml
// Q1/Q2); the window form, which separates the small terms, -132.5 dB.
bool rows_group(std::vector<GemmLayout::Group<GemmRowsArgs>>& out, const ResampleStage& s, int64_t c0, int64_t l,
                bool single_group, bool split_main) {
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
  GemmRowsArgs a{};
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
  const int kSliceAlign = 8;
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
    while (a.b_stages > 2 && resample_rows_smem_bytes(0, a.b_stages, stage_bytes) + turn > budget) --a.b_stages;
    if (resample_rows_smem_bytes(0, a.b_stages, stage_bytes) + turn > budget) return false;
  } else if (resample_rows_smem_bytes(2, 3, stage_bytes) <= budget) { a.a_stages = 2; a.b_stages = 3; }
  else if (resample_rows_smem_bytes(3, 2, stage_bytes) <= budget) { a.a_stages = 3; a.b_stages = 2; }
  else if (resample_rows_smem_bytes(2, 2, stage_bytes) <= budget) { a.a_stages = 2; a.b_stages = 2; }
  else return false;
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
      const size_t base = ((size_t)chunk_meta[(size_t)ch].x + (size_t)run.bytes_at) / 4;
      put_tf32_split(img, base, run.width, tcol - run.start, kk, s.bank[(size_t)(ph * taps + t)]);
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
  out.push_back({a, std::move(img), std::move(chunk_meta), std::move(slice_meta)});
  return true;
}

}  // namespace

std::vector<float2> fft1024_pass_twiddles() {
  const std::vector<float2> w = unit_roots<float2>(1024, 1024);
  std::vector<float2> pass(1024);
  for (int k1 = 0; k1 < 32; ++k1)
    for (int n2 = 0; n2 < 32; ++n2) pass[(size_t)(k1 * 32 + n2)] = w[(size_t)(k1 * n2)];
  return pass;
}

// The 32-point DFT in real arithmetic, F[n = (k, c')][j = (m, c)] with (re, im)
// interleaved: out_re = sum in_re cos + in_im sin, out_im = sum in_im cos - in_re sin
// (angle 2 pi m k / 32).  Two fp16 images (leading 11 bits, remainder) in the K-major
// SWIZZLE_128B operand layout: row n is 128 bytes, its 16-byte chunk q sits at position
// q ^ (n mod 8).
std::vector<__half> dft32_split_images() {
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
  return images;
}

// Filter m's band [band_lo, band_hi) is read in 4-bin steps from an even bin b0 <=
// band_lo; eight consecutive filters make a round (neighbouring bands have similar
// lengths), lane (i, j) of the round's warp carries filter i for frame pair j.  The two
// filters of a quarter-warp start on 16-byte groups of opposite parity (b0 / 2 odd against
// even; one of them moves two bins down, weights zero there) so that the eight 16-byte
// loads of a quarter-warp, whose four frame pairs sit 32 bytes apart, fall in eight
// distinct bank groups.  Weights are stored [round][step][filter] x float4 = one 128-byte
// run per warp load.  Rounds go longest-first onto the lightest of the four warps.
PairSchedule pair_schedule(const std::vector<double>& weights, const std::vector<int>& band_lo,
                           const std::vector<int>& band_hi, int64_t n_mels, int64_t bins) {
  PairSchedule sc;
  const int kBins = 1032;                                  // power row incl. zeroed tail (stft2048p.cu)
  if (bins != 1025 || n_mels > 32767) return {};
  constexpr int F = kPairFilters;                          // filters per round (lane = filter, frame pair)
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
    if (rd.steps > 510 || 4 * rd.steps > kBins) return {};
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
  if (sc.w.size() >= (1u << 24)) return {};
  const int warps = kPairTile / 2;
  const auto lists = deal_longest_first(built, warps, 10, 30, sc.rounds);
  sc.items.assign((size_t)(warps * sc.rounds * F), PairMelItem{0, 0, -1});   // idle: no steps
  for (int wi = 0; wi < warps; ++wi)
    for (size_t r = 0; r < lists[(size_t)wi].size(); ++r) {
      const Round& rd = built[(size_t)lists[(size_t)wi][r]];
      for (int i = 0; i < F; ++i) {
        PairMelItem& it = sc.items[((size_t)wi * (size_t)sc.rounds + r) * F + (size_t)i];
        it.w4_steps = (int)(rd.base / 4 + (size_t)i) | ((rd.steps / 2) << 24);
        it.h0 = (unsigned short)(rd.b0[i] >> 1);
        it.m = (short)rd.m[i];
      }
    }
  return sc;
}

// Every filter's band, starting on a float4 of the power row, is cut into pieces of at
// most `ps` float4 steps; a lane carries one piece for all the frames of its tile (one
// weight load feeds 4 FMAs per frame) and leaves a partial sum in slot `pid` = j * mpad +
// m for the j-th piece of filter m (at most four per filter: `ps` grows with the longest
// band; the write-out adds the pcnt[m] of them up).  Rounds of 32 lanes share one step
// count.  They are filled longest pieces first out of a window of candidates, so that the
// lanes of a quarter-warp get distinct start residues (start / 4 mod 8) where the window
// allows: their 16-byte power-row loads then fall in distinct bank groups.  Weights are
// stored [round][step][lane] x float4, a contiguous run per warp-wide load.  Rounds go to
// the group's warps longest-first onto the lightest warp.
PieceSchedule piece_schedule(const std::vector<double>& weights, const std::vector<int>& band_lo,
                             const std::vector<int>& band_hi, int64_t n_mels, int64_t bins, int warps,
                             int ps, int window) {
  PieceSchedule sc;
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
  if (ps > 255) return {};
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
    if (rd.steps * 4 > row_floats) return {};
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
  const auto lists = deal_longest_first(built, warps, 21, 20, sc.rounds);
  const size_t zero_off = sc.vals.size();            // idle rounds: one step over zero weights
  sc.vals.insert(sc.vals.end(), (size_t)(32 * 4), 0.0f);
  if (sc.vals.size() >= (1u << 24)) return {};
  sc.pieces.assign((size_t)(warps * sc.rounds * 32), MelPiece{});
  for (int w = 0; w < warps; ++w)
    for (int r = 0; r < sc.rounds; ++r)
      for (int t = 0; t < 32; ++t) {
        MelPiece& out = sc.pieces[((size_t)w * (size_t)sc.rounds + (size_t)r) * 32 + (size_t)t];
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
  return sc;
}

GemmLayout gemm_layout(const ResampleStage& s) {
  GemmLayout out;
  const int64_t l = s.l, m = s.m, k = s.k, taps = 2 * k + 1;
  if (s.exec != kExecGemm || l > 1024) return out;
  const int64_t width = group_width(l);
  // long stages (many K-chunks = long accumulation chains) separate the small terms of the
  // main shift when tensor memory has room for the extra accumulator; SMB_ROWS_SPLIT=0/1 forces
  const bool want_split = getenv("SMB_ROWS_SPLIT") ? atoi(getenv("SMB_ROWS_SPLIT")) != 0 : (m + 31) / 32 >= 8;
  for (int attempt = want_split ? 0 : 1; attempt < 2; ++attempt) {
    bool ok = true;
    for (int64_t c0 = 0; c0 < l && ok; c0 += width)
      ok = rows_group(out.rows, s, c0, std::min<int64_t>(width, l - c0), l <= 160, attempt == 0);
    if (ok) break;
    out.rows.clear();
  }
  for (int c0 = 0; c0 < l; c0 += (int)width) {
    GemmLayout::Group<GemmResampleArgs> g;
    GemmResampleArgs& a = g.a;
    a.col_begin = c0;
    a.l = (int)std::min<int64_t>(width, l - c0);
    a.n_pad = (a.l + 15) / 16 * 16;
    a.m = (int)m;
    a.l_total = (int)l;
    // rows of G (K index) this group's columns touch: d(r) = floor(r M / L) .. + taps - 1
    const int64_t d_first = ((int64_t)c0 * m) / l;
    const int64_t d_last = ((int64_t)(c0 + a.l - 1) * m) / l + taps - 1;
    const int chunk_begin = (int)(d_first / 32);
    a.k = (int)k - 32 * chunk_begin;                          // the group's first K-chunk is chunk 0
    a.chunks = (int)(d_last / 32) - chunk_begin + 1;
    a.tmem_cols = 32;
    while (a.tmem_cols < 3 * a.n_pad) a.tmem_cols *= 2;
    // G is banded: chunk ch only has nonzeros in a run of columns.  Store and
    // multiply just that run, widened to multiples of 16 columns; the group's
    // first two chunks keep the full width because their first products
    // zero-initialise the accumulators.
    std::vector<int> cmin((size_t)a.chunks, a.n_pad), cmax((size_t)a.chunks, -1);
    for (int r = 0; r < a.l; ++r) {
      const int64_t d = ((int64_t)(c0 + r) * m) / l;
      for (int64_t ch = d / 32; ch <= (d + taps - 1) / 32; ++ch) {
        const size_t rel = (size_t)(ch - chunk_begin);
        cmin[rel] = std::min(cmin[rel], r);
        cmax[rel] = std::max(cmax[rel], r);
      }
    }
    g.chunk_meta.resize((size_t)a.chunks);
    size_t total_floats = 0;
    for (int ch = 0; ch < a.chunks; ++ch) {
      int col0 = 0, ncols = a.n_pad;
      if (ch >= 2 && cmax[(size_t)ch] >= 0) {
        col0 = cmin[(size_t)ch] / 16 * 16;
        ncols = (cmax[(size_t)ch] + 1 - col0 + 15) / 16 * 16;
      } else if (ch >= 2) {
        ncols = 16;                                          // empty chunk: a zero slice
      }
      g.chunk_meta[(size_t)ch] = make_int4((int)(total_floats * 4), col0, ncols, 0);
      total_floats += (size_t)2 * ncols * 32;
    }
    g.images.assign(total_floats, 0.0f);
    for (int r = 0; r < a.l; ++r) {
      const int64_t col = c0 + r;
      const int64_t d = (col * m) / l, ph = (col * m) % l;
      for (int64_t t = 0; t < taps; ++t) {
        const int64_t j = d + t;                               // row of G
        const int64_t ch = j / 32 - chunk_begin, kk = j % 32;
        const int4 mt = g.chunk_meta[(size_t)ch];
        // row r - mt.y of the stored slice
        put_tf32_split(g.images, (size_t)mt.x / 4, mt.z, r - mt.y, kk, s.bank[(size_t)(ph * taps + t)]);
      }
    }
    out.windows.push_back(std::move(g));
  }
  return out;
}

}  // namespace smb
