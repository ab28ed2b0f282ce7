// 32-point forward complex FFT held entirely in registers (one thread, natural
// order in and out): n = 8a + b, k = c + 4d -> eight 4-point DFTs over a, twiddle
// W32^(bc) with compile-time constants, four 8-point DFTs over b.  Also the warp-wide
// FFT 1024 built from it and the split twiddles of the real FFT 2048.  Shared by the
// fft-2048 STFT, overlap-save and iSTFT kernels and the micro-benchmark.
#pragma once
#include <cuda_runtime.h>

namespace smb {
namespace fft32impl {

__device__ constexpr float kW32C[32] = {
    1.0f, 0.9807852804032304f, 0.9238795325112867f, 0.8314696123025452f,
    0.7071067811865476f, 0.5555702330196023f, 0.38268343236508984f, 0.19509032201612833f,
    0.0f, -0.1950903220161282f, -0.3826834323650897f, -0.555570233019602f,
    -0.7071067811865475f, -0.8314696123025453f, -0.9238795325112867f, -0.9807852804032304f,
    -1.0f, -0.9807852804032304f, -0.9238795325112868f, -0.8314696123025455f,
    -0.7071067811865477f, -0.5555702330196022f, -0.38268343236509034f, -0.19509032201612866f,
    0.0f, 0.1950903220161283f, 0.38268343236509f, 0.5555702330196018f,
    0.7071067811865474f, 0.8314696123025452f, 0.9238795325112865f, 0.9807852804032303f};
__device__ constexpr float kW32S[32] = {
    0.0f, -0.19509032201612825f, -0.3826834323650898f, -0.5555702330196022f,
    -0.7071067811865475f, -0.8314696123025452f, -0.9238795325112867f, -0.9807852804032304f,
    -1.0f, -0.9807852804032304f, -0.9238795325112867f, -0.8314696123025455f,
    -0.7071067811865476f, -0.5555702330196022f, -0.3826834323650899f, -0.1950903220161286f,
    0.0f, 0.19509032201612836f, 0.38268343236508967f, 0.555570233019602f,
    0.7071067811865475f, 0.8314696123025452f, 0.9238795325112865f, 0.9807852804032303f,
    1.0f, 0.9807852804032304f, 0.9238795325112866f, 0.8314696123025455f,
    0.7071067811865477f, 0.5555702330196022f, 0.3826834323650904f, 0.19509032201612872f};

// W_64^k2 = exp(-2 pi i k2 / 64), k2 < 16: the split twiddle W_2048^(l + 32 k2) of the
// real FFT 2048 is the lane's W_2048^l (a 32-entry table) times one of these constants.
__device__ constexpr float kW64C[16] = {
    1.0f, 0.9951847266721969f, 0.9807852804032304f, 0.9569403357322088f,
    0.9238795325112867f, 0.881921264348355f, 0.8314696123025452f, 0.773010453362737f,
    0.7071067811865476f, 0.6343932841636455f, 0.5555702330196023f, 0.4713967368259978f,
    0.38268343236508984f, 0.29028467725446233f, 0.19509032201612833f, 0.09801714032956077f};
__device__ constexpr float kW64S[16] = {
    0.0f, -0.0980171403295606f, -0.19509032201612825f, -0.2902846772544623f,
    -0.3826834323650898f, -0.47139673682599764f, -0.5555702330196022f, -0.6343932841636455f,
    -0.7071067811865475f, -0.773010453362737f, -0.8314696123025452f, -0.8819212643483549f,
    -0.9238795325112867f, -0.9569403357322089f, -0.9807852804032304f, -0.9951847266721968f};

__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }

// v * W32^E with E a compile-time exponent: trivial rotations cost no multiply.
template <int E>
__device__ __forceinline__ float2 rot32(float2 v) {
  if constexpr (E == 0) return v;
  else if constexpr (E == 8) return make_float2(v.y, -v.x);
  else if constexpr (E == 16) return make_float2(-v.x, -v.y);
  else if constexpr (E == 24) return make_float2(-v.y, v.x);
  else if constexpr (E == 4) {
    const float r = 0.7071067811865476f;
    return make_float2((v.x + v.y) * r, (v.y - v.x) * r);
  } else if constexpr (E == 12) {
    const float r = 0.7071067811865476f;
    return make_float2((v.y - v.x) * r, -(v.x + v.y) * r);
  } else {
    constexpr float c = kW32C[E], s = kW32S[E];
    return make_float2(v.x * c - v.y * s, v.x * s + v.y * c);
  }
}

__device__ __forceinline__ void fft4(float2 a0, float2 a1, float2 a2, float2 a3,
                                     float2& x0, float2& x1, float2& x2, float2& x3) {
  const float2 t0 = cadd(a0, a2), t1 = csub(a0, a2), t2 = cadd(a1, a3);
  const float2 d = csub(a1, a3);
  const float2 t3 = make_float2(d.y, -d.x);     // -i (a1 - a3)
  x0 = cadd(t0, t2);
  x2 = csub(t0, t2);
  x1 = cadd(t1, t3);
  x3 = csub(t1, t3);
}

// 8-point forward DFT of v[0..7], natural order in and out.
__device__ __forceinline__ void fft8(float2 (&v)[8]) {
  float2 e0, e1, e2, e3, o0, o1, o2, o3;
  fft4(v[0], v[2], v[4], v[6], e0, e1, e2, e3);
  fft4(v[1], v[3], v[5], v[7], o0, o1, o2, o3);
  o1 = rot32<4>(o1);
  o2 = rot32<8>(o2);
  o3 = rot32<12>(o3);
  v[0] = cadd(e0, o0); v[4] = csub(e0, o0);
  v[1] = cadd(e1, o1); v[5] = csub(e1, o1);
  v[2] = cadd(e2, o2); v[6] = csub(e2, o2);
  v[3] = cadd(e3, o3); v[7] = csub(e3, o3);
}

template <int B>
__device__ __forceinline__ void fft32_column(const float2 (&x)[32], float2 (&y)[32]) {
  float2 r0, r1, r2, r3;
  fft4(x[B], x[8 + B], x[16 + B], x[24 + B], r0, r1, r2, r3);
  y[B * 4 + 0] = r0;
  y[B * 4 + 1] = rot32<(B * 1) % 32>(r1);
  y[B * 4 + 2] = rot32<(B * 2) % 32>(r2);
  y[B * 4 + 3] = rot32<(B * 3) % 32>(r3);
}

template <int C>
__device__ __forceinline__ void fft32_row(const float2 (&y)[32], float2 (&x)[32]) {
  float2 v[8];
#pragma unroll
  for (int b = 0; b < 8; ++b) v[b] = y[b * 4 + C];
  fft8(v);
#pragma unroll
  for (int d = 0; d < 8; ++d) x[C + 4 * d] = v[d];
}

// 32-point forward DFT in registers, natural order in and out:
// n = 8a + b, k = c + 4d  ->  4-point DFTs over a, twiddle W32^(bc), 8-point over b.
// One float32 instruction per real operation.
__device__ __forceinline__ void fft32_scalar(float2 (&x)[32]) {
  float2 y[32];
  fft32_column<0>(x, y); fft32_column<1>(x, y); fft32_column<2>(x, y); fft32_column<3>(x, y);
  fft32_column<4>(x, y); fft32_column<5>(x, y); fft32_column<6>(x, y); fft32_column<7>(x, y);
  fft32_row<0>(y, x); fft32_row<1>(y, x); fft32_row<2>(y, x); fft32_row<3>(y, x);
}

// ---- packed form --------------------------------------------------------------------
// sm_100 issues float32 adds, multiplies and FMAs on register PAIRS (FADD2 / FMUL2 /
// FFMA2: two lanes per issue slot).  tools/bench_f32x2.cu shows they run at half the
// instruction rate of the scalar forms (0.49 against 0.98 per clock per scheduler): they
// free issue slots, not the FMA pipe.  Alone the packed transform takes 512 cycles per
// warp against 533 (tools/bench_fft32.cu); inside the fused STFT kernel, whose other
// phases compete for the same issue slots, it is worth 7 % (1.58 -> 1.47 ms, same box,
// back to back), so stft2048.cu calls it.  The OLS and iSTFT kernels measured slower
// with it (4.50 -> 4.55 ms, 3.43 -> 3.62 ms) and keep the scalar form.  A C2 carries two complex numbers side by side,
// the real parts in one pair and the imaginary parts in another, so that every
// butterfly -- including the rotations by -i, which only swap the roles of the two
// pairs -- runs on both at once.  The pairing is chosen so that no value ever has to
// move between pairs:
//   * columns: the 4-point DFTs over a for b and b + 4 share their first stage;
//     their second stage is written out per column (scalar adds), which lets it
//     drop its results straight into the row pairing;
//   * rows: the 8-point DFTs over b for c and c + 2 run side by side in full, and
//     so do the twiddles W32^(b c) of the pair (c = 1, c = 3).
struct C2 { float2 re, im; };

__device__ __forceinline__ float2 pk_add(float2 a, float2 b) {
  unsigned long long ra, rb, rc;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("add.f32x2 %0, %1, %2;" : "=l"(rc) : "l"(ra), "l"(rb));
  float2 r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(rc));
  return r;
}
__device__ __forceinline__ float2 pk_sub(float2 a, float2 b) {
  unsigned long long ra, rb, rc;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("sub.f32x2 %0, %1, %2;" : "=l"(rc) : "l"(ra), "l"(rb));
  float2 r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(rc));
  return r;
}
__device__ __forceinline__ float2 pk_mul(float2 a, float2 b) {
  unsigned long long ra, rb, rc;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("mul.f32x2 %0, %1, %2;" : "=l"(rc) : "l"(ra), "l"(rb));
  float2 r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(rc));
  return r;
}
__device__ __forceinline__ float2 pk_fma(float2 a, float2 b, float2 c) {
  unsigned long long ra, rb, rc, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rc) : "f"(c.x), "f"(c.y));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  float2 r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(rd));
  return r;
}
__device__ __forceinline__ C2 c2add(C2 a, C2 b) { return C2{pk_add(a.re, b.re), pk_add(a.im, b.im)}; }
__device__ __forceinline__ C2 c2sub(C2 a, C2 b) { return C2{pk_sub(a.re, b.re), pk_sub(a.im, b.im)}; }
// a + (-i) b and a - (-i) b:  -i (x + i y) = y - i x
__device__ __forceinline__ C2 c2add_mi(C2 a, C2 b) { return C2{pk_add(a.re, b.im), pk_sub(a.im, b.re)}; }
__device__ __forceinline__ C2 c2sub_mi(C2 a, C2 b) { return C2{pk_sub(a.re, b.im), pk_add(a.im, b.re)}; }

__device__ __forceinline__ void fft4p(C2 a0, C2 a1, C2 a2, C2 a3, C2& x0, C2& x1, C2& x2, C2& x3) {
  const C2 t0 = c2add(a0, a2), t1 = c2sub(a0, a2), t2 = c2add(a1, a3), d = c2sub(a1, a3);
  x0 = c2add(t0, t2);
  x2 = c2sub(t0, t2);
  x1 = c2add_mi(t1, d);
  x3 = c2sub_mi(t1, d);
}

// two 8-point forward DFTs side by side, natural order in and out
__device__ __forceinline__ void fft8p(C2 (&v)[8]) {
  C2 e0, e1, e2, e3, o0, o1, o2, o3;
  fft4p(v[0], v[2], v[4], v[6], e0, e1, e2, e3);
  fft4p(v[1], v[3], v[5], v[7], o0, o1, o2, o3);
  const float r = 0.7071067811865476f;
  const float2 rr = make_float2(r, r), nr = make_float2(-r, -r);
  // o1 W8^1 = ((x + y) r, (y - x) r);  o3 W8^3 = ((y - x) r, -(x + y) r);  o2 W8^2 = -i o2
  const C2 p1 = C2{pk_mul(pk_add(o1.re, o1.im), rr), pk_mul(pk_sub(o1.im, o1.re), rr)};
  const C2 p3 = C2{pk_mul(pk_sub(o3.im, o3.re), rr), pk_mul(pk_add(o3.re, o3.im), nr)};
  v[0] = c2add(e0, o0);    v[4] = c2sub(e0, o0);
  v[1] = c2add(e1, p1);    v[5] = c2sub(e1, p1);
  v[2] = c2add_mi(e2, o2); v[6] = c2sub_mi(e2, o2);
  v[3] = c2add(e3, p3);    v[7] = c2sub(e3, p3);
}

// columns b = B and B + 4: shared first stage (packed), second stage and the
// twiddles W32^(b c) per column, results in the row pairing (c, c + 2)
template <int B>
__device__ __forceinline__ void fft32p_columns(const float2 (&x)[32], C2 (&v02)[8], C2 (&v13)[8]) {
  C2 a[4];
#pragma unroll
  for (int q = 0; q < 4; ++q)
    a[q] = C2{make_float2(x[8 * q + B].x, x[8 * q + B + 4].x), make_float2(x[8 * q + B].y, x[8 * q + B + 4].y)};
  const C2 t0 = c2add(a[0], a[2]), t1 = c2sub(a[0], a[2]), t2 = c2add(a[1], a[3]), d = c2sub(a[1], a[3]);
  {  // column B (the low halves)
    const float2 y0 = make_float2(t0.re.x + t2.re.x, t0.im.x + t2.im.x);
    const float2 y2 = rot32<(2 * B) % 32>(make_float2(t0.re.x - t2.re.x, t0.im.x - t2.im.x));
    const float2 y1 = make_float2(t1.re.x + d.im.x, t1.im.x - d.re.x);
    const float2 y3 = make_float2(t1.re.x - d.im.x, t1.im.x + d.re.x);
    v02[B] = C2{make_float2(y0.x, y2.x), make_float2(y0.y, y2.y)};
    v13[B] = C2{make_float2(y1.x, y3.x), make_float2(y1.y, y3.y)};
  }
  {  // column B + 4 (the high halves)
    const float2 y0 = make_float2(t0.re.y + t2.re.y, t0.im.y + t2.im.y);
    const float2 y2 = rot32<(2 * (B + 4)) % 32>(make_float2(t0.re.y - t2.re.y, t0.im.y - t2.im.y));
    const float2 y1 = make_float2(t1.re.y + d.im.y, t1.im.y - d.re.y);
    const float2 y3 = make_float2(t1.re.y - d.im.y, t1.im.y + d.re.y);
    v02[B + 4] = C2{make_float2(y0.x, y2.x), make_float2(y0.y, y2.y)};
    v13[B + 4] = C2{make_float2(y1.x, y3.x), make_float2(y1.y, y3.y)};
  }
}
// (y1, y3) of column b times (W32^b, W32^(3b)), both at once
template <int B>
__device__ __forceinline__ void twiddle13(C2& v) {
  if constexpr (B == 0) return;
  constexpr float c1 = kW32C[B], s1 = kW32S[B], c3 = kW32C[(3 * B) % 32], s3 = kW32S[(3 * B) % 32];
  const float2 C = make_float2(c1, c3), S = make_float2(s1, s3), nS = make_float2(-s1, -s3);
  const float2 re = pk_fma(v.im, nS, pk_mul(v.re, C));
  const float2 im = pk_fma(v.im, C, pk_mul(v.re, S));
  v = C2{re, im};
}

__device__ __forceinline__ void fft32_packed(float2 (&x)[32]) {
  C2 v02[8], v13[8];
  fft32p_columns<0>(x, v02, v13); fft32p_columns<1>(x, v02, v13);
  fft32p_columns<2>(x, v02, v13); fft32p_columns<3>(x, v02, v13);
  twiddle13<1>(v13[1]); twiddle13<2>(v13[2]); twiddle13<3>(v13[3]); twiddle13<4>(v13[4]);
  twiddle13<5>(v13[5]); twiddle13<6>(v13[6]); twiddle13<7>(v13[7]);
  fft8p(v02);
  fft8p(v13);
#pragma unroll
  for (int d = 0; d < 8; ++d) {
    x[4 * d + 0] = make_float2(v02[d].re.x, v02[d].im.x);
    x[4 * d + 2] = make_float2(v02[d].re.y, v02[d].im.y);
    x[4 * d + 1] = make_float2(v13[d].re.x, v13[d].im.x);
    x[4 * d + 3] = make_float2(v13[d].re.y, v13[d].im.y);
  }
}

// The transform the kernels call (-DSMB_FFT32_PACKED=1 selects the packed form).
__device__ __forceinline__ void fft32(float2 (&x)[32]) {
#if defined(SMB_FFT32_PACKED) && SMB_FFT32_PACKED
  fft32_packed(x);
#else
  fft32_scalar(x);
#endif
}

// Forward complex FFT of 1024 points spread over a warp, as 32 x 32 with the twiddle
// W_1024^(k1 n2) and one transposition through the warp's padded buffer `ex`
// ([32][kFft1024ExStride] complex): in, lane = n mod 32 and register = n div 32; out,
// lane = k mod 32 and register = k div 32.  tw4 holds the twiddles as
// [16][32] x (k1, k1 + 1) pairs.
constexpr int kFft1024ExStride = 34;   // padded transpose row (complex)
__device__ __forceinline__ void fft1024(float2 (&a)[32], float2* ex, const float4* tw4, int lane) {
  fft32(a);                                     // a[k1] = Y[n2 = lane][k1]
#pragma unroll
  for (int k1 = 0; k1 < 32; k1 += 2) {          // twiddle W_1024^(k1 n2), transpose
    const float4 t = tw4[(k1 >> 1) * 32 + lane];
    ex[k1 * kFft1024ExStride + lane] =
        k1 == 0 ? a[0] : make_float2(a[k1].x * t.x - a[k1].y * t.y, a[k1].x * t.y + a[k1].y * t.x);
    ex[(k1 + 1) * kFft1024ExStride + lane] = make_float2(a[k1 + 1].x * t.z - a[k1 + 1].y * t.w,
                                                         a[k1 + 1].x * t.w + a[k1 + 1].y * t.z);
  }
  __syncwarp();
  const float4* e4 = reinterpret_cast<const float4*>(ex + lane * kFft1024ExStride);
#pragma unroll
  for (int n2 = 0; n2 < 32; n2 += 2) {
    const float4 v = e4[n2 >> 1];
    a[n2] = make_float2(v.x, v.y);
    a[n2 + 1] = make_float2(v.z, v.w);
  }
  __syncwarp();
  fft32(a);                                     // a[k2] = Z[lane + 32 k2]
}

}  // namespace fft32impl
}  // namespace smb
