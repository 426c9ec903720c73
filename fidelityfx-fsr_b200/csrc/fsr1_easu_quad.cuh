// fsr1_easu_quad.cuh — the per-pixel half of EASU at exactly 2x, shared by the tiled EASU kernels
// (fsr1_easu_tiled.cu) and the fused EASU->RCAS kernel (fsr1_fused.cu).
//
// At 2x (con0 = {.5,.5,-.25,-.25}) the four output pixels (2k+1,2k+2)x(2m+1,2m+2) share the 4x4 tap window of input
// cell (k,m).  A lane owns that quad: it loads the 12 taps and the 4 per-texel term vectors once, every tap offset is
// a compile-time constant, and the arithmetic is packed over the horizontally adjacent pixel pair (A: px=.25, B: px=.75):
//   fp32 (f32x2: FFMA2/FMUL2/FADD2)  bilinear blend of the f,g,j,k texel terms (ffx_fsr1.h:383-386), normalise, stretch,
//                                     lobe, clip (:389-409) -> the quadratic form (qa,qb,qc), lob, clp of each pixel
//   half2                             12 taps (:423-434): d2 = qa ox^2 + qb ox oy + qc oy^2, window weight, accumulate;
//                                     de-ringing clamp (:416-419,437)
// Everything that decides the filter's ORIENTATION stays fp32 (in half it is ill-conditioned where gradients nearly
// cancel: the reference's own H path differs from its F path by up to 0.1); the taps — the bulk of the arithmetic —
// are half2 and keep the result within ~3e-3 of the fp32 oracle (tolerance 1e-2).
#pragma once
#include "fsr1_easu_common.cuh"

namespace fsr1 {

__device__ __forceinline__ float texel_luma(uint2 t) {  // 2*luma = 0.5 B + (0.5 R + G); exact in fp32
  const float2 rg = __half22float2(u2h2(t.x));
  return fmaf(__low2float(u2h2(t.y)), 0.5f, fmaf(rg.x, 0.5f, rg.y));
}

// Window weight of two pixels at squared distance d2, times 4: (25/16 (2/5 d2 - 1)^2 - 9/16)(lob d2 - 1)^2
// (ffx_fsr1.h:255-270) = (d2 - 1)(d2 - 4)(lob d2 - 1)^2 / 4.  With v = lob d2 - 1 and p = (d2 - 1) v the product is
// p (p - 3 v): four HFMA2/HMUL2 instead of five, and no rounded sum of large terms (each factor is one FMA of the exact
// d2 v).  The factor 4 is common to every tap of a pixel and cancels in the normalisation by the sum of the weights.
// The clamp min(d2, clp) is a packed 16-bit INTEGER min (VIMNMX.S16x2, integer pipe): clp > 0, so comparing the bit
// patterns as signed integers orders every non-negative d2 correctly and returns d2 itself when rounding made it slightly
// negative — identical to __hmin2 for finite inputs, off the pipe the HFMA2s use.
__device__ __forceinline__ __half2 tap_weight_unclamped(__half2 d2, __half2 lob) {
  const __half2 v = __hfma2(lob, d2, h2c(-1.0f));
  const __half2 p = __hfma2(d2, v, __hneg2(v));
  return __hmul2(p, __hfma2(v, h2c(-3.0f), p));
}
__device__ __forceinline__ __half2 tap_weight(__half2 d2, __half2 lob, __half2 clp) {
#ifdef FSR1_CPU_EMU
  const uint32_t r = emu_min_s16x2(h22u(d2), h22u(clp));
#else
  uint32_t r;
  asm("min.s16x2 %0, %1, %2;" : "=r"(r) : "r"(h22u(d2)), "r"(h22u(clp)));
#endif
  return tap_weight_unclamped(u2h2(r), lob);
}

// ---- per-pixel filter shape of a pixel PAIR in packed f32x2 (.x = pixel A, .y = pixel B) ---------------------------
// From the blended (dir, len): normalise (zro branch, APrxLoRsqF1), stretch (APrxLoRcpF1), len2, lob, clp
// (ffx_fsr1.h:389-409), then the coefficients of the rotated, anisotropically scaled distance
//   d2(ox,oy) = qa ox^2 + qb ox oy + qc oy^2,  qa = l2x^2 dx^2 + l2y^2 dy^2,  qc = l2x^2 dy^2 + l2y^2 dx^2,
//   qb = 2 dx dy (l2x^2 - l2y^2).
__device__ __forceinline__ float2 mk2(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ float2 bc2(float a) { return make_float2(a, a); }
struct Shape2 { float2 qa, qb, qc, lob, clp; };
__device__ __forceinline__ Shape2 pixel_shape2(float2 dx, float2 dy, float2 len) {
  const float2 dirR = __ffma2_rn(dx, dx, __fmul2_rn(dy, dy));
  const bool zx = dirR.x < (1.0f / 32768.0f), zy = dirR.y < (1.0f / 32768.0f);
  const float2 rs = mk2(zx ? 1.0f : prx_lo_rsq(dirR.x), zy ? 1.0f : prx_lo_rsq(dirR.y));
  dx = __fmul2_rn(mk2(zx ? 1.0f : dx.x, zy ? 1.0f : dx.y), rs);
  dy = __fmul2_rn(dy, rs);
  len = __fmul2_rn(len, bc2(0.5f));
  len = __fmul2_rn(len, len);
  const float2 dx2 = __fmul2_rn(dx, dx), dy2 = __fmul2_rn(dy, dy);
  const float2 rmax = mk2(prx_lo_rcp(fmaxf(fabsf(dx.x), fabsf(dy.x))), prx_lo_rcp(fmaxf(fabsf(dx.y), fabsf(dy.y))));
  const float2 stretch = __fmul2_rn(__fadd2_rn(dx2, dy2), rmax);
  const float2 l2x = __ffma2_rn(__fadd2_rn(stretch, bc2(-1.0f)), len, bc2(1.0f));
  const float2 l2y = __ffma2_rn(bc2(-0.5f), len, bc2(1.0f));
  Shape2 s;
  s.lob = __ffma2_rn(bc2((float)((1.0 / 4.0 - 0.04) - 0.5)), len, bc2(0.5f));
  s.clp = mk2(prx_lo_rcp(s.lob.x), prx_lo_rcp(s.lob.y));
  const float2 X2 = __fmul2_rn(l2x, l2x), Y2 = __fmul2_rn(l2y, l2y);
  s.qa = __ffma2_rn(X2, dx2, __fmul2_rn(Y2, dy2));
  s.qc = __ffma2_rn(X2, dy2, __fmul2_rn(Y2, dx2));
  s.qb = __fmul2_rn(__fmul2_rn(__fmul2_rn(dx, dy), bc2(2.0f)), __ffma2_rn(Y2, bc2(-1.0f), X2));
  return s;
}
struct ShapeH { __half2 qa, qb, qc, lob, clp; };  // the same, rounded once to half2 (pixel A, pixel B) for the tap loop
__device__ __forceinline__ ShapeH to_half(const Shape2& s) {
  return ShapeH{__floats2half2_rn(s.qa.x, s.qa.y), __floats2half2_rn(s.qb.x, s.qb.y), __floats2half2_rn(s.qc.x, s.qc.y),
                __floats2half2_rn(s.lob.x, s.lob.y), __floats2half2_rn(s.clp.x, s.clp.y)};
}

// ---- tile geometry of the 2x kernels --------------------------------------------------------------------------------
constexpr int kQCX = 32;        // cells per tile in x (= 64 output pixels); one lane per cell
constexpr int kQBW = kQCX + 4;  // TMA box width: 36 texels (35 needed, even width)
constexpr int kQSW = kQBW - 2;  // inner texels carrying terms: 34 per row
// NW warps per CTA, each warp owns 2 cell rows: cells per tile 32 x 2NW, box 36 x (2NW+3), terms 34 x (2NW+1)
template <int NW> struct QuadCfg {
  static constexpr int kCY = 2 * NW, kBH = kCY + 3, kSH = kBH - 2, kElems = kQBW * kBH;
  static constexpr int kPad = ((kElems * 8 + 127) / 128) * 128 / 8;  // buffer stride keeping 128B alignment
};

// One pixel pair (A: px=.25, B: px=.75) of the quad; kBottom selects py=.75.  t = the 12 taps (RG,BA); every tap offset is
// a constant.  Rows 0 and 3 (two taps each) use d2 = qa ox^2 + qc oy^2 + qb ox oy against immediates; rows 1 and 2 (four
// taps each) the factored form d2 = ox (qa ox + qb oy) + qc oy^2 with the row terms qb oy, qc oy^2 hoisted; the four
// nearest taps f g j k skip min(d2, clp): at exactly 2x their offsets are <= .75 per axis, so d2 <= 1.125 len2.x^2
// (1 + eps) < clp = 1/lob for every len in [0,1] (1.24 (1 + .56 len)^2 vs .94 / (.5 - .29 len)).  Far taps are
// accumulated first, the near taps (the large weights) last: 45 % less rounding error in the half accumulators.
// Returns the pair's colour per channel as (pixel A, pixel B).
template <bool kBottom>
__device__ __forceinline__ void quad_pair(const uint2 (&t)[4][4], const ShapeH& s, __half2 mnR, __half2 mnG, __half2 mnB,
                                          __half2 mxR, __half2 mxG, __half2 mxB, __half2& oR, __half2& oG, __half2& oB) {
  const __half2 qa = s.qa, qb = s.qb, qc = s.qc, lob = s.lob, clp = s.clp;
  const __half2 kZero = h2c(0.0f);
  __half2 aR = kZero, aG = kZero, aB = kZero, aW = kZero;
  constexpr float py = kBottom ? 0.75f : 0.25f;
#define FSR1_QACC(R, K, W)                                                                                  \
  {                                                                                                         \
    const __half2 w = (W);                                                                                  \
    const __half2 rg = u2h2(t[R][K].x), ba = u2h2(t[R][K].y);                                               \
    aR = __hfma2(__low2half2(rg), w, aR);                                                                   \
    aG = __hfma2(__high2half2(rg), w, aG);                                                                  \
    aB = __hfma2(__low2half2(ba), w, aB);                                                                   \
    aW = __hadd2(aW, w);                                                                                    \
  }
#define FSR1_QTAP(R, K)                                                                                     \
  {                                                                                                         \
    constexpr float oxA = (float)((K)-1) - 0.25f, oxB = (float)((K)-1) - 0.75f, oy = (float)((R)-1) - py;     \
    const __half2 d2 = __hfma2(qa, __floats2half2_rn(oxA * oxA, oxB * oxB),                                  \
                               __hfma2(qc, __floats2half2_rn(oy * oy, oy * oy),                              \
                                       __hmul2(qb, __floats2half2_rn(oxA * oy, oxB * oy))));                 \
    FSR1_QACC(R, K, tap_weight(d2, lob, clp))                                                               \
  }
#define FSR1_QTAP_ROW(R, K, INNER)                                                                          \
  {                                                                                                         \
    constexpr float oxA = (float)((K)-1) - 0.25f, oxB = (float)((K)-1) - 0.75f;                               \
    const __half2 ox = __floats2half2_rn(oxA, oxB);                                                         \
    const __half2 d2 = __hfma2(__hfma2(qa, ox, rowB##R), ox, rowC##R);                                       \
    FSR1_QACC(R, K, (INNER) ? tap_weight_unclamped(d2, lob) : tap_weight(d2, lob, clp))                     \
  }
  constexpr float oy1 = 0.0f - py, oy2 = 1.0f - py;
  const __half2 rowB1 = __hmul2(qb, h2c(oy1)), rowC1 = __hmul2(qc, h2c(oy1 * oy1));
  const __half2 rowB2 = __hmul2(qb, h2c(oy2)), rowC2 = __hmul2(qc, h2c(oy2 * oy2));
  FSR1_QTAP(0, 1) FSR1_QTAP(0, 2) FSR1_QTAP_ROW(1, 0, false) FSR1_QTAP_ROW(1, 3, false)
  FSR1_QTAP_ROW(2, 0, false) FSR1_QTAP_ROW(2, 3, false) FSR1_QTAP(3, 1) FSR1_QTAP(3, 2)
  FSR1_QTAP_ROW(1, 1, true) FSR1_QTAP_ROW(1, 2, true) FSR1_QTAP_ROW(2, 1, true) FSR1_QTAP_ROW(2, 2, true)
#undef FSR1_QTAP_ROW
#undef FSR1_QTAP
#undef FSR1_QACC
  const float2 aWf = __half22float2(aW);
  const __half2 r = __floats2half2_rn(rcp_approx(aWf.x), rcp_approx(aWf.y));
  oR = __hmin2(mxR, __hmax2(mnR, __hmul2(aR, r)));
  oG = __hmin2(mxG, __hmax2(mnG, __hmul2(aG, r)));
  oB = __hmin2(mxB, __hmax2(mnB, __hmul2(aB, r)));
}

// ---- where a quad's pixels go -----------------------------------------------------------------------------------------
// RGBA16F (8 B/px) or UNORM (4 B/px) rows of a global image; alpha = 1 (FSR_Pass.hlsl:80)
struct StoreHalf {
  static constexpr int kBpp = 8;
  static __device__ __forceinline__ void put(unsigned char* o, uint2 v, bool ok) {
    if (ok) *reinterpret_cast<uint2*>(o) = v;
  }
};
// kBits = 8: R8G8B8A8_UNORM, 10: R10G10B10A2_UNORM.  x * (2^n - 1) + 1024 lands in [1024, 2048), where the ulp of a half
// is 1: one HFMA2 rounds to the nearest code value and leaves it in the low mantissa bits (alpha 1.0 -> all ones).
template <int kBits> struct StoreUnorm {
  static constexpr int kBpp = 4;
  static __device__ __forceinline__ void put(unsigned char* o, uint2 v, bool ok) {
    const __half2 sc = h2c(kBits == 8 ? 255.0f : 1023.0f), k1024 = h2c(1024.0f);
    const uint32_t t0 = h22u(__hfma2(u2h2(v.x), sc, k1024)), t1 = h22u(__hfma2(u2h2(v.y), sc, k1024));
    uint32_t w;
    if (kBits == 8) w = __byte_perm(t0, t1, 0x6420);  // R, G = bytes 0, 2 of t0; B, A = bytes 0, 2 of t1
    else w = (t0 & 0x3ffu) | (((t0 >> 16) & 0x3ffu) << 10) | ((t1 & 0x3ffu) << 20) | 0xC0000000u;
    if (ok) *reinterpret_cast<uint32_t*>(o) = w;
  }
};
template <typename ST> struct GlobalSink {
  unsigned char* row;  // address of pixel A of the quad's TOP row
  long long pitch;
  bool okA, okB;
  __device__ __forceinline__ void put(bool bottom, __half2 oR, __half2 oG, __half2 oB) const {
    const __half2 one = h2c(1.0f);
    unsigned char* o = row + (bottom ? pitch : 0);
    ST::put(o, make_uint2(h22u(__lows2half2(oR, oG)), h22u(__lows2half2(oB, one))), okA);
    ST::put(o + ST::kBpp, make_uint2(h22u(__highs2half2(oR, oG)), h22u(__highs2half2(oB, one))), okB);
  }
};

// The quad of cell (lane, r) of a tile: taps from `tile` (row pitch kPitch texels), per-texel terms from S (row pitch kSPitch).
// doTop / doBottom select the output rows 2m+1 / 2m+2; the sink receives each row's pixel pair.
template <typename Sink, int kPitch = kQBW, int kSPitch = kQSW>
__device__ __forceinline__ void quad_compute(const uint2* __restrict__ tile, const float4* __restrict__ S, int lane, int r,
                                             bool doTop, bool doBottom, const Sink& sink) {
  uint2 tp[4][4];
  const uint2* t0 = tile + r * kPitch + lane;
#pragma unroll
  for (int R = 0; R < 4; R++)
#pragma unroll
    for (int K = 0; K < 4; K++)
      if (!((R == 0 || R == 3) && (K == 0 || K == 3))) tp[R][K] = t0[R * kPitch + K];
  const float4* s0 = S + r * kSPitch + lane;
  const float4 f = s0[0], g = s0[1], j = s0[kSPitch], k = s0[kSPitch + 1];
  // de-ringing bounds of the quad: min/max of f,g,j,k per channel, broadcast to both lanes
  const __half2 mnRG = __hmin2(__hmin2(u2h2(tp[1][1].x), u2h2(tp[1][2].x)), __hmin2(u2h2(tp[2][1].x), u2h2(tp[2][2].x)));
  const __half2 mxRG = __hmax2(__hmax2(u2h2(tp[1][1].x), u2h2(tp[1][2].x)), __hmax2(u2h2(tp[2][1].x), u2h2(tp[2][2].x)));
  const __half2 mnBA = __hmin2(__hmin2(u2h2(tp[1][1].y), u2h2(tp[1][2].y)), __hmin2(u2h2(tp[2][1].y), u2h2(tp[2][2].y)));
  const __half2 mxBA = __hmax2(__hmax2(u2h2(tp[1][1].y), u2h2(tp[1][2].y)), __hmax2(u2h2(tp[2][1].y), u2h2(tp[2][2].y)));
  const __half2 mnR = __low2half2(mnRG), mnG = __high2half2(mnRG), mnB = __low2half2(mnBA);
  const __half2 mxR = __low2half2(mxRG), mxG = __high2half2(mxRG), mxB = __low2half2(mxBA);
  // packed pair (A: px=.25, B: px=.75): T = top texel row f,g blended horizontally, Bm = bottom texel row j,k
  // (blend order f,g,j,k as in the reference, ffx_fsr1.h:383-386)
  const float2 wF = mk2(0.75f, 0.25f), wG = mk2(0.25f, 0.75f);
  const float2 Tx = __ffma2_rn(bc2(g.x), wG, __fmul2_rn(bc2(f.x), wF)), Ty = __ffma2_rn(bc2(g.y), wG, __fmul2_rn(bc2(f.y), wF));
  const float2 Tz = __ffma2_rn(bc2(g.z), wG, __fmul2_rn(bc2(f.z), wF));
  const float2 Bx = __ffma2_rn(bc2(k.x), wG, __fmul2_rn(bc2(j.x), wF)), By = __ffma2_rn(bc2(k.y), wG, __fmul2_rn(bc2(j.y), wF));
  const float2 Bz = __ffma2_rn(bc2(k.z), wG, __fmul2_rn(bc2(j.z), wF));
  __half2 oR, oG, oB;
  if (doTop) {
    const ShapeH s = to_half(pixel_shape2(__ffma2_rn(Bx, bc2(0.25f), __fmul2_rn(Tx, bc2(0.75f))),
                                          __ffma2_rn(By, bc2(0.25f), __fmul2_rn(Ty, bc2(0.75f))),
                                          __ffma2_rn(Bz, bc2(0.25f), __fmul2_rn(Tz, bc2(0.75f)))));
    quad_pair<false>(tp, s, mnR, mnG, mnB, mxR, mxG, mxB, oR, oG, oB);
    sink.put(false, oR, oG, oB);
  }
  if (doBottom) {
    const ShapeH s = to_half(pixel_shape2(__ffma2_rn(Bx, bc2(0.75f), __fmul2_rn(Tx, bc2(0.25f))),
                                          __ffma2_rn(By, bc2(0.75f), __fmul2_rn(Ty, bc2(0.25f))),
                                          __ffma2_rn(Bz, bc2(0.75f), __fmul2_rn(Tz, bc2(0.25f)))));
    quad_pair<true>(tp, s, mnR, mnG, mnB, mxR, mxG, mxB, oR, oG, oB);
    sink.put(true, oR, oG, oB);
  }
}

// Phase 3 for one lane and one cell row r of a tile whose box origin is (gx0, gy0): the quad of output pixels
// (2k+1,2k+2)x(2m+1,2m+2) of cell k = gx0+1+lane, m = gy0+1+r, stored to the output image.
// kFast: the tile lies strictly inside the image and the row range, so every bounds predicate is true and is dropped at
// compile time (tile-uniform branch in the kernels).
template <bool kFast, typename ST = StoreHalf>
__device__ __forceinline__ void quad_cell(const EasuParams& p, const uint2* __restrict__ tile, const float4* __restrict__ S,
                                          int gx0, int gy0, int lane, int r) {
  const int oxA = (gx0 + 1 + lane) * 2 + 1;  // cell k = gx0 + 1 + lane -> output columns 2k+1, 2k+2
  const int oyT = (gy0 + 1 + r) * 2 + 1;     // output rows 2m+1 (top pair), 2m+2 (bottom pair)
  const bool rowT = kFast || (oyT >= p.y0 && oyT < p.y1), rowB = kFast || (oyT + 1 >= p.y0 && oyT + 1 < p.y1);
  if (!kFast && (oxA >= p.out.w || !(rowT || rowB))) return;
  GlobalSink<ST> sink;
  sink.row = p.out.base + (long long)(oyT - p.out.row0) * p.out.pitch + (long long)oxA * ST::kBpp;
  sink.pitch = p.out.pitch;
  sink.okA = kFast || oxA >= 0;
  sink.okB = kFast || oxA + 1 < p.out.w;
  quad_compute(tile, S, lane, r, rowT, rowB, sink);
}

// Zero-filled out-of-image texels of a TMA box -> clamp-to-edge (the reference samples through a CLAMP sampler,
// sample/src/DX12/FSR_Filter.cpp:48-53).  Sources are always in-image positions (never rewritten), destinations always
// out-of-image ones (never read), so no intermediate barrier.  T = texel type, `stride` = row pitch of the buffer in texels.
template <typename T>
__device__ __forceinline__ void clamp_fixup(T* tile, int stride, int BW, int BH, int gx0, int gy0, int W, int H, int lane, int warp,
                                            int nwarps) {
  for (int j = warp; j < BH; j += nwarps) {
    const int cy = clampi(gy0 + j, 0, H - 1) - gy0;
    for (int i = lane; i < BW; i += 32) {
      const int cx = clampi(gx0 + i, 0, W - 1) - gx0;
      if ((cx != i || cy != j) && cx >= 0 && cx < BW && cy >= 0 && cy < BH) tile[j * stride + i] = tile[cy * stride + cx];
    }
  }
}

}  // namespace fsr1
