// ubench_tap_mma.cu — the 2x EASU tap loop with its accumulate on the FMA pipe (production quad_pair, fsr1_easu_quad.cuh)
// against the same loop with the accumulate moved to the tensor pipe (mma.sync m16n8k16, fp32 accumulators).
// Both variants compute the same d2 and window weights; they differ only in how sum_tap w * (R,G,B,1) is formed.
//
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o /tmp/ubench_tap_mma tools/ubench_tap_mma.cu && /tmp/ubench_tap_mma
//
// Geometry (one warp = one row of 32 cells = 64 output pixels per output row, as in easu_h_quad2x_kernel):
//   group  8 consecutive lanes (cells); its 16 output pixels of one row are the M = 16 rows of the MMA.
//   K      pixel block b (cells 4b .. 4b+3, 8 pixels) has its own 24 texels (4 rows x 7 columns without the 4 corners
//          no cell of the block reads), so A is block-diagonal: K = 48 = 3 k16 steps, 6 of the 12 8x8 sub-tiles of A
//          are zero and are not loaded.  Texel k of block b: row R, column c' (+4b), kidx = off(R) + c', off = -1,5,12,18.
//   W      lane (b, c') stores its half2 (wA, wB) of tap (R,K) with one STS.32 at base(lane) + (off(R)+K)*16: the
//          per-lane base folds in c', so every store uses an immediate offset.  Blocks are 400 B apart: the 32 lanes'
//          stores of one tap hit 32 different banks.  Entries no cell writes stay zero from the initial fill.
//   B      a 16-byte copy (R,G,B,1,0,0,0,0) of every texel: ldmatrix.trans rows; channel 3 makes the MMA return sum w.
//          Loaded once per cell row, used by the top and the bottom output row.
//   D      (R,G | B,sum w) of pixels g, g+8 at lanes t = 0 / 1; staged through shared memory (STS.64) and read back by
//          the lane that owns the cell (2 x LDS.128), which normalises in fp32 and applies the de-ringing clamp.
//
// The timed kernels run 4 warps per CTA at 6 CTAs per SM over a persistent grid; each warp loops over cell rows of a
// tile held in shared memory.  The program also checks that both variants give the same pixels (to half rounding of the
// accumulators) and prints the largest difference.
#include <cstdio>
#include <cstdint>
#include <cmath>
#include <vector>
#include "../fidelityfx-fsr_b200/csrc/fsr1_easu_quad.cuh"

using namespace fsr1;

constexpr int NW = 4, kCtasPerSm = 6, kRowsPerWarp = 4096, kTW = 40;
constexpr int kOff[4] = {-1, 5, 12, 18};

struct __align__(128) Smem {
  uint2 tile[NW][4][kTW];
  uint4 X[NW][4][kTW];
  __align__(16) unsigned char W[NW][8 * 400];
  float4 O[NW][4][16];
};

__device__ __forceinline__ float hrand(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  return (x & 0xffffff) * (1.0f / 16777216.0f);
}

__device__ __forceinline__ void ldsm_x2_t(uint32_t& r0, uint32_t& r1, uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr));
}
__device__ __forceinline__ void mma16816(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// the 12 window weights of the pixel pair of one output row, stored to W (same d2 / weight arithmetic as quad_pair)
template <bool kBottom>
__device__ __forceinline__ void store_weights(const ShapeH& s, uint32_t wbase) {
  const __half2 qa = s.qa, qb = s.qb, qc = s.qc, lob = s.lob, clp = s.clp;
  constexpr float py = kBottom ? 0.75f : 0.25f;
#define TW_STORE(R, K, W) asm volatile("st.shared.b32 [%0+%1], %2;" ::"r"(wbase), "n"((kOff[R] + (K)) * 16), "r"(h22u(W)) : "memory");
#define TW_TAP(R, K)                                                                                            \
  {                                                                                                             \
    constexpr float oxA = (float)((K)-1) - 0.25f, oxB = (float)((K)-1) - 0.75f, oy = (float)((R)-1) - py;         \
    const __half2 d2 = __hfma2(qa, __floats2half2_rn(oxA * oxA, oxB * oxB),                                      \
                               __hfma2(qc, __floats2half2_rn(oy * oy, oy * oy), __hmul2(qb, __floats2half2_rn(oxA * oy, oxB * oy)))); \
    TW_STORE(R, K, tap_weight(d2, lob, clp))                                                                    \
  }
#define TW_ROW(R, K, INNER)                                                                                     \
  {                                                                                                             \
    constexpr float oxA = (float)((K)-1) - 0.25f, oxB = (float)((K)-1) - 0.75f;                                   \
    const __half2 ox = __floats2half2_rn(oxA, oxB);                                                             \
    const __half2 d2 = __hfma2(__hfma2(qa, ox, rowB##R), ox, rowC##R);                                           \
    TW_STORE(R, K, (INNER) ? tap_weight_unclamped(d2, lob) : tap_weight(d2, lob, clp))                          \
  }
  constexpr float oy1 = 0.0f - py, oy2 = 1.0f - py;
  const __half2 rowB1 = __hmul2(qb, h2c(oy1)), rowC1 = __hmul2(qc, h2c(oy1 * oy1));
  const __half2 rowB2 = __hmul2(qb, h2c(oy2)), rowC2 = __hmul2(qc, h2c(oy2 * oy2));
  TW_TAP(0, 1) TW_TAP(0, 2) TW_ROW(1, 0, false) TW_ROW(1, 3, false) TW_ROW(2, 0, false) TW_ROW(2, 3, false)
  TW_TAP(3, 1) TW_TAP(3, 2) TW_ROW(1, 1, true) TW_ROW(1, 2, true) TW_ROW(2, 1, true) TW_ROW(2, 2, true)
#undef TW_ROW
#undef TW_TAP
#undef TW_STORE
}

// one output row of the warp's 32 cells through the tensor pipe; returns this lane's pixel pair, clamped
template <bool kBottom>
__device__ __forceinline__ void mma_row(const ShapeH& s, uint32_t wbase, uint32_t wwarp, const uint32_t (&aoff)[3],
                                        const uint32_t (&b)[4][3][2], float4* Ow, int lane, __half2 mnR, __half2 mnG,
                                        __half2 mnB, __half2 mxR, __half2 mxG, __half2 mxB, __half2& oR, __half2& oG, __half2& oB) {
  store_weights<kBottom>(s, wbase);
  __syncwarp();
#pragma unroll
  for (int gi = 0; gi < 4; gi++) {
    float d[4] = {0.f, 0.f, 0.f, 0.f};
    uint32_t x0, x1;
    const uint32_t wg = wwarp + gi * 800;
    ldsm_x2_t(x0, x1, wg + aoff[0]);  // block 0 rows 0-7 -> a0, rows 8-15 -> a2
    mma16816(d, x0, 0u, x1, 0u, b[gi][0][0], b[gi][0][1]);
    ldsm_x2_t(x0, x1, wg + aoff[1]);  // block 0 rows 16-23 -> a0, block 1 rows 0-7 -> a3
    mma16816(d, x0, 0u, 0u, x1, b[gi][1][0], b[gi][1][1]);
    ldsm_x2_t(x0, x1, wg + aoff[2]);  // block 1 rows 8-15 -> a1, rows 16-23 -> a3
    mma16816(d, 0u, x0, 0u, x1, b[gi][2][0], b[gi][2][1]);
    const int g = lane >> 2, t = lane & 3;
    if (t < 2) {
      reinterpret_cast<float2*>(&Ow[gi * 16 + g])[t] = make_float2(d[0], d[1]);
      reinterpret_cast<float2*>(&Ow[gi * 16 + g + 8])[t] = make_float2(d[2], d[3]);
    }
  }
  __syncwarp();
  const float4 pA = Ow[(lane >> 3) * 16 + 2 * (lane & 7)], pB = Ow[(lane >> 3) * 16 + 2 * (lane & 7) + 1];
  __syncwarp();
  const float rA = rcp_approx(pA.w), rB = rcp_approx(pB.w);
  oR = __hmin2(mxR, __hmax2(mnR, __floats2half2_rn(pA.x * rA, pB.x * rB)));
  oG = __hmin2(mxG, __hmax2(mnG, __floats2half2_rn(pA.y * rA, pB.y * rB)));
  oB = __hmin2(mxB, __hmax2(mnB, __floats2half2_rn(pA.z * rA, pB.z * rB)));
}

template <bool kMma>
__global__ void __launch_bounds__(NW * 32, kCtasPerSm) tap_kernel(uint32_t* out, uint32_t* first, int rows, uint32_t eps_bits) {
  __shared__ Smem sm;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < NW * 4 * kTW; i += NW * 32) {
    const uint32_t h = blockIdx.x * 7919u + i * 131u;
    const __half2 rg = __floats2half2_rn(hrand(h), hrand(h + 1)), ba = __floats2half2_rn(hrand(h + 2), 1.0f);
    (&sm.tile[0][0][0])[i] = make_uint2(h22u(rg), h22u(ba));
    (&sm.X[0][0][0])[i] = make_uint4(h22u(rg), (h22u(ba) & 0xffffu) | 0x3c000000u, 0u, 0u);
  }
  for (int i = tid; i < NW * 8 * 400 / 4; i += NW * 32) reinterpret_cast<uint32_t*>(&sm.W[0][0])[i] = 0u;
  __syncthreads();
  // per-lane filter shape (fp32 analysis of the production kernel on random terms), rounded to half once
  const uint32_t seed = (blockIdx.x * NW + warp) * 32 + lane;
  const float2 dx = mk2(hrand(seed * 3) - 0.5f, hrand(seed * 3 + 7) - 0.5f), dy = mk2(hrand(seed * 5 + 1) - 0.5f, hrand(seed * 5 + 9) - 0.5f);
  const float2 len = mk2(hrand(seed * 11), hrand(seed * 11 + 3));
  ShapeH s = to_half(pixel_shape2(dx, dy, len));
  const __half2 eps = u2h2(eps_bits);  // 0 at run time: keeps the shape a loop-carried value
  const uint2* t0 = &sm.tile[warp][0][lane];
  uint32_t sink = 0, firstv = 0;
  // tensor-pipe addressing, once per lane
  const int gi = lane >> 3, c = lane & 7, bk = c >> 2, cp = c & 3;
  const uint32_t wwarp = smem_u32(&sm.W[warp][0]);
  const uint32_t wbase = wwarp + (2 * gi + bk) * 400 + cp * 20;
  uint32_t aoff[3];
  {
    const int j = (lane >> 3) & 1, i = lane & 7;
    aoff[0] = (8 * j + i) * 16;
    aoff[1] = j ? 400 + i * 16 : (16 + i) * 16;
    aoff[2] = 400 + (8 + 8 * j + i) * 16;
  }
  uint32_t boff[3];  // texel of K row (lane & 15) of each k16 step, relative to the group's first texel column
#pragma unroll
  for (int st = 0; st < 3; st++) {
    const int k = 16 * st + (lane & 15), blk = k >= 24 ? 1 : 0, kk = k - 24 * blk;
    const int R = kk < 5 ? 0 : kk < 12 ? 1 : kk < 19 ? 2 : 3;
    boff[st] = (uint32_t)(R * kTW + 4 * blk + kk - (R == 0 ? -1 : R == 1 ? 5 : R == 2 ? 12 : 18)) * 16u;
  }
  const uint32_t xwarp = smem_u32(&sm.X[warp][0][0]);
  float4* Ow = &sm.O[warp][0][0];
#pragma unroll 1
  for (int it = 0; it < rows; it++) {
    s.qa = __hadd2(s.qa, eps);
    __half2 oR, oG, oB;
    uint32_t v = 0;
    if (!kMma) {
      uint2 tp[4][4];
#pragma unroll
      for (int R = 0; R < 4; R++)
#pragma unroll
        for (int K = 0; K < 4; K++)
          if (!((R == 0 || R == 3) && (K == 0 || K == 3))) tp[R][K] = t0[R * kTW + K];
      const __half2 mnRG = __hmin2(__hmin2(u2h2(tp[1][1].x), u2h2(tp[1][2].x)), __hmin2(u2h2(tp[2][1].x), u2h2(tp[2][2].x)));
      const __half2 mxRG = __hmax2(__hmax2(u2h2(tp[1][1].x), u2h2(tp[1][2].x)), __hmax2(u2h2(tp[2][1].x), u2h2(tp[2][2].x)));
      const __half2 mnBA = __hmin2(__hmin2(u2h2(tp[1][1].y), u2h2(tp[1][2].y)), __hmin2(u2h2(tp[2][1].y), u2h2(tp[2][2].y)));
      const __half2 mxBA = __hmax2(__hmax2(u2h2(tp[1][1].y), u2h2(tp[1][2].y)), __hmax2(u2h2(tp[2][1].y), u2h2(tp[2][2].y)));
      quad_pair<false>(tp, s, __low2half2(mnRG), __high2half2(mnRG), __low2half2(mnBA), __low2half2(mxRG), __high2half2(mxRG), __low2half2(mxBA), oR, oG, oB);
      v ^= h22u(oR) * 3u ^ h22u(oG) * 5u ^ h22u(oB) * 7u;
      if (it == 0) { first[seed * 6 + 0] = h22u(oR); first[seed * 6 + 1] = h22u(oG); first[seed * 6 + 2] = h22u(oB); }
      quad_pair<true>(tp, s, __low2half2(mnRG), __high2half2(mnRG), __low2half2(mnBA), __low2half2(mxRG), __high2half2(mxRG), __low2half2(mxBA), oR, oG, oB);
    } else {
      const uint2 f = t0[kTW + 1], g = t0[kTW + 2], j = t0[2 * kTW + 1], k = t0[2 * kTW + 2];
      const __half2 mnRG = __hmin2(__hmin2(u2h2(f.x), u2h2(g.x)), __hmin2(u2h2(j.x), u2h2(k.x)));
      const __half2 mxRG = __hmax2(__hmax2(u2h2(f.x), u2h2(g.x)), __hmax2(u2h2(j.x), u2h2(k.x)));
      const __half2 mnBA = __hmin2(__hmin2(u2h2(f.y), u2h2(g.y)), __hmin2(u2h2(j.y), u2h2(k.y)));
      const __half2 mxBA = __hmax2(__hmax2(u2h2(f.y), u2h2(g.y)), __hmax2(u2h2(j.y), u2h2(k.y)));
      uint32_t b[4][3][2];
#pragma unroll
      for (int q = 0; q < 4; q++)
#pragma unroll
        for (int st = 0; st < 3; st++) ldsm_x2_t(b[q][st][0], b[q][st][1], xwarp + q * 8 * 16 + boff[st]);
      mma_row<false>(s, wbase, wwarp, aoff, b, Ow, lane, __low2half2(mnRG), __high2half2(mnRG), __low2half2(mnBA),
                     __low2half2(mxRG), __high2half2(mxRG), __low2half2(mxBA), oR, oG, oB);
      v ^= h22u(oR) * 3u ^ h22u(oG) * 5u ^ h22u(oB) * 7u;
      if (it == 0) { first[seed * 6 + 0] = h22u(oR); first[seed * 6 + 1] = h22u(oG); first[seed * 6 + 2] = h22u(oB); }
      mma_row<true>(s, wbase, wwarp, aoff, b, Ow, lane, __low2half2(mnRG), __high2half2(mnRG), __low2half2(mnBA),
                    __low2half2(mxRG), __high2half2(mxRG), __low2half2(mxBA), oR, oG, oB);
    }
    v ^= h22u(oR) * 11u ^ h22u(oG) * 13u ^ h22u(oB) * 17u;
    if (it == 0) { firstv = 1; first[seed * 6 + 3] = h22u(oR); first[seed * 6 + 4] = h22u(oG); first[seed * 6 + 5] = h22u(oB); }
    sink += v;
  }
  out[seed] = sink + firstv;
}

static float h2f_host(uint16_t h) {
  const uint32_t s = (h >> 15) & 1, e = (h >> 10) & 31, m = h & 1023;
  float v = e == 0 ? ldexpf((float)m, -24) : e == 31 ? INFINITY : ldexpf((float)(m | 1024), (int)e - 25);
  return s ? -v : v;
}

int main() {
  int sms = 0, khz = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, 0);
  const int grid = sms * kCtasPerSm, lanes = grid * NW * 32;
  uint32_t *out, *first[2];
  cudaMalloc(&out, lanes * 4);
  cudaMalloc(&first[0], lanes * 24);
  cudaMalloc(&first[1], lanes * 24);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  printf("device SMs %d, nominal SM clock %.0f MHz; %d CTAs x %d warps, %d cell rows per warp (2 output rows each)\n", sms,
         khz / 1e3, grid, NW, kRowsPerWarp);
  float best[2] = {1e30f, 1e30f};
  for (int rep = 0; rep < 5; rep++)
    for (int v = 0; v < 2; v++) {
      cudaEventRecord(e0);
      if (v) tap_kernel<true><<<grid, NW * 32>>>(out, first[1], kRowsPerWarp, 0u);
      else tap_kernel<false><<<grid, NW * 32>>>(out, first[0], kRowsPerWarp, 0u);
      cudaEventRecord(e1);
      cudaEventSynchronize(e1);
      float ms = 0;
      cudaEventElapsedTime(&ms, e0, e1);
      if (cudaGetLastError() != cudaSuccess) { printf("launch failed\n"); return 1; }
      if (ms < best[v]) best[v] = ms;
    }
  const double quads = (double)lanes * kRowsPerWarp;  // one lane-iteration = one quad (4 output pixels)
  for (int v = 0; v < 2; v++)
    printf("%-34s best of 5: %8.3f ms  %7.2f Gpix/s  %6.2f ns per warp cell-row  (%5.1f SM cycles at nominal clock)\n",
           v ? "accumulate on tensor pipe (mma)" : "accumulate on FMA pipe (HFMA2)", best[v], 4.0 * quads / (best[v] * 1e6),
           best[v] * 1e6 / (quads / 32.0 / sms), best[v] * 1e-3 * khz * 1e3 / (quads / 32.0 / sms));
  std::vector<uint16_t> h0(lanes * 12), h1(lanes * 12);
  cudaMemcpy(h0.data(), first[0], lanes * 24, cudaMemcpyDeviceToHost);
  cudaMemcpy(h1.data(), first[1], lanes * 24, cudaMemcpyDeviceToHost);
  double mx = 0, sum = 0;
  for (size_t i = 0; i < h0.size(); i++) {
    const double d = fabs((double)h2f_host(h0[i]) - h2f_host(h1[i]));
    mx = d > mx ? d : mx;
    sum += d;
  }
  printf("pixels of the first cell row: max |mma - hfma2| = %.3g, mean %.3g over %zu values\n", mx, sum / h0.size(), h0.size());
  return 0;
}
