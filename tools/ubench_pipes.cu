// ubench_pipes.cu — issue-rate microbenchmark for the instruction classes the EASU/RCAS kernels are made of.
// Answers, on the part itself, the questions DESIGN.md §4 argues from: how many warp-instructions per clock per SM
// do FFMA, HFMA2 (packed half), FFMA2 (packed f32x2), HMNMX2 / integer ALU ops and LDS sustain, alone and MIXED
// (does an ALU or FP32 instruction issue in the shadow of an HFMA2?).
//
//   nvcc -O3 -gencode arch=compute_100a,code=sm_100a -o /tmp/ubench_pipes tools/ubench_pipes.cu && /tmp/ubench_pipes
//
// Method: 2 x SMs CTAs of 256 threads, every thread runs kIters x 64 inline-PTX instructions over 8 independent
// dependency chains (latency hidden), clock64() around the loop; rate = warp-instructions executed on CTA 0's SM
// (8 warps x the number of CTAs that %smid shows on that SM) divided by the cycles of CTA 0's slowest warp.
// Operands are thread-varying runtime values so nothing folds or moves to the uniform datapath.
// (Round-1 run, profiles/r01_ubench_pipes.txt, predates the %smid count and assumed 2 CTAs on the SM: see its header.)
// The "events" column times the same launch with CUDA events instead: warp-instructions of the whole grid per SM over the
// kernel's wall time, per NOMINAL clock (so it reads low when the part runs below nominal, and it includes launch cost).
// SASS per loop iteration (ptxas folds and splits some PTX instructions): python tools/sass_tools.py loops <binary>.
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>

constexpr int kIters = 2000;

#define CHAINS8(OP) OP(0) OP(1) OP(2) OP(3) OP(4) OP(5) OP(6) OP(7)
#define REP8(X) X X X X X X X X

// ---- single-class bodies (64 instructions per iteration) ----------------------------------------
#define FFMA3(i) asm volatile("fma.rn.f32 %0, %1, %2, %0;" : "+f"(f[i]) : "f"(fb), "f"(fc));
#define FFMAI(i) asm volatile("fma.rn.f32 %0, %0, 0f3F800001, %1;" : "+f"(f[i]) : "f"(fc));
#define HFMA3(i) asm volatile("fma.rn.f16x2 %0, %1, %2, %0;" : "+r"(h[i]) : "r"(hb), "r"(hc));
#define HFMAI(i) asm volatile("fma.rn.f16x2 %0, %0, %1, %2;" : "+r"(h[i]) : "r"(0x3c013c01u), "r"(hc));
#define HMUL(i)  asm volatile("mul.rn.f16x2 %0, %0, %1;" : "+r"(h[i]) : "r"(hb));
#define HADD(i)  asm volatile("add.rn.f16x2 %0, %0, %1;" : "+r"(h[i]) : "r"(hb));
#define HMIN(i)  asm volatile("min.f16x2 %0, %0, %1;" : "+r"(h[i]) : "r"(h[(i + 1) & 7]));
#define FFMA2(i) asm volatile("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d[i]) : "l"(db), "l"(dc));
// integer / min ops take a NEIGHBOUR chain as second operand so that ptxas cannot fold repeated applications
#define IADD(i)  asm volatile("add.s32 %0, %0, %1;" : "+r"(u[i]) : "r"(u[(i + 1) & 7]));
#define LOP(i)   asm volatile("prmt.b32 %0, %0, %1, 0x5432;" : "+r"(u[i]) : "r"(u[(i + 1) & 7]));
#define FMNMX(i) asm volatile("min.f32 %0, %0, %1;" : "+f"(f[i]) : "f"(f[(i + 1) & 7]));
#define IMIN16(i) asm volatile("min.s16x2 %0, %0, %1;" : "+r"(u[i]) : "r"(u[(i + 1) & 7]));
#define LDS(i)   asm volatile("ld.volatile.shared.b32 %0, [%1];" : "=r"(u[i]) : "r"(saddr + 4 * i));
#define MUFU(i)  asm volatile("rsqrt.approx.ftz.f32 %0, %0;" : "+f"(f[i]));
// tensor pipe (the legacy warp-synchronous MMA; chain i accumulates into c[i][0..3], A and B are runtime registers)
#define MMA(i)   asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};" \
                              : "+f"(c[i][0]), "+f"(c[i][1]), "+f"(c[i][2]), "+f"(c[i][3]) : "r"(hb), "r"(hc), "r"(h[0]), "r"(hb), "r"(hc), "r"(hb));
// (its four results are folded into chain i by two LOP3, or ptxas drops every load whose result is overwritten unread)
#define LDSMT(i) { uint32_t r0, r1, r2, r3;                                                                   \
                   asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"         \
                                : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(laddr + 512 * (i)));             \
                   u[i] ^= r0 ^ r1 ^ r2 ^ r3; }

// ---- mixed bodies: 4 of A then 4 of B per 8-group, on disjoint registers --------------------------
#define MIX(A, B) A(0) B(0) A(1) B(1) A(2) B(2) A(3) B(3) A(4) B(4) A(5) B(5) A(6) B(6) A(7) B(7)
// one MMA then 4 (8) HFMA2 on 8 chains: the shape of a tap loop whose accumulate went to the tensor pipe
#define MIX4(i) MMA(i) HFMA3(0) HFMA3(2) HFMA3(4) HFMA3(6)
#define MIX8(i) MMA(i) HFMA3(0) HFMA3(1) HFMA3(2) HFMA3(3) HFMA3(4) HFMA3(5) HFMA3(6) HFMA3(7)

#define KERNEL(NAME, BODY, PER_ITER)                                                                      \
  __global__ void __launch_bounds__(256) NAME(unsigned long long* out, float fb, float fc, uint32_t hb,  \
                                              uint32_t hc, uint32_t ub, unsigned long long db,           \
                                              unsigned long long dc) {                                    \
    __shared__ __align__(16) uint32_t sm[8 * 256];                                                        \
    for (int i = threadIdx.x; i < 8 * 256; i += 256) sm[i] = i;                                           \
    __syncthreads();                                                                                      \
    const uint32_t saddr = (uint32_t)__cvta_generic_to_shared(sm) + (threadIdx.x & 31) * 4;              \
    /* ldmatrix row address of this lane: 32 consecutive 16-byte rows, conflict-free per 8-lane phase */  \
    const uint32_t laddr = (uint32_t)__cvta_generic_to_shared(sm) + (threadIdx.x & 31) * 16;             \
    float f[8], c[8][4];                                                                                  \
    uint32_t h[8], u[8], q[8][2];                                                                         \
    unsigned long long d[8];                                                                              \
    for (int i = 0; i < 8; i++) {                                                                         \
      f[i] = fb + i + threadIdx.x; h[i] = hb + i + (threadIdx.x & 3); u[i] = ub * (i + 1) + threadIdx.x * 2654435761u; \
      d[i] = db + i + threadIdx.x; c[i][0] = c[i][1] = c[i][2] = c[i][3] = fb * i; q[i][0] = q[i][1] = i;   \
    }          \
    const long long t0 = clock64();                                                                       \
    _Pragma("unroll 1") for (int it = 0; it < kIters; it++) { BODY }                                                          \
    const long long t1 = clock64();                                                                       \
    float acc = 0;                                                                                        \
    for (int i = 0; i < 8; i++)                                                                           \
      acc += f[i] + (float)h[i] + (float)u[i] + (float)d[i] + c[i][0] + c[i][1] + c[i][2] + c[i][3] + (float)(q[i][0] ^ q[i][1]); \
    if (acc == 123.456f) out[1] = 1;                                                                      \
    if (blockIdx.x == 0) atomicMax(out, (unsigned long long)(t1 - t0));                                   \
    if (threadIdx.x == 0) { uint32_t sid; asm("mov.u32 %0, %%smid;" : "=r"(sid)); out[2 + blockIdx.x] = sid; } \
  }                                                                                                       \
  static_assert(PER_ITER > 0, "");

KERNEL(k_ffma3, REP8(CHAINS8(FFMA3)), 64)
KERNEL(k_ffmai, REP8(CHAINS8(FFMAI)), 64)
KERNEL(k_hfma3, REP8(CHAINS8(HFMA3)), 64)
KERNEL(k_hfmai, REP8(CHAINS8(HFMAI)), 64)
KERNEL(k_hmul, REP8(CHAINS8(HMUL)), 64)
KERNEL(k_hadd, REP8(CHAINS8(HADD)), 64)
KERNEL(k_hmin, REP8(CHAINS8(HMIN)), 64)
KERNEL(k_ffma2, REP8(CHAINS8(FFMA2)), 64)
KERNEL(k_iadd, REP8(CHAINS8(IADD)), 64)
KERNEL(k_prmt, REP8(CHAINS8(LOP)), 64)
KERNEL(k_hfma_hadd, REP8(MIX(HFMA3, HADD)), 128)
#define TAPMIX HFMA3(0) HFMA3(1) HFMA3(2) HMIN(3) HFMA3(4) HFMA3(5) HFMA3(6) FFMA3(7)
KERNEL(k_tapmix, REP8(TAPMIX TAPMIX), 128)
KERNEL(k_fmnmx, REP8(CHAINS8(FMNMX)), 64)
KERNEL(k_lds, REP8(CHAINS8(LDS)), 64)
KERNEL(k_mufu, REP8(CHAINS8(MUFU)), 64)
KERNEL(k_hfma_ffma, REP8(MIX(HFMA3, FFMA3)), 128)
KERNEL(k_hfma_iadd, REP8(MIX(HFMA3, IADD)), 128)
KERNEL(k_hfma_hmin, REP8(MIX(HFMA3, HMIN)), 128)
KERNEL(k_hfma_lds, REP8(MIX(HFMA3, LDS)), 128)
KERNEL(k_hfma_mufu, REP8(MIX(HFMA3, MUFU)), 128)
KERNEL(k_ffma_iadd, REP8(MIX(FFMA3, IADD)), 128)
KERNEL(k_ffma_lop, REP8(MIX(FFMA3, LOP)), 128)
KERNEL(k_hfma_ffma2, REP8(MIX(HFMA3, FFMA2)), 128)
KERNEL(k_ffma_ffma2, REP8(MIX(FFMA3, FFMA2)), 128)
KERNEL(k_hfmai_ffmai, REP8(MIX(HFMAI, FFMAI)), 128)
KERNEL(k_imin16, REP8(CHAINS8(IMIN16)), 64)
KERNEL(k_hfma_imin16, REP8(MIX(HFMA3, IMIN16)), 128)
KERNEL(k_hfma_prmt, REP8(MIX(HFMA3, LOP)), 128)
KERNEL(k_ffma2_prmt, REP8(MIX(FFMA2, LOP)), 128)
KERNEL(k_ffma2_hmin, REP8(MIX(FFMA2, HMIN)), 128)
#define TAPMIX2 HFMA3(0) HFMA3(1) HFMA3(2) IMIN16(3) HFMA3(4) HFMA3(5) HFMA3(6) FFMA2(7)
KERNEL(k_tapmix2, REP8(TAPMIX2 TAPMIX2), 128)
KERNEL(k_mma, REP8(CHAINS8(MMA)), 64)
KERNEL(k_mma_hfma4, REP8(CHAINS8(MIX4)), 320)
KERNEL(k_mma_hfma8, REP8(CHAINS8(MIX8)), 576)
KERNEL(k_ldsm, CHAINS8(LDSMT), 8)

typedef void (*kern_t)(unsigned long long*, float, float, uint32_t, uint32_t, uint32_t, unsigned long long,
                       unsigned long long);

int main() {
  int sms = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  unsigned long long* out;
  cudaMalloc(&out, 16 + 8 * 4096);
  static unsigned long long host[2 + 4096];
  struct { const char* name; kern_t k; int per_iter; const char* what; } tests[] = {
      {"FFMA 3-reg", k_ffma3, 64, "fma.rn.f32 d,a,b,d"},
      {"FFMA imm", k_ffmai, 64, "fma.rn.f32 d,d,imm,c"},
      {"HFMA2 3-reg", k_hfma3, 64, "fma.rn.f16x2 d,a,b,d"},
      {"HFMA2 imm", k_hfmai, 64, "fma.rn.f16x2 d,d,imm,c"},
      {"HMUL2", k_hmul, 64, "mul.rn.f16x2"},
      {"HADD2", k_hadd, 64, "add.rn.f16x2"},
      {"HMNMX2", k_hmin, 64, "min.f16x2"},
      {"FFMA2 (f32x2)", k_ffma2, 64, "fma.rn.f32x2 (2 fp32 FMAs per lane)"},
      {"IADD", k_iadd, 64, "add.s32"},
      {"PRMT", k_prmt, 64, "prmt.b32"},
      {"HFMA2 + HADD2 1:1", k_hfma_hadd, 128, "alternating"},
      {"HFMA2 x3 : FFMA x1 ...", k_tapmix, 128, "8 x (6 HFMA2, 1 HMNMX2, 1 FFMA) + 64 more of the same: the EASU tap mix"},
      {"FMNMX", k_fmnmx, 64, "min.f32"},
      {"LDS.32", k_lds, 64, "ld.shared.b32, conflict-free"},
      {"MUFU.RSQ", k_mufu, 64, "rsqrt.approx.ftz.f32"},
      {"HFMA2 + FFMA 1:1", k_hfma_ffma, 128, "alternating"},
      {"HFMA2 + IADD 1:1", k_hfma_iadd, 128, "alternating"},
      {"HFMA2 + HMNMX2 1:1", k_hfma_hmin, 128, "alternating"},
      {"HFMA2 + LDS 1:1", k_hfma_lds, 128, "alternating"},
      {"HFMA2 + MUFU 1:1", k_hfma_mufu, 128, "alternating"},
      {"FFMA + IADD 1:1", k_ffma_iadd, 128, "alternating"},
      {"FFMA + PRMT 1:1", k_ffma_lop, 128, "alternating"},
      {"HFMA2 + FFMA2 1:1", k_hfma_ffma2, 128, "alternating"},
      {"FFMA + FFMA2 1:1", k_ffma_ffma2, 128, "alternating"},
      {"HFMA2 imm + FFMA imm 1:1", k_hfmai_ffmai, 128, "alternating"},
      {"VIMNMX.S16x2", k_imin16, 64, "min.s16x2 (packed integer min)"},
      {"HFMA2 + VIMNMX.S16x2 1:1", k_hfma_imin16, 128, "alternating"},
      {"HFMA2 + PRMT 1:1", k_hfma_prmt, 128, "alternating"},
      {"FFMA2 + PRMT 1:1", k_ffma2_prmt, 128, "alternating"},
      {"FFMA2 + HMNMX2 1:1", k_ffma2_hmin, 128, "alternating"},
      {"tap mix, int clamp, FFMA2", k_tapmix2, 128, "8 x (6 HFMA2, 1 VIMNMX.S16x2, 1 FFMA2)"},
      {"HMMA.16816.F32", k_mma, 64, "mma.sync m16n8k16 f32.f16.f16.f32 (2048 FMAs per warp-instruction)"},
      {"HMMA + HFMA2 1:4", k_mma_hfma4, 320, "per MMA 4 HFMA2; rate counts both"},
      {"HMMA + HFMA2 1:8", k_mma_hfma8, 576, "per MMA 8 HFMA2; rate counts both"},
      {"LDSM.16.MT88.4", k_ldsm, 8, "ldmatrix.x4.trans, 512 B per warp-instruction, conflict-free (+ 2 LOP3 each)"},
  };
  int khz = 0;
  cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, 0);
  printf("device SMs: %d; warp-instructions per clock64 tick per SM; nominal SM clock %.0f MHz\n", sms, khz / 1e3);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  for (auto& t : tests) {
    double best = 0, best_ev = 0;
    for (int rep = 0; rep < 3; rep++) {
      cudaMemset(out, 0, 16 + 8 * 4096);
      cudaEventRecord(e0);
      t.k<<<sms * 2, 256>>>(out, 1.0001f, 0.5f, 0x3c003c01u, 0x38003801u, 3u, 0x3f8000013f800002ull, 0x3f0000003f000001ull);
      cudaEventRecord(e1);
      cudaMemcpy(host, out, 16 + 8 * (size_t)(sms * 2), cudaMemcpyDeviceToHost);
      const unsigned long long cyc = host[0];
      int ctas = 0;  // CTAs resident on the SM whose CTA 0 was timed (the block scheduler does not deal exactly 2 per SM)
      for (int b = 0; b < sms * 2; b++) ctas += host[2 + b] == host[2];
      if (cudaGetLastError() != cudaSuccess || cyc == 0) { printf("%-26s FAILED\n", t.name); break; }
      const double rate = 8.0 * ctas * (double)t.per_iter * kIters / (double)cyc;
      if (rate > best) best = rate;
      float ms_ev = 0;  // CUDA events: every warp of the grid over the kernel's wall time, per SM and per nominal clock
      cudaEventElapsedTime(&ms_ev, e0, e1);
      const double ev = 2.0 * 8.0 * (double)t.per_iter * kIters / (ms_ev * 1e-3 * khz * 1e3);
      if (ev > best_ev) best_ev = ev;
      if (rep == 2 && &t == &tests[0]) {  // calibrate the tick against wall clock (kernel time ~ timed loop, launch overhead small at 0.3+ ms)
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        printf("CTAs resident on the timed SM: %d (%d warps); clock64 advanced %.0f ticks in a %.3f ms kernel => <= %.0f MHz tick rate\n",
               ctas, 8 * ctas, (double)cyc, ms, (double)cyc / (ms * 1e3));
      }
    }
    printf("%-26s %5.2f inst/clk/SM  events %5.2f   (%s)\n", t.name, best, best_ev, t.what);
  }
  cudaFree(out);
  return 0;
}
