// painter_b200 — shared device-side PTX wrappers for sm_100a (mbarrier, TMA, tcgen05/TMEM).
// Everything here is raw inline PTX; no CUTLASS dependency.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdio.h>
#include <stdint.h>

namespace pk {

// ----------------------------------------------------------------------------------------------
// Watchdog: every mbarrier wait is bounded. A dead pipeline traps (-> cudaErrorLaunchFailure)
// instead of hanging the GPU.
// ----------------------------------------------------------------------------------------------
#ifndef PK_WAIT_TIMEOUT_NS
#define PK_WAIT_TIMEOUT_NS 4000000000ull  // 4 s
#endif

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

// One elected lane of a fully converged warp (elect.sync): keeps the surrounding control flow warp-uniform so that
// ptxas can hold MMA / TMA descriptors in uniform registers instead of R2UR-ing them per instruction.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------- mbarrier --------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done != 0;
}
static __device__ __noinline__ void mbar_wait_slow(uint32_t bar, uint32_t parity) {
  const uint64_t t0 = globaltimer_ns();
  while (!mbar_try_wait(bar, parity)) {
    if (globaltimer_ns() - t0 > PK_WAIT_TIMEOUT_NS) {
      printf("[painter_b200] mbarrier wait timeout: block %d thread %d bar 0x%x parity %u\n",
             blockIdx.x, threadIdx.x, bar, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
#pragma unroll 1
  for (int i = 0; i < 64; ++i)
    if (mbar_try_wait(bar, parity)) return;
  mbar_wait_slow(bar, parity);
}

// ------------------------------------------- TMA ----------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar,
                                            int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* m, uint32_t bar,
                                            int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* m, uint32_t bar,
                                            int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// TMA store (shared -> global, bulk-group completion)
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all committed groups have finished READING their shared-memory source (the buffer may be overwritten)
__device__ __forceinline__ void tma_store_wait_read0() {
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
// all committed groups have completed (writes performed)
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ----------------------------------------- tcgen05 --------------------------------------------
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// whole warp; writes TMEM base address to *holder (shared memory)
__device__ __forceinline__ void tmem_alloc(uint32_t holder_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(holder_smem),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc,
                                        uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]
__device__ __forceinline__ void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc,
                                        uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on mbarrier when all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}

// Shared-memory matrix descriptor, SWIZZLE_128B, Blackwell version bit set.
//  K-major operand tile  [rows][64 bf16]  (TMA box {64, rows}, 128B swizzle): lbo ignored, sbo = 1024
//  MN-major operand tile [k rows][64 bf16 of MN] : sbo = 1024 (8 k-rows), lbo = bytes between 64-wide MN groups
__device__ __forceinline__ uint64_t make_sdesc(uint32_t smem_addr, uint32_t lbo_bytes,
                                               uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= 1ull << 46;  // descriptor version (sm_100)
  d |= 2ull << 61;  // SWIZZLE_128B
  return d;
}
// Advance a descriptor's start address by `bytes` (multiple of 16; stays inside the 14-bit field for any smem offset).
__device__ __forceinline__ uint64_t sdesc_add(uint64_t desc, uint32_t bytes) {
  return desc + static_cast<uint64_t>(bytes >> 4);
}
// Instruction descriptor for kind::f16, bf16 x bf16 -> fp32.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, bool a_mn_major,
                                                       bool b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(a_mn_major) << 15) |
         (static_cast<uint32_t>(b_mn_major) << 16) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}

// ----- TMEM <-> registers (32 lanes x 32 bit, thread i of the warp <-> TMEM lane base+i) -----
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_st_x8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
               "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
      "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
      "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
      "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]),
      "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]),
      "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_wait_st() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// ---------------------------------------- misc math -------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16_round(float x) {
  return __bfloat162float(__float2bfloat16_rn(x));
}
// erf-GELU (nn.GELU(), exact form) and its derivative.  erf through Abramowitz-Stegun 7.1.26
// (|error| <= 1.5e-7 absolute: three orders below bf16 resolution, at ~1/3 of erff's instruction count):
//   erf(u) = 1 - (a1 t + ... + a5 t^5) exp(-u^2),  t = 1 / (1 + p u),  u >= 0.
// With u = |x| / sqrt(2) the same exponential exp(-x^2 / 2) also gives the Gaussian density the derivative needs.
__device__ __forceinline__ void gelu_parts(float x, float& cdf, float& pdf) {
  const float u = fabsf(x) * 0.70710678118654752f;
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, u, 1.0f)));
  float e;  // exp(-u^2) = exp2(-u^2 * log2(e))
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(u * u * -1.4426950408889634f));
  float poly = fmaf(1.061405429f, t, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  const float half_erfc = 0.5f * poly * t * e;        // 0.5 * erfc(u)
  cdf = x >= 0.f ? 1.0f - half_erfc : half_erfc;      // Phi(x)
  pdf = 0.39894228040143268f * e;                     // phi(x)
}
__device__ __forceinline__ float gelu_erf(float x) {
  float cdf, pdf;
  gelu_parts(x, cdf, pdf);
  return x * cdf;
}
__device__ __forceinline__ float gelu_erf_grad(float x) {
  float cdf, pdf;
  gelu_parts(x, cdf, pdf);
  return fmaf(x, pdf, cdf);
}
// GEMM-epilogue variant (fc1 forward, fc2 dgrad: 51 M activations per block application, where the epilogue's issue
// slots are what bounds the kernel).  Phi(x) = 0.5 + 0.5 tanh(x P(x^2)) with P fitted to the EXACT erf form
// (minimax over |x| <= 8: |x Phi_fit - gelu_erf| <= 2.5e-5, derivative error <= 1.1e-4 - the textbook "tanh GELU"
// constants would be 20x worse); one MUFU (tanh.approx, rel. error 2^-11) instead of two, ~8 FMA-pipe instructions
// instead of ~15.  Both absolute errors sit an order of magnitude below the bf16 rounding of activations near 1 (2^-9);
// relative to small values they do not (bf16 ulps of gelu(z): ~9 for z in [-4, -3), ~250 below -4).  Measured on
// a B200 (1000 W power limit) over every bf16 z in [-12, 12] (tests/test_gpu_kernel_contracts.py, scripts/gelu_epilogue_error.py), with
// tanh.approx: |gelu error| <= 0.70 (1 bf16 ulp + 2^-15), |gelu' error| <= 0.65 (1 bf16 ulp + 2^-13).
// The argument is clamped at x^2 = 64, where tanh has long saturated (P turns over beyond |x| ~ 11).
__device__ __forceinline__ float tanh_approx(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
constexpr float GELU_P0 = 0.7975078789040602f, GELU_P1 = 0.037005650567220924f, GELU_P2 = -0.00035151747747947537f;
__device__ __forceinline__ float gelu_fast(float x) {
  const float u = fminf(x * x, 64.0f);
  const float p = fmaf(fmaf(GELU_P2, u, GELU_P1), u, GELU_P0);
  const float t = tanh_approx(x * p);
  const float hx = 0.5f * x;
  return fmaf(hx, t, hx);
}
__device__ __forceinline__ float gelu_fast_grad(float x) {
  const float u = fminf(x * x, 64.0f);
  const float p = fmaf(fmaf(GELU_P2, u, GELU_P1), u, GELU_P0);
  const float q = fmaf(fmaf(5.0f * GELU_P2, u, 3.0f * GELU_P1), u, GELU_P0);   // d/dx [x P(x^2)]
  const float t = tanh_approx(x * p);
  const float s = fmaf(-t, t, 1.0f);
  return fmaf(0.5f * x * s, q, fmaf(0.5f, t, 0.5f));
}
// exp2 on the MUFU pipe (ex2.approx.ftz): inputs here are <= 0 after the running-max subtraction or bounded by
// the lazy-rescale threshold, so flush-to-zero of denormal results is exactly what softmax wants.
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// Packed fp32 pairs (sm_100 FFMA2 / FADD2 / FMUL2): one issue slot for two lanes of work.  The softmax warps of the
// attention kernels are issue-bound (~17 instructions per score), so the per-score arithmetic runs on register pairs.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack_f2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ f32x2 pack_u2(uint32_t lo, uint32_t hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
  return r;
}
__device__ __forceinline__ void unpack_f2(f32x2 v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 fma_f2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ f32x2 add_f2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ f32x2 mul_f2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
// The GEMM-epilogue GELU / GELU' on a PAIR of activations: the same operations in the same order as gelu_fast /
// gelu_fast_grad (bit-identical results), with the polynomial and the products on packed fp32 pairs - 10 resp. 16
// issue slots per pair instead of 16 resp. 28 (the fc1 / fc2-dgrad epilogues are what bounds those GEMMs).
__device__ __forceinline__ f32x2 gelu_clamped_sq(f32x2 x2) {
  float u0, u1;
  unpack_f2(mul_f2(x2, x2), u0, u1);
  return pack_f2(fminf(u0, 64.0f), fminf(u1, 64.0f));
}
__device__ __forceinline__ void gelu_fast_pair(float x0, float x1, float& g0, float& g1) {
  const f32x2 x2 = pack_f2(x0, x1);
  const f32x2 u2 = gelu_clamped_sq(x2);
  const f32x2 p2 = fma_f2(fma_f2(pack_f2(GELU_P2, GELU_P2), u2, pack_f2(GELU_P1, GELU_P1)), u2,
                          pack_f2(GELU_P0, GELU_P0));
  float a0, a1;
  unpack_f2(mul_f2(x2, p2), a0, a1);
  const f32x2 t2 = pack_f2(tanh_approx(a0), tanh_approx(a1));
  const f32x2 hx2 = mul_f2(pack_f2(0.5f, 0.5f), x2);
  unpack_f2(fma_f2(hx2, t2, hx2), g0, g1);
}
// (d0, d1) = (y0 * gelu'(x0), y1 * gelu'(x1))
__device__ __forceinline__ void gelu_fast_grad_mul_pair(float x0, float x1, float y0, float y1, float& d0, float& d1) {
  const f32x2 x2 = pack_f2(x0, x1);
  const f32x2 u2 = gelu_clamped_sq(x2);
  const f32x2 p2 = fma_f2(fma_f2(pack_f2(GELU_P2, GELU_P2), u2, pack_f2(GELU_P1, GELU_P1)), u2,
                          pack_f2(GELU_P0, GELU_P0));
  const f32x2 q2 = fma_f2(fma_f2(pack_f2(5.0f * GELU_P2, 5.0f * GELU_P2), u2, pack_f2(3.0f * GELU_P1, 3.0f * GELU_P1)),
                          u2, pack_f2(GELU_P0, GELU_P0));
  float a0, a1;
  unpack_f2(mul_f2(x2, p2), a0, a1);
  const float t0 = tanh_approx(a0), t1 = tanh_approx(a1);
  const f32x2 t2 = pack_f2(t0, t1);
  const f32x2 s2 = fma_f2(pack_f2(-t0, -t1), t2, pack_f2(1.0f, 1.0f));
  const f32x2 hxs2 = mul_f2(mul_f2(pack_f2(0.5f, 0.5f), x2), s2);
  const f32x2 g2 = fma_f2(hxs2, q2, fma_f2(pack_f2(0.5f, 0.5f), t2, pack_f2(0.5f, 0.5f)));
  unpack_f2(mul_f2(pack_f2(y0, y1), g2), d0, d1);
}

// exp2 of a pair of scores.  Where a softmax pass is bound by the MUFU pipe (16 ex2 / clk / SM) rather than by issue
// slots, a compile-time fraction of the pairs (mask: one bit per pair position modulo 4) is evaluated on the FMA / ALU
// pipes instead (measured, B = 8 geometry, scripts/attn_poly_sweep.sh: the first pass of the dK/dV kernel - which does
// nothing but exponentials - gains 8 % at 25 %; the forward and the dQ kernel are issue-bound and lose, so they keep
// mask 0):
// Cody-Waite range reduction with the round-to-nearest magic constant (x = n + f, |f| <= 0.5), a degree-3 minimax
// polynomial for 2^f (max rel. error 7.5e-5 - far below the bf16 rounding of P / dS) and the exponent added as an
// integer.  Arguments are clamped at -126 (masked scores arrive as -inf and must come out as ~0).
#ifndef PK_EXP_POLY_MASK_FWD
#define PK_EXP_POLY_MASK_FWD 0x0
#endif
#ifndef PK_EXP_POLY_MASK_DQ
#define PK_EXP_POLY_MASK_DQ 0x0
#endif
#ifndef PK_EXP_POLY_MASK_DKV
#define PK_EXP_POLY_MASK_DKV 0x8
#endif
__device__ __forceinline__ void exp2_poly_pair(float t0, float t1, float& e0, float& e1) {
  t0 = fmaxf(t0, -126.0f);
  t1 = fmaxf(t1, -126.0f);
  const f32x2 x2 = pack_f2(t0, t1);
  const f32x2 z2 = add_f2(x2, pack_f2(12582912.0f, 12582912.0f));          // n in the low mantissa bits
  const f32x2 n2 = add_f2(z2, pack_f2(-12582912.0f, -12582912.0f));         // float(n)
  const f32x2 f2 = fma_f2(n2, pack_f2(-1.0f, -1.0f), x2);                   // f = x - n
  f32x2 p2 = fma_f2(pack_f2(0.055170804f, 0.055170804f), f2, pack_f2(0.24260928f, 0.24260928f));
  p2 = fma_f2(p2, f2, pack_f2(0.69326097f, 0.69326097f));
  p2 = fma_f2(p2, f2, pack_f2(0.99992818f, 0.99992818f));
  float z0, z1, p0, p1;
  unpack_f2(z2, z0, z1);
  unpack_f2(p2, p0, p1);
  e0 = __int_as_float(__float_as_int(p0) + (__float_as_int(z0) << 23));
  e1 = __int_as_float(__float_as_int(p1) + (__float_as_int(z1) << 23));
}
// pair_idx must be a compile-time constant after unrolling (the branch folds away)
template <int MASK>
__device__ __forceinline__ void exp2_pair(int pair_idx, float t0, float t1, float& e0, float& e1) {
  if ((MASK >> (pair_idx & 3)) & 1) {
    exp2_poly_pair(t0, t1, e0, e1);
  } else {
    e0 = fast_exp2(t0);
    e1 = fast_exp2(t1);
  }
}

// Programmatic dependent launch (host_common.h): let the next kernel of the stream be scheduled / block until the
// previous grid has completed and flushed.  Both are no-ops for a kernel launched without the attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace pk
