// painter_b200 — fused attention backward with decomposed relative-position bias (sm_100a, tcgen05).
//
// Two kernels, both recomputing S = Q.K^T (+bias) tile by tile like the forward (attention_fwd.cu):
//
//  A) attn_bwd_dq_kernel   CTA = 128 query rows, loops over key tiles (112 keys = R image rows).
//       dP = dO.V^T, P = exp2(t - LSE), dS = P * (dP - delta)
//       dQ   = 0.125 * dS.K  +  Gh^.T_h  +  Gw^.T_w          (all on tensor cores)
//       dT_h = Gh^^T.Q , dT_w = Gw^^T.Q                       (tensor cores; per-CTA partials -> reduction kernel)
//     where Gh'[r,i] = sum_{u in image row i} dS[r,u], Gw'[r,j] = sum_{u in image col j} dS[r,u] and
//     Gh^[r,t] = Gh'[r, i_r + h-1 - t] is the Toeplitz re-indexing matching the table row t.
//     Also emits rel_h / rel_w (log2e-scaled bias rows) for kernel B; delta = rowsum(dO * O) comes from a coalesced
//     pre-pass (attn_delta_kernel).
//
//  B) attn_bwd_dkv_kernel  CTA = one key tile, loops over query tiles.
//       dV = P^T.dO , dK = 0.125 * dS^T.Q     (P / dS tiles in smem are read as MN-major A operands)
//     three rotating TMEM score buffers, two-pass softmax (p from S, then dS from dP).
//
// Roles (352 threads): warps 0-7 softmax (lane quarter x column half), warp 8 TMA producer, warp 9 issues the score
// MMAs (S, dP), warp 10 the accumulation MMAs (dQ + epilogue | dK, dV); hand-offs through per-buffer mbarriers.
//
// Reference math: autograd of models_painter.py:80-86 + vitdet_utils.py:113-123 (SURVEY.md Appendix A4).
#include "common.cuh"
#include "host_common.h"
#include "../../include/painter_b200.h"

namespace pk {

constexpr int AB_BM = 128;
constexpr int AB_KT = 112;
constexpr int AB_THREADS = 352;   // 8 softmax warps + TMA warp + two tcgen05 issuing warps (scores | accumulations)
constexpr int AB_SMX = 256;       // softmax threads
constexpr float AB_LOG2E = 1.4426950408889634f;

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// ================================================================================================
// Kernel A
// ================================================================================================
// smem map (offsets from the 1024-aligned base)
constexpr uint32_t A_SQ = 0;                    // Q tile 128 x 128 B
constexpr uint32_t A_SDO = 16384;               // dO tile
constexpr uint32_t A_SDS = 32768;               // 2 x dS tile (2 K-blocks each, double-buffered); T_h staged in
                                                // buffer 0 during the prologue; epilogue: G^ buffer (<= 4 K-blocks)
constexpr uint32_t A_SKV = A_SDS + 65536;       // kv_stages (2 or 3) x (K 14336 | V 14336)
constexpr uint32_t A_STH = A_SKV;               // epilogue: T_h reload (<= 28 KiB) over stage 0
constexpr uint32_t A_STW = A_SKV + 28672;       // epilogue: T_w reload (<= 14 KiB) over stage 1
// rel_h rows fp32 [128][h+1] follow the K/V stages (Gh' sums overwrite them in place): A_SKV + kv_stages * 28672
// (separate K x4 / V x2 rings were tried: the MMA warp never waits on TMA here - the extra commit + barrier per tile
// cost 4 % - so the coupled ring stays)

struct AttnBwdArgs {
  int h, N, heads;
  int th_pad, tw_pad;
  int relh_bytes;   // size of the rel_h / Gh' region
  float scale_log2;
  const __nv_bfloat16* O;    // [B*N, C]
  const __nv_bfloat16* dO;   // [B*N, C]
  const float* lse;          // [B*heads, N]
  float* delta;              // [B*heads, N]
  // bias rows handed from kernel A to kernel B (log2e-scaled), stored per 128-query tile with the QUERY ROW INNERMOST
  // so that the one-thread-per-row accesses of both kernels are coalesced (a warp touches 128 / 512 contiguous bytes;
  // with the row-major [N, W] layout every lane owned its own 112-byte row and a warp-wide load spread over ~30 cache
  // lines - the fetch of the next tile's operands stalled kernel B's softmax warps for 400-1100 cycles per tile):
  float* relh_g;             // [B*heads, q tiles, h, 128]
  float* relw_g;             // [B*heads, q tiles, W/4, 128] float4   (W % 4 != 0: [B*heads, q tiles, W, 128] floats)
  __nv_bfloat16* dqkv;       // [B*N, 3C]
  float* dt_ws;              // [CTAs of kernel A][64][2h-1 + 2W-1] fp32 partial table gradients, table row innermost:
                             // the row owners' stores are then 128 contiguous bytes per warp (row-major slices made
                             // every 16-byte store of a warp hit its own cache line: ~3 k cycles per CTA)
  long long* trace;          // optional debug timeline of CTA (0,0,0): [kernel][role][iter][event]
  int debug;                 // measurement aids: bit 1 trace the last (b, head) CTA instead of the first,
                             // bit 2 skip kernel A, bit 3 skip kernel B (scripts/time_attn_parts.py)
  int kv_stages;             // kernel A: K/V ring depth (3 normally; 2 when shared memory is short)
  int rel_ready;             // relh_g / relw_g were written by the forward (pk_attn_fwd_save): kernel A loads its bias
                             // rows instead of recomputing G_h / G_w (two MMAs + the Toeplitz gathers) and emitting them
};

// debug timeline: `ab_tr` (one predicate register per thread, set at kernel entry) selects the traced CTA, so a
// stamp costs a clock read and a store instead of several special-register reads
#define AB_TRACE_INIT()                                                                                    \
  const bool ab_tr = a.trace != nullptr && blockIdx.x == 0 &&                                              \
                     blockIdx.y == ((a.debug & 2) ? gridDim.y - 1 : 0) &&                                  \
                     blockIdx.z == ((a.debug & 2) ? gridDim.z - 1 : 0)
#define AB_TRACE(kern, role, it, ev)                                                                       \
  do {                                                                                                     \
    if (ab_tr && (it) < 16 && ((role) == 1 || (threadIdx.x & 31) == 0))                                    \
      a.trace[(((kern) * 2 + (role)) * 16 + (it)) * 8 + (ev)] = clock64();                                   \
  } while (0)

template <int W>
__global__ void __launch_bounds__(AB_THREADS, 1)
attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                   const __grid_constant__ CUtensorMap tmdO, const __grid_constant__ CUtensorMap tmTh,
                   const __grid_constant__ CUtensorMap tmTw, const AttnBwdArgs a) {
  constexpr int R = AB_KT / W;
  AB_TRACE_INIT();
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_base = smem_u32(smem_raw);
  const uint32_t base = (raw_base + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - raw_base);

  const uint32_t sQ = base + A_SQ, sdO = base + A_SDO, sdS = base + A_SDS, sKV = base + A_SKV;
  const int KS = a.kv_stages;
  const uint32_t srelh_off = A_SKV + static_cast<uint32_t>(KS) * 28672u;
  float* relh_gen = reinterpret_cast<float*>(gen + srelh_off);
  const uint32_t bar0 = base + srelh_off + a.relh_bytes;
  const uint32_t bar_q = bar0, bar_kf = bar0 + 8 /*4*/, bar_ke = bar0 + 40 /*4*/,
                 bar_p1 = bar0 + 72, bar_df = bar0 + 80 /*2*/,
                 bar_s = bar0 + 104 /*2*/, bar_p0 = bar0 + 120, bar_g = bar0 + 128,
                 bar_gr = bar0 + 136, bar_e = bar0 + 144, bar_er = bar0 + 152, bar_t = bar0 + 160,
                 bar_gw = bar0 + 168;  // G_w retired (single completion; bar_g completes twice and would alias)
  const uint32_t holder = bar0 + 176;
  const uint32_t bar_e2 = bar0 + 184;  // single-phase epilogue: the table-gradient MMAs (issued by warp 9) retired
  volatile uint32_t* holder_gen =
      reinterpret_cast<volatile uint32_t*>(gen + srelh_off + a.relh_bytes + 176);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * AB_BM;
  const int head = blockIdx.y, b = blockIdx.z;
  const int C = a.heads * 64;
  const int h = a.h;
  const int num_tiles = (h + R - 1) / R;
  // Epilogue copies of the tables (MN-major B operands).  With a 3-deep ring the stage last used by tile
  // num_tiles-3 idles for the final two tiles: if both tables fit there they are reloaded two tiles early and their
  // TMA latency disappears from the epilogue; otherwise they land on stages 0/1 after the main loop has retired.
  const bool early_tables =
      KS == 3 && num_tiles >= 3 && static_cast<uint32_t>(a.th_pad + a.tw_pad) * 128u <= 28672u;
  // Single-phase epilogue: when Gh^ needs at most two 64-column K-blocks (th_pad <= 128) it lives in dS buffer 0 and
  // Gw^ in dS buffer 1, the Gw' exchange between the column halves goes through the (dead) dO tile, and ONE batch of
  // MMAs / one TMEM read-out replaces the two dependent rounds (the epilogue was 12 k of a CTA's 48 k cycles at 56x28:
  // profiles/r02_attn_cta_timelines.txt).
  const bool merged_ep = a.th_pad <= 128 && static_cast<uint32_t>(W + 1) * AB_BM * 4u <= 16384u;
  const uint32_t sTh = early_tables ? sKV + static_cast<uint32_t>(num_tiles % 3) * 28672u : base + A_STH;
  const uint32_t sTw = early_tables ? sTh + static_cast<uint32_t>(a.th_pad) * 128u : base + A_STW;

  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmKV);
    tma_prefetch_desc(&tmdO);
    mbar_init(bar_q, 1);
    for (int q = 0; q < 4; ++q) {
      mbar_init(bar_kf + 8 * q, 1);
      mbar_init(bar_ke + 8 * q, 1);
    }
    mbar_init(bar_s, 1);
    mbar_init(bar_s + 8, 1);
    mbar_init(bar_p0, AB_SMX / 32);
    mbar_init(bar_p1, AB_SMX / 32);
    mbar_init(bar_df, 1);
    mbar_init(bar_df + 8, 1);
    mbar_init(bar_g, 1);
    mbar_init(bar_gr, AB_SMX);
    mbar_init(bar_e, 1);
    mbar_init(bar_er, AB_SMX);
    mbar_init(bar_t, 1);
    mbar_init(bar_gw, 1);
    mbar_init(bar_e2, 1);
    fence_barrier_init();
  }
  if (warp == 9) tmem_alloc(holder, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *holder_gen;
  // S / dP double-buffered: buffer b at columns 224 b (S) and 224 b + 112 (dP); dQ accumulator at 448
  const uint32_t tS = tmem, tdQ = tmem + 448;
  pdl_launch_dependents();   // programmatic dependent launch (host_common.h); no global access above this line
  pdl_wait();

  if (warp == 8) {
    if (lane == 0) {
      // ------------------------------------ TMA producer ------------------------------------
      mbar_expect_tx(bar_q, 32768u + (a.rel_ready ? 0u : static_cast<uint32_t>(a.th_pad + a.tw_pad) * 128u));
      tma_load_3d(sQ, &tmQ, bar_q, head * 64, q0, b);
      tma_load_3d(sdO, &tmdO, bar_q, head * 64, q0, b);
      if (!a.rel_ready) {
        tma_load_2d(sdS, &tmTh, bar_q, 0, 0);                 // T_h: th_pad <= 224 rows -> 28 KiB <= 32 KiB
        tma_load_2d(sKV + (KS - 1) * 28672 + 14336, &tmTw, bar_q, 0, 0);  // T_w in the last stage's V buffer
      }
      for (int j = 0; j < num_tiles; ++j) {
        const int st = j % KS;
        if (j >= KS) mbar_wait(bar_ke + 8 * st, ((j / KS) - 1) & 1);
        if (j == KS - 1 && !a.rel_ready) mbar_wait(bar_gw, 0);  // G_w MMA done with T_w (last stage's V buffer)
        mbar_expect_tx(bar_kf + 8 * st, 2 * AB_KT * 128);
        tma_load_3d(sKV + st * 28672, &tmKV, bar_kf + 8 * st, C + head * 64, j * AB_KT, b);
        tma_load_3d(sKV + st * 28672 + 14336, &tmKV, bar_kf + 8 * st, 2 * C + head * 64, j * AB_KT, b);
        AB_TRACE(0, 0, j, 5);
      }
      // epilogue: reload the tables as MN-major B operands (early into the idle stage, else once every main-loop
      // MMA has retired)
      if (early_tables) mbar_wait(bar_ke + 8 * (num_tiles % 3), ((num_tiles - 3) / 3) & 1);
      else mbar_wait(bar_e, 0);
      mbar_expect_tx(bar_t, static_cast<uint32_t>(a.th_pad + a.tw_pad) * 128u);
      tma_load_2d(sTh, &tmTh, bar_t, 0, 0);
      tma_load_2d(sTw, &tmTw, bar_t, 0, 0);
    }
  } else if (warp == 9) {
    {
      // -------------------------------------- MMA issuer --------------------------------------
      // warp-uniform control flow; the tcgen05 instructions themselves are issued by one elected lane
      mbar_wait(bar_q, 0);
      tc_fence_after();
      if (!a.rel_ready) {
      {  // G_w = Q . T_w^T
        const uint32_t idesc = make_idesc_bf16(128, a.tw_pad, false, false);
        const uint32_t sT = sKV + (KS - 1) * 28672 + 14336;
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_ss(tS, make_sdesc(sQ + k * 32, 16, 1024), make_sdesc(sT + k * 32, 16, 1024), idesc, k != 0);
          umma_commit(bar_g);
          umma_commit(bar_gw);
        }
        __syncwarp();
      }
      mbar_wait(bar_gr, 0);
      tc_fence_after();
      {  // G_h = Q . T_h^T
        const uint32_t idesc = make_idesc_bf16(128, a.th_pad, false, false);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_ss(tS, make_sdesc(sQ + k * 32, 16, 1024), make_sdesc(sdS + k * 32, 16, 1024), idesc, k != 0);
          umma_commit(bar_g);
        }
        __syncwarp();
      }
      mbar_wait(bar_gr, 1);
      tc_fence_after();
      }
      const uint32_t idesc_s = make_idesc_bf16(128, AB_KT, false, false);
      const uint64_t dQ0 = make_sdesc(sQ, 16, 1024), ddO0 = make_sdesc(sdO, 16, 1024);
      // Scores issuer: S/dP of tile j go out as soon as their TMEM buffer (j & 1) has been read by the softmax warps
      // (tile j-2, barrier bar_p[j & 1]) and the K/V stage has landed; the accumulation MMAs are issued by warp 10,
      // so neither stream waits behind the other's issue latency (a burst of 7-8 small MMAs costs 600-900 cycles).
      for (int j = 0; j < num_tiles; ++j) {
        const int st = j & 1, ks = j % KS;
        const uint32_t sK = sKV + ks * 28672, sV = sK + 14336;
        const uint64_t dK0 = make_sdesc(sK, 16, 1024), dV0 = make_sdesc(sV, 16, 1024);
        const uint32_t tSb = tS + st * 224, tdPb = tSb + 112;
        AB_TRACE(0, 0, j, 0);
        if (j >= 2) mbar_wait(st ? bar_p1 : bar_p0, ((j >> 1) - 1) & 1);
        mbar_wait(bar_kf + 8 * ks, (j / KS) & 1);
        AB_TRACE(0, 0, j, 1);
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss(tSb, sdesc_add(dQ0, k * 32), sdesc_add(dK0, k * 32), idesc_s, k != 0);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss(tdPb, sdesc_add(ddO0, k * 32), sdesc_add(dV0, k * 32), idesc_s, k != 0);
          umma_commit(bar_s + 8 * st);
        }
        __syncwarp();
        AB_TRACE(0, 0, j, 2);
      }
      if (merged_ep) {
        // single-phase epilogue, second issuer: the 16 table-gradient MMAs go out from this (now idle) warp while
        // warp 10 issues the 11 dQ-bias MMAs - a lone thread dispatches a short burst at 100-190 cycles per MMA
        const uint32_t idesc_tt = make_idesc_bf16(128, 64, true, true);
        mbar_wait(bar_er, 0);
        tc_fence_after();
        if (elect_one()) {
          for (int mh = 0; mh * 128 < a.th_pad; ++mh)
#pragma unroll
            for (int kk = 0; kk < 8; ++kk)
              umma_ss(tS + mh * 64, make_sdesc(sdS + (2 * mh) * 16384 + kk * 2048, 16384, 1024),
                      make_sdesc(sQ + kk * 2048, 16, 1024), idesc_tt, kk != 0);
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_ss(tS + 128, make_sdesc(sdS + 32768 + kk * 2048, 16384, 1024), make_sdesc(sQ + kk * 2048, 16, 1024),
                    idesc_tt, kk != 0);
          umma_commit(bar_e2);
        }
        __syncwarp();
      }
    }
  } else if (warp == 10) {
    {
      // ------------------------------ accumulation issuer (dQ, epilogue) ------------------------------
      const uint32_t idesc_dq = make_idesc_bf16(128, 64, false, true);
      for (int j = 0; j < num_tiles; ++j) {
        const int st = j & 1;
        mbar_wait(st ? bar_p1 : bar_p0, (j >> 1) & 1);
        AB_TRACE(0, 0, j, 3);
        tc_fence_after();
        const uint64_t ddS0 = make_sdesc(sdS + st * 32768, 16, 1024);
        const uint64_t dK0 = make_sdesc(sKV + (j % KS) * 28672, 16, 1024);
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < AB_KT / 16; ++kk)
            umma_ss(tdQ, sdesc_add(ddS0, (kk >> 2) * 16384 + (kk & 3) * 32), sdesc_add(dK0, kk * 2048), idesc_dq,
                    (j | kk) != 0);
          umma_commit(bar_ke + 8 * (j % KS));   // K/V stage free (S/dP of this tile retired before p(j))
          umma_commit(bar_df + 8 * st);         // dS buffer free
        }
        __syncwarp();
        AB_TRACE(0, 0, j, 4);
      }
      if (elect_one()) umma_commit(bar_e);  // completion #1 (parity 0): main loop retired
      __syncwarp();
      const uint32_t idesc_tt = make_idesc_bf16(128, 64, true, true);
      if (merged_ep) {
        // ---- single-phase epilogue (both Toeplitz operands fit next to each other: Gh^ in dS buffer 0, Gw^ in
        // buffer 1): dQ += Gh^ . T_h + Gw^ . T_w here; dT_h = Gh^^T . Q -> columns [0, 128) and dT_w = Gw^^T . Q ->
        // [128, 192) from warp 9
        mbar_wait(bar_er, 0);
        mbar_wait(bar_t, 0);
        tc_fence_after();
        if (elect_one()) {
          for (int kk = 0; kk < a.th_pad / 16; ++kk)
            umma_ss(tdQ, make_sdesc(sdS + (kk >> 2) * 16384 + (kk & 3) * 32, 16, 1024),
                    make_sdesc(sTh + kk * 2048, 16, 1024), idesc_dq, 1u);
          for (int kk = 0; kk < a.tw_pad / 16; ++kk)
            umma_ss(tdQ, make_sdesc(sdS + 32768 + (kk >> 2) * 16384 + (kk & 3) * 32, 16, 1024),
                    make_sdesc(sTw + kk * 2048, 16, 1024), idesc_dq, 1u);
          umma_commit(bar_e);  // completion #2 (parity 1); the table-gradient MMAs: warp 9 -> bar_e2
        }
        __syncwarp();
      } else {
      // ---- epilogue phase 1: dQ += Gh^ . T_h ; dT_h = Gh^^T . Q ----
      mbar_wait(bar_er, 0);
      mbar_wait(bar_t, 0);
      tc_fence_after();
      if (elect_one()) {
        for (int kk = 0; kk < a.th_pad / 16; ++kk)
          umma_ss(tdQ, make_sdesc(sdS + (kk >> 2) * 16384 + (kk & 3) * 32, 16, 1024),
                  make_sdesc(sTh + kk * 2048, 16, 1024), idesc_dq, 1u);
        for (int mh = 0; mh * 128 < a.th_pad; ++mh)
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_ss(tS + mh * 64, make_sdesc(sdS + (2 * mh) * 16384 + kk * 2048, 16384, 1024),
                    make_sdesc(sQ + kk * 2048, 16, 1024), idesc_tt, kk != 0);
        umma_commit(bar_e);  // completion #2 (parity 1)
      }
      __syncwarp();
      // ---- epilogue phase 2: dQ += Gw^ . T_w ; dT_w = Gw^^T . Q ----
      mbar_wait(bar_er, 1);
      tc_fence_after();
      if (elect_one()) {
        for (int kk = 0; kk < a.tw_pad / 16; ++kk)
          umma_ss(tdQ, make_sdesc(sdS + (kk >> 2) * 16384 + (kk & 3) * 32, 16, 1024),
                  make_sdesc(sTw + kk * 2048, 16, 1024), idesc_dq, 1u);
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)
          umma_ss(tS, make_sdesc(sdS + kk * 2048, 16384, 1024), make_sdesc(sQ + kk * 2048, 16, 1024), idesc_tt,
                  kk != 0);
        umma_commit(bar_e);  // completion #3 (parity 0)
      }
      __syncwarp();
      }
    }
  } else {
    // ------------------------------------ softmax warps ------------------------------------
    // 8 warps: warps 0..3 own key columns [0,56) of every tile, warps 4..7 columns [56,112) (warp 8 = TMA, warps 9 / 10 =
    // MMA issuers: highest ids win the issue arbitration, they are the critical path); the two warps with
    // the same (warp & 3) share the 32 TMEM lanes (= query rows) of that quarter.
    constexpr int RH = R / 2;  // image rows per half tile (56 % W == 0 for every supported W)
    static_assert(RH * 2 == R && (AB_KT / 2) % W == 0, "tile halves must be whole image rows");
    const int quarter = warp & 3;
    const int half = warp >> 2;
    const int cbase = half * (AB_KT / 2);
    const int row = quarter * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(quarter * 32) << 16;
    int t = q0 + row;
    const bool valid = t < a.N;
    if (!valid) t = a.N - 1;
    const int i_r = t / W, j_r = t - i_r * W;
    const int ldr = h + 1;
    float* my_relh = relh_gen + static_cast<size_t>(row) * ldr;
    float* my_gh = my_relh;  // rel_h[i] is consumed (tile i / R) before Gh'[i] is produced: same storage
    const size_t bh = static_cast<size_t>(b) * a.heads + head;
    // this CTA's slice of the table-gradient workspace: [2h-1 + 2W-1][64] fp32 partial sums (plain stores; a
    // reduction kernel adds the slices - 1664 CTAs x 10.6 K same-address atomics were ~half of this kernel's time)
    const size_t ws_rows = static_cast<size_t>(2 * h - 1 + 2 * W - 1);
    float* ws_cta = a.dt_ws + (bh * gridDim.x + blockIdx.x) * ws_rows * 64;

    if (row == 0 && half == 0) AB_TRACE(0, 1, 15, 0);
    // delta = rowsum(dO * O) comes from attn_delta_kernel (coalesced pre-pass), LSE from the forward
    const float delta = a.delta[bh * a.N + t];
    const float lse = a.lse[bh * a.N + t];

    if (row == 0 && half == 0) AB_TRACE(0, 1, 15, 1);
    // ---- rel_w -> registers (+ global for kernel B) ----
    float relw[W];
    if (a.rel_ready) {
      // bias rows kept by the forward: rel_w as W/4 coalesced 16-byte loads, this column half's rel_h values (the
      // image rows it will meet in the main loop - no other thread reads or writes them) into the private smem row
      const float* pw = a.relw_g + (bh * gridDim.x + blockIdx.x) * static_cast<size_t>(W) * AB_BM;
      if constexpr (W % 4 == 0) {
#pragma unroll
        for (int j = 0; j < W / 4; ++j) {
          const float4 q4 = __ldg(reinterpret_cast<const float4*>(pw) + j * AB_BM + row);
          relw[4 * j] = q4.x; relw[4 * j + 1] = q4.y; relw[4 * j + 2] = q4.z; relw[4 * j + 3] = q4.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < W; ++j) relw[j] = __ldg(pw + j * AB_BM + row);
      }
      // (batches of 32 independent read-only loads, then the smem stores: every dependent round trip to global memory
      // costs ~2 k cycles here - a load-store-load chain per image row measured 8.7 k cycles, two batches of 16 still 7 k)
      const float* ph = a.relh_g + (bh * gridDim.x + blockIdx.x) * static_cast<size_t>(h) * AB_BM + row;
      constexpr int CH = RH >= 32 ? 1 : 32 / RH;   // tiles per batch (56 x 28 grid: all 14 tiles in ONE round trip)
      for (int jb = 0; jb < num_tiles; jb += CH) {
        float tmp[CH][RH];
#pragma unroll
        for (int jj = 0; jj < CH; ++jj)
#pragma unroll
          for (int r = 0; r < RH; ++r) {
            const int i = (jb + jj) * R + half * RH + r;
            tmp[jj][r] = i < h ? __ldg(ph + static_cast<size_t>(i) * AB_BM) : 0.f;
          }
#pragma unroll
        for (int jj = 0; jj < CH; ++jj)
#pragma unroll
          for (int r = 0; r < RH; ++r) {
            const int i = (jb + jj) * R + half * RH + r;
            if (i < h) my_relh[i] = tmp[jj][r];
          }
      }
    } else {
    {
      float* scratch = relh_gen + (static_cast<size_t>(half) * 128 + row) * 17;
      mbar_wait(bar_g, 0);
      tc_fence_after();
      for (int c0 = 0; c0 < a.tw_pad; c0 += 16) {
        uint32_t v[16];
        tmem_ld_x16(tS + lane_addr + c0, v);
        tmem_wait_ld();
#pragma unroll
        for (int c = 0; c < 16; ++c) scratch[c] = __uint_as_float(v[c]) * AB_LOG2E;
#pragma unroll
        for (int j = 0; j < W; ++j) {
          const int tt = j_r + (W - 1) - j - c0;
          if (tt >= 0 && tt < 16) relw[j] = scratch[tt];
        }
      }
      tc_fence_before();
      __syncwarp();
      mbar_arrive(bar_gr);
      if (half == 0) {
        // every row of the tile is written (rows past N hold the finite values of the clamped token: kernel B masks
        // them through its -inf row bias but must not meet uninitialised memory)
        float* dst = a.relw_g + (bh * gridDim.x + blockIdx.x) * static_cast<size_t>(W) * AB_BM;
        if constexpr (W % 4 == 0) {
#pragma unroll
          for (int j = 0; j < W / 4; ++j)
            reinterpret_cast<float4*>(dst)[j * AB_BM + row] =
                make_float4(relw[4 * j], relw[4 * j + 1], relw[4 * j + 2], relw[4 * j + 3]);
        } else {
#pragma unroll
          for (int j = 0; j < W; ++j) dst[j * AB_BM + row] = relw[j];
        }
      }
    }
    if (row == 0 && half == 0) AB_TRACE(0, 1, 15, 2);
    // ---- rel_h -> smem (+ global): written by half 0, read by both halves after the first bar_s ----
    {
      mbar_wait(bar_g, 1);
      tc_fence_after();
      // 16-row chunks of the table alternate between the two column halves (both own the same 32 TMEM lanes)
      for (int c0 = half * 16; c0 < a.th_pad; c0 += 32) {
        uint32_t v[16];
        tmem_ld_x16(tS + lane_addr + c0, v);
        tmem_wait_ld();
#pragma unroll
        for (int c = 0; c < 16; ++c) {
          const int i = i_r + (h - 1) - (c0 + c);
          if (i >= 0 && i < h) my_relh[i] = __uint_as_float(v[c]) * AB_LOG2E;
        }
      }
      tc_fence_before();
      asm volatile("bar.sync 1, %0;" ::"n"(AB_SMX) : "memory");
      // rel_h rows to global for kernel B, row-innermost: each thread copies its own row (the two column halves take
      // alternate image rows): smem reads at stride h+1 floats (odd: conflict-free), global stores of 128 contiguous
      // bytes per warp.  It finishes before the arrive below, i.e. before any thread can start overwriting rel_h rows
      // with Gh' (first bar_s needs all arrivals)
      {
        float* dst = a.relh_g + (bh * gridDim.x + blockIdx.x) * static_cast<size_t>(h) * AB_BM + row;
        for (int i = half; i < h; i += 2) dst[static_cast<size_t>(i) * AB_BM] = my_relh[i];
      }
      __syncwarp();
      mbar_arrive(bar_gr);
    }
    }
    if (row == 0 && half == 0) AB_TRACE(0, 1, 15, 3);
    // Per-score arithmetic on packed fp32 pairs (FFMA2 / FADD2 / FMUL2) when W is even (a pair of adjacent keys then
    // shares its image row): bias add, scale-fma, (dP - delta), p * (.), row-sum and column-sum accumulations cost
    // one issue slot per two scores.  Masking costs nothing: invalid image rows / query rows get a bias of -inf,
    // so p = exp2(-inf) = 0 and dS = 0 (S and dP of out-of-range rows are finite: TMA zero-fills them).
    constexpr bool PK2 = (W % 2 == 0);
    float gw[W];
    f32x2 gw2[PK2 ? W / 2 : 1], relw2[PK2 ? W / 2 : 1];
#pragma unroll
    for (int j = 0; j < W; ++j) gw[j] = 0.f;
    if constexpr (PK2) {
#pragma unroll
      for (int j = 0; j < W / 2; ++j) {
        gw2[j] = pack_f2(0.f, 0.f);
        relw2[j] = pack_f2(relw[2 * j], relw[2 * j + 1]);
      }
    }
    const float sc = a.scale_log2;
    const f32x2 sc2 = pack_f2(sc, sc), nd2 = pack_f2(-delta, -delta);
    for (int j = 0; j < num_tiles; ++j) {
      if (row == 0 && half == 0) AB_TRACE(0, 1, j, 0);
      mbar_wait(bar_s + 8 * (j & 1), (j >> 1) & 1);
      if (row == 0 && half == 0) AB_TRACE(0, 1, j, 1);
      tc_fence_after();
      float hb[RH], gh[RH];
      f32x2 hb2[RH], gh2[RH];
#pragma unroll
      for (int r = 0; r < RH; ++r) {
        const int i = j * R + half * RH + r;
        hb[r] = (i < h && valid) ? my_relh[i] - lse : -INFINITY;
        gh[r] = 0.f;
        hb2[r] = pack_f2(hb[r], hb[r]);
        gh2[r] = pack_f2(0.f, 0.f);
      }
      const uint32_t tS_h = tS + (j & 1) * 224 + lane_addr + cbase, tdP_h = tS_h + 112;
      const uint32_t sdS_j = sdS + (j & 1) * 32768;
      if (j >= 2) mbar_wait(bar_df + 8 * (j & 1), ((j >> 1) - 1) & 1);  // dQ(j-2) has drained this dS buffer
      // 56 columns per thread as 7 chunks of 8, software-pipelined: the TMEM loads of chunk ci + 1 are in flight
      // while chunk ci is processed (two softmax warps per scheduler cannot hide a tcgen05.ld round trip per chunk)
      uint32_t v[2][8], w[2][8];
      tmem_ld_x8(tS_h, v[0]);
      tmem_ld_x8(tdP_h, w[0]);
#pragma unroll
      for (int ci = 0; ci < 7; ++ci) {
        const int c0 = ci * 8;
        tmem_wait_ld();
        if (ci + 1 < 7) {
          tmem_ld_x8(tS_h + c0 + 8, v[(ci + 1) & 1]);
          tmem_ld_x8(tdP_h + c0 + 8, w[(ci + 1) & 1]);
        }
        uint32_t dsb[4];
#pragma unroll
        for (int c = 0; c < 8; c += 2) {
          const int kc = c0 + c;
          const uint32_t v0 = v[ci & 1][c], v1 = v[ci & 1][c + 1], w0 = w[ci & 1][c], w1 = w[ci & 1][c + 1];
          float d0, d1;
          if constexpr (PK2) {
            const f32x2 t2 = fma_f2(pack_u2(v0, v1), sc2, add_f2(hb2[kc / W], relw2[(kc % W) / 2]));
            float t0, t1;
            unpack_f2(t2, t0, t1);
            float p0, p1;
            exp2_pair<PK_EXP_POLY_MASK_DQ>(c >> 1, t0, t1, p0, p1);
            const f32x2 d2 = mul_f2(pack_f2(p0, p1), add_f2(pack_u2(w0, w1), nd2));
            gh2[kc / W] = add_f2(gh2[kc / W], d2);
            gw2[(kc % W) / 2] = add_f2(gw2[(kc % W) / 2], d2);
            unpack_f2(d2, d0, d1);
          } else {
            const int k1 = kc + 1;
            d0 = fast_exp2(fmaf(__uint_as_float(v0), sc, hb[kc / W] + relw[kc % W])) * (__uint_as_float(w0) - delta);
            d1 = fast_exp2(fmaf(__uint_as_float(v1), sc, hb[k1 / W] + relw[k1 % W])) * (__uint_as_float(w1) - delta);
            gh[kc / W] += d0;
            gh[k1 / W] += d1;
            gw[kc % W] += d0;
            gw[k1 % W] += d1;
          }
          dsb[c / 2] = pack_bf16x2(d0, d1);
        }
        const int g8 = (cbase + c0) >> 3;  // 8-column group inside the 112-wide tile
        st_shared_v4(sdS_j + (g8 >> 3) * 16384 + row * 128 + (((g8 & 7) ^ (row & 7)) << 4), dsb[0], dsb[1], dsb[2],
                     dsb[3]);
      }
#pragma unroll
      for (int r = 0; r < RH; ++r) {
        const int i = j * R + half * RH + r;
        if constexpr (PK2) {
          float g0, g1;
          unpack_f2(gh2[r], g0, g1);
          gh[r] = g0 + g1;
        }
        if (i < h) my_gh[i] = gh[r];
      }
      if (row == 0 && half == 0) AB_TRACE(0, 1, j, 2);
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive((j & 1) ? bar_p1 : bar_p0);
      if (row == 0 && half == 0) AB_TRACE(0, 1, j, 3);
    }
    if constexpr (PK2) {
#pragma unroll
      for (int j = 0; j < W / 2; ++j) unpack_f2(gw2[j], gw[2 * j], gw[2 * j + 1]);
    }

    if (row == 0 && half == 0) AB_TRACE(0, 1, 15, 4);
    __nv_bfloat16* qrow = a.dqkv + (static_cast<size_t>(b) * a.N + t) * (3 * C) + head * 64 + half * 32;
    if (merged_ep) {
      // ---------------- single-phase epilogue ----------------
      // Gw' totals of the two column halves through the dO tile (dead once the main loop has retired; row stride W+1
      // floats: conflict-free), then both Toeplitz operands x 8 as bf16 16-byte chunks: Gh^ -> dS buffer 0, Gw^ ->
      // dS buffer 1 (dS is stored unscaled: the accumulator holds 8 * dQ_bias + dS.K, the read-out multiplies by 1/8)
      mbar_wait(bar_e, 0);
      tc_fence_after();
      float* xch = reinterpret_cast<float*>(gen + A_SDO) + static_cast<size_t>(row) * (W + 1);
      if (half == 1) {
#pragma unroll
        for (int j = 0; j < W; ++j) xch[j] = gw[j];
      }
      for (int c0 = half * 8; c0 < a.th_pad; c0 += 16) {
        float g[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const int i = i_r + (h - 1) - (c0 + c);
          g[c] = (i >= 0 && i < h) ? my_gh[i] * 8.0f : 0.f;
        }
        const uint32_t addr = sdS + (c0 >> 6) * 16384 + row * 128 + ((((c0 & 63) >> 3) ^ (row & 7)) << 4);
        st_shared_v4(addr, pack_bf16x2(g[0], g[1]), pack_bf16x2(g[2], g[3]), pack_bf16x2(g[4], g[5]),
                     pack_bf16x2(g[6], g[7]));
      }
      asm volatile("bar.sync 1, %0;" ::"n"(AB_SMX) : "memory");
      if (half == 0) {
#pragma unroll
        for (int j = 0; j < W; ++j) xch[j] += gw[j];
      }
      asm volatile("bar.sync 1, %0;" ::"n"(AB_SMX) : "memory");
      for (int c0 = half * 8; c0 < a.tw_pad; c0 += 16) {
        float g[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const int j = j_r + (W - 1) - (c0 + c);
          g[c] = (j >= 0 && j < W) ? xch[j] * 8.0f : 0.f;
        }
        const uint32_t addr = sdS + 32768 + (c0 >> 6) * 16384 + row * 128 + ((((c0 & 63) >> 3) ^ (row & 7)) << 4);
        st_shared_v4(addr, pack_bf16x2(g[0], g[1]), pack_bf16x2(g[2], g[3]), pack_bf16x2(g[4], g[5]),
                     pack_bf16x2(g[6], g[7]));
      }
      // the dT MMAs read 128 operand columns (M = 128) of each buffer: zero what lies beyond th_pad / tw_pad
      for (int c0 = a.th_pad + half * 8; c0 < 128; c0 += 16) {
        const uint32_t addr = sdS + (c0 >> 6) * 16384 + row * 128 + ((((c0 & 63) >> 3) ^ (row & 7)) << 4);
        st_shared_v4(addr, 0u, 0u, 0u, 0u);
      }
      for (int c0 = a.tw_pad + half * 8; c0 < 128; c0 += 16) {
        const uint32_t addr = sdS + 32768 + (c0 >> 6) * 16384 + row * 128 + ((((c0 & 63) >> 3) ^ (row & 7)) << 4);
        st_shared_v4(addr, 0u, 0u, 0u, 0u);
      }
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(bar_er);
      if (row == 0 && half == 0) AB_TRACE(0, 1, 15, 5);
      // ---------------- read-out: dT_h / dT_w partials, dQ -> bf16 (each half owns 32 of the 64 columns) ----------
      mbar_wait(bar_e2, 0);
      tc_fence_after();
      if (row == 0 && half == 0) AB_TRACE(0, 1, 15, 6);
      for (int mh = 0; mh * 128 < a.th_pad; ++mh) {
        const int tt = mh * 128 + row;
#pragma unroll
        for (int c0 = 0; c0 < 32; c0 += 16) {
          uint32_t v[16];
          tmem_ld_x16(tS + lane_addr + mh * 64 + half * 32 + c0, v);
          tmem_wait_ld();
          if (tt < 2 * h - 1) {
            float* dst = ws_cta + static_cast<size_t>(half * 32 + c0) * ws_rows + tt;
#pragma unroll
            for (int q = 0; q < 16; ++q) dst[static_cast<size_t>(q) * ws_rows] = __uint_as_float(v[q]) * 0.125f;
          }
        }
      }
#pragma unroll
      for (int c0 = 0; c0 < 32; c0 += 16) {
        uint32_t v[16];
        tmem_ld_x16(tS + lane_addr + 128 + half * 32 + c0, v);
        tmem_wait_ld();
        if (row < 2 * W - 1) {
          float* dst = ws_cta + static_cast<size_t>(half * 32 + c0) * ws_rows + (2 * h - 1 + row);
#pragma unroll
          for (int q = 0; q < 16; ++q) dst[static_cast<size_t>(q) * ws_rows] = __uint_as_float(v[q]) * 0.125f;
        }
      }
      mbar_wait(bar_e, 1);
      tc_fence_after();
#pragma unroll
      for (int c0 = 0; c0 < 32; c0 += 16) {
        uint32_t o[16];
        tmem_ld_x16(tdQ + lane_addr + half * 32 + c0, o);
        tmem_wait_ld();
        if (valid) {
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            uint4 u;
            u.x = pack_bf16x2(__uint_as_float(o[q * 8 + 0]) * 0.125f, __uint_as_float(o[q * 8 + 1]) * 0.125f);
            u.y = pack_bf16x2(__uint_as_float(o[q * 8 + 2]) * 0.125f, __uint_as_float(o[q * 8 + 3]) * 0.125f);
            u.z = pack_bf16x2(__uint_as_float(o[q * 8 + 4]) * 0.125f, __uint_as_float(o[q * 8 + 5]) * 0.125f);
            u.w = pack_bf16x2(__uint_as_float(o[q * 8 + 6]) * 0.125f, __uint_as_float(o[q * 8 + 7]) * 0.125f);
            *reinterpret_cast<uint4*>(qrow + c0 + q * 8) = u;
          }
        }
      }
      if (row == 0 && half == 0) AB_TRACE(0, 1, 15, 7);
    } else {
    // ---------------- epilogue phase 1: Gh^ x 8 (bf16, K-major / MN-major dual view) ----------------
    // (dS is stored unscaled, so the accumulator holds 8 * dQ_bias + dS.K; the final read-out multiplies by 1/8)
    mbar_wait(bar_e, 0);
    tc_fence_after();
    for (int c0 = half * 8; c0 < a.th_pad; c0 += 16) {
      float g[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int i = i_r + (h - 1) - (c0 + c);
        g[c] = (i >= 0 && i < h) ? my_gh[i] * 8.0f : 0.f;
      }
      const uint32_t addr = sdS + (c0 >> 6) * 16384 + row * 128 + ((((c0 & 63) >> 3) ^ (row & 7)) << 4);
      st_shared_v4(addr, pack_bf16x2(g[0], g[1]), pack_bf16x2(g[2], g[3]), pack_bf16x2(g[4], g[5]),
                   pack_bf16x2(g[6], g[7]));
    }
    fence_proxy_async_smem();
    tc_fence_before();
    mbar_arrive(bar_er);
    if (row == 0 && half == 0) AB_TRACE(0, 1, 15, 5);
    // ---------------- epilogue phase 2: dT_h partials, then Gw^ x 8 ----------------
    mbar_wait(bar_e, 1);
    tc_fence_after();
    for (int mh = 0; mh * 128 < a.th_pad; ++mh) {
      const int tt = mh * 128 + row;
#pragma unroll
      for (int c0 = 0; c0 < 32; c0 += 16) {
        uint32_t v[16];
        tmem_ld_x16(tS + lane_addr + mh * 64 + half * 32 + c0, v);
        tmem_wait_ld();
        if (tt < 2 * h - 1) {
          float* dst = ws_cta + static_cast<size_t>(half * 32 + c0) * ws_rows + tt;
#pragma unroll
          for (int q = 0; q < 16; ++q) dst[static_cast<size_t>(q) * ws_rows] = __uint_as_float(v[q]) * 0.125f;
        }
      }
    }
    {
      // Total column sums Gw'[row][j] (both column halves) through smem (the rel_h / Gh' rows are dead by now), then
      // the Toeplitz re-indexed operand row Gw^[row][t] = 8 * Gw'[row][j_r + W-1 - t] is assembled from them in
      // registers and written as whole 16-byte chunks, the two halves sharing the chunks.  (Round 1 scattered 2-byte
      // stores instead: 32 rows of a warp hit one bank - a 32-way conflict per store, ~3.5 k cycles per CTA.)
      float* xch = relh_gen + static_cast<size_t>(row) * (W + 1);     // row stride W+1 floats: conflict-free
      if (half == 1) {
#pragma unroll
        for (int j = 0; j < W; ++j) xch[j] = gw[j];
      }
      asm volatile("bar.sync 1, %0;" ::"n"(AB_SMX) : "memory");
      if (half == 0) {
#pragma unroll
        for (int j = 0; j < W; ++j) xch[j] += gw[j];
      }
      asm volatile("bar.sync 1, %0;" ::"n"(AB_SMX) : "memory");
      for (int c0 = half * 8; c0 < a.tw_pad; c0 += 16) {
        float g[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const int j = j_r + (W - 1) - (c0 + c);
          g[c] = (j >= 0 && j < W) ? xch[j] * 8.0f : 0.f;
        }
        const uint32_t addr = sdS + (c0 >> 6) * 16384 + row * 128 + ((((c0 & 63) >> 3) ^ (row & 7)) << 4);
        st_shared_v4(addr, pack_bf16x2(g[0], g[1]), pack_bf16x2(g[2], g[3]), pack_bf16x2(g[4], g[5]),
                     pack_bf16x2(g[6], g[7]));
      }
      // the dT_w MMAs read 128 operand columns (M = 128): zero what lies beyond tw_pad
      for (int c0 = a.tw_pad + half * 8; c0 < 128; c0 += 16) {
        const uint32_t addr = sdS + (c0 >> 6) * 16384 + row * 128 + ((((c0 & 63) >> 3) ^ (row & 7)) << 4);
        st_shared_v4(addr, 0u, 0u, 0u, 0u);
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    mbar_arrive(bar_er);
    if (row == 0 && half == 0) AB_TRACE(0, 1, 15, 6);
    // ---------------- epilogue phase 3: dT_w partials, dQ -> bf16 (each half owns 32 of the 64 columns) -----------
    mbar_wait(bar_e, 0);
    tc_fence_after();
#pragma unroll
    for (int c0 = 0; c0 < 32; c0 += 16) {
      uint32_t v[16];
      tmem_ld_x16(tS + lane_addr + half * 32 + c0, v);
      tmem_wait_ld();
      if (row < 2 * W - 1) {
        float* dst = ws_cta + static_cast<size_t>(half * 32 + c0) * ws_rows + (2 * h - 1 + row);
#pragma unroll
        for (int q = 0; q < 16; ++q) dst[static_cast<size_t>(q) * ws_rows] = __uint_as_float(v[q]) * 0.125f;
      }
    }
#pragma unroll
    for (int c0 = 0; c0 < 32; c0 += 16) {
      uint32_t o[16];
      tmem_ld_x16(tdQ + lane_addr + half * 32 + c0, o);
      tmem_wait_ld();
      if (valid) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          uint4 u;
          u.x = pack_bf16x2(__uint_as_float(o[q * 8 + 0]) * 0.125f, __uint_as_float(o[q * 8 + 1]) * 0.125f);
          u.y = pack_bf16x2(__uint_as_float(o[q * 8 + 2]) * 0.125f, __uint_as_float(o[q * 8 + 3]) * 0.125f);
          u.z = pack_bf16x2(__uint_as_float(o[q * 8 + 4]) * 0.125f, __uint_as_float(o[q * 8 + 5]) * 0.125f);
          u.w = pack_bf16x2(__uint_as_float(o[q * 8 + 6]) * 0.125f, __uint_as_float(o[q * 8 + 7]) * 0.125f);
          *reinterpret_cast<uint4*>(qrow + c0 + q * 8) = u;
        }
      }
    }
    if (row == 0 && half == 0) AB_TRACE(0, 1, 15, 7);
    }
  }

  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 9) tmem_dealloc(tmem, 512);
}

// ================================================================================================
// Kernel B
// ================================================================================================
constexpr uint32_t B_SK = 0;                 // K tile 112 x 128 B
constexpr uint32_t B_SV = 14336;             // V tile
constexpr uint32_t B_SQ = 28672;             // 3 stages x (Q 16384 | dO 16384): deep enough to hide the TMA latency
constexpr uint32_t B_SP = B_SQ + 98304;      // 2 x P tile  (2 K-blocks each, double-buffered)
constexpr uint32_t B_SDS = B_SP + 65536;     // dS tile (single: the dK MMAs of tile i are issued first and release it)
constexpr uint32_t B_BARS = B_SDS + 32768;

template <int W>
__global__ void __launch_bounds__(AB_THREADS, 1)
attn_bwd_dkv_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                    const __grid_constant__ CUtensorMap tmdO, const AttnBwdArgs a) {
  constexpr int R = AB_KT / W;
  AB_TRACE_INIT();
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_base = smem_u32(smem_raw);
  const uint32_t base = (raw_base + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - raw_base);
  const uint32_t sK = base + B_SK, sV = base + B_SV, sQ0 = base + B_SQ, sP = base + B_SP, sdS = base + B_SDS;
  const uint32_t bar0 = base + B_BARS;
  const uint32_t bar_kv = bar0, bar_qf = bar0 + 8 /*3*/, bar_qe = bar0 + 32 /*3*/, bar_s = bar0 + 56 /*2*/,
                 bar_p0 = bar0 + 72, bar_o = bar0 + 80, bar_dp = bar0 + 88 /* +136 */, bar_dsf = bar0 + 96,
                 bar_p1 = bar0 + 112, bar_pe = bar0 + 120 /*2*/, bar_dp1 = bar0 + 136, bar_sc = bar0 + 144 /*2*/;
  const uint32_t holder = bar0 + 104;
  volatile uint32_t* holder_gen = reinterpret_cast<volatile uint32_t*>(gen + B_BARS + 104);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int jt = blockIdx.x;  // key tile
  const int head = blockIdx.y, b = blockIdx.z;
  const int C = a.heads * 64;
  const int h = a.h;
  const int num_q = (a.N + AB_BM - 1) / AB_BM;

  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmKV);
    tma_prefetch_desc(&tmdO);
    mbar_init(bar_kv, 1);
    for (int q = 0; q < 3; ++q) {
      mbar_init(bar_qf + 8 * q, 1);
      mbar_init(bar_qe + 8 * q, 1);
    }
    mbar_init(bar_s, 1);
    mbar_init(bar_s + 8, 1);
    mbar_init(bar_dp, 1);
    mbar_init(bar_dp1, 1);
    mbar_init(bar_sc, AB_SMX / 32);
    mbar_init(bar_sc + 8, AB_SMX / 32);
    mbar_init(bar_dsf, 1);
    mbar_init(bar_p0, AB_SMX / 32);
    mbar_init(bar_p1, AB_SMX / 32);
    mbar_init(bar_pe, 1);
    mbar_init(bar_pe + 8, 1);
    mbar_init(bar_o, 1);
    fence_barrier_init();
  }
  if (warp == 9) tmem_alloc(holder, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *holder_gen;
  // Three 112-column score buffers rotate between S and dP (dV at 336, dK at 400): tile i keeps S in buffer
  // s_i = (3 - i % 3) % 3 and dP in d_i = (s_i + 1) % 3.  S(i+1) lands in the third buffer while tile i is being
  // processed; dP(i+1) reuses S(i)'s buffer as soon as the softmax warps have finished their first pass (p = exp2(.)
  // needs S only), so neither score MMA of the next tile waits for the end of the current one.
  const uint32_t tS = tmem, tdV = tmem + 336, tdK = tmem + 400;
  pdl_launch_dependents();
  pdl_wait();

  if (warp == 8) {
    if (lane == 0) {
      mbar_expect_tx(bar_kv, 2 * AB_KT * 128);
      tma_load_3d(sK, &tmKV, bar_kv, C + head * 64, jt * AB_KT, b);
      tma_load_3d(sV, &tmKV, bar_kv, 2 * C + head * 64, jt * AB_KT, b);
      for (int i = 0; i < num_q; ++i) {
        const int st = i % 3;
        if (i >= 3) mbar_wait(bar_qe + 8 * st, ((i / 3) - 1) & 1);
        mbar_expect_tx(bar_qf + 8 * st, 32768);
        tma_load_3d(sQ0 + st * 32768, &tmQ, bar_qf + 8 * st, head * 64, i * AB_BM, b);
        tma_load_3d(sQ0 + st * 32768 + 16384, &tmdO, bar_qf + 8 * st, head * 64, i * AB_BM, b);
      }
    }
  } else if (warp == 9) {
    {
      const uint32_t idesc_s = make_idesc_bf16(128, AB_KT, false, false);
      const uint32_t idesc_tt = make_idesc_bf16(128, 64, true, true);
      mbar_wait(bar_kv, 0);
      const uint64_t dK0 = make_sdesc(sK, 16, 1024), dV0 = make_sdesc(sV, 16, 1024);
      // Pipeline: S(i+1) is issued while the softmax warps work on tile i; dP(i+1) right after they hand back
      // tile i, ahead of the 16 accumulation MMAs of tile i, so the next softmax pass overlaps those.
      auto issue_s = [&](int i) {
        const int qs = i % 3;
        const uint64_t dQ0 = make_sdesc(sQ0 + qs * 32768, 16, 1024);
        mbar_wait(bar_qf + 8 * qs, (i / 3) & 1);
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_ss(tS + ((3 - i % 3) % 3) * 112, sdesc_add(dQ0, k * 32), sdesc_add(dK0, k * 32), idesc_s, k != 0);
          umma_commit(bar_s + 8 * (i & 1));
        }
        __syncwarp();
      };
      auto issue_dp = [&](int i) {
        const uint64_t ddO0 = make_sdesc(sQ0 + (i % 3) * 32768 + 16384, 16, 1024);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_ss(tS + ((4 - i % 3) % 3) * 112, sdesc_add(ddO0, k * 32), sdesc_add(dV0, k * 32), idesc_s, k != 0);
          umma_commit((i & 1) ? bar_dp1 : bar_dp);
        }
        __syncwarp();
      };
      // Scores issuer (buffer rotation above): dP(i+1) after the first softmax pass of tile i (bar_sc), S(i+2) after
      // the whole of tile i (bar_p).  The 16 accumulation MMAs of a tile are issued by warp 10.
      issue_s(0);
      issue_dp(0);
      if (num_q > 1) issue_s(1);
      for (int i = 0; i + 1 < num_q; ++i) {
        AB_TRACE(1, 0, i, 0);
        mbar_wait(bar_sc + 8 * (i & 1), (i >> 1) & 1);
        tc_fence_after();
        issue_dp(i + 1);
        AB_TRACE(1, 0, i, 5);
        if (i + 2 < num_q) {
          mbar_wait((i & 1) ? bar_p1 : bar_p0, (i >> 1) & 1);
          tc_fence_after();
          issue_s(i + 2);
          AB_TRACE(1, 0, i, 2);
        }
      }
    }
  } else if (warp == 10) {
    {
      // ------------------------------ accumulation issuer (dK, dV) ------------------------------
      const uint32_t idesc_tt = make_idesc_bf16(128, 64, true, true);
      for (int i = 0; i < num_q; ++i) {
        const int qs = i % 3;
        mbar_wait((i & 1) ? bar_p1 : bar_p0, (i >> 1) & 1);
        AB_TRACE(1, 0, i, 3);
        tc_fence_after();
        const uint64_t dQ0 = make_sdesc(sQ0 + qs * 32768, 16, 1024), ddO0 = make_sdesc(sQ0 + qs * 32768 + 16384, 16, 1024);
        const uint64_t dP0 = make_sdesc(sP + (i & 1) * 32768, 16384, 1024), ddS0 = make_sdesc(sdS, 16384, 1024);
        // dK[keys, d] += dS^T . Q first (releases the single dS buffer), then dV[keys, d] += P^T . dO
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_ss(tdK, sdesc_add(ddS0, kk * 2048), sdesc_add(dQ0, kk * 2048), idesc_tt, (i | kk) != 0);
          umma_commit(bar_dsf);
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_ss(tdV, sdesc_add(dP0, kk * 2048), sdesc_add(ddO0, kk * 2048), idesc_tt, (i | kk) != 0);
          umma_commit(bar_qe + 8 * qs);        // Q/dO stage free (S(i), dP(i) retired before p(i))
          umma_commit(bar_pe + 8 * (i & 1));   // P buffer free
        }
        __syncwarp();
        AB_TRACE(1, 0, i, 4);
      }
      if (elect_one()) umma_commit(bar_o);
      __syncwarp();
    }
  } else {
    // 8 softmax warps, same column split as kernel A
    constexpr int RH = R / 2;
    const int quarter = warp & 3;
    const int half = warp >> 2;
    const int cbase = half * (AB_KT / 2);
    const int row = quarter * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(quarter * 32) << 16;
    const size_t bh = static_cast<size_t>(b) * a.heads + head;
    const float sc = a.scale_log2;
    const int keys_valid = (h - jt * R) * W - cbase;
    // Per-row operands of a query tile (LSE, delta, R/2 rel_h values, W rel_w values) come from global memory:
    // they are fetched one tile AHEAD into registers so that their latency hides behind the current tile's work.
    float lse_n = 0.f, delta_n = 0.f, hb_n[RH], relw_n[W];
    bool valid_n = false;
    auto fetch = [&](int i) {
      int t = i * AB_BM + row;
      valid_n = t < a.N;
      if (!valid_n) t = a.N - 1;
      lse_n = a.lse[bh * a.N + t];
      delta_n = a.delta[bh * a.N + t];
      // row-innermost tiles written by kernel A: coalesced (128 B per warp for rel_h, 512 B per warp for rel_w)
      const float* ph = a.relh_g + (bh * num_q + i) * static_cast<size_t>(h) * AB_BM + row;
#pragma unroll
      for (int r = 0; r < RH; ++r) {
        const int ii = jt * R + half * RH + r;
        hb_n[r] = ph[static_cast<size_t>(ii < h ? ii : h - 1) * AB_BM];
      }
      const float* pw = a.relw_g + (bh * num_q + i) * static_cast<size_t>(W) * AB_BM;
      if constexpr (W % 4 == 0) {
#pragma unroll
        for (int j = 0; j < W / 4; ++j) {
          const float4 q4 = reinterpret_cast<const float4*>(pw)[j * AB_BM + row];
          relw_n[4 * j] = q4.x; relw_n[4 * j + 1] = q4.y; relw_n[4 * j + 2] = q4.z; relw_n[4 * j + 3] = q4.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < W; ++j) relw_n[j] = pw[j * AB_BM + row];
      }
    };
    fetch(0);
    for (int i = 0; i < num_q; ++i) {
      // packed fp32 pairs + -inf masking as in kernel A (invalid key rows of this tile / invalid query rows -> p = 0)
      constexpr bool PK2 = (W % 2 == 0);
      if (row == 0 && half == 0) AB_TRACE(1, 1, i, 5);
      const bool valid = valid_n;
      const float lse = lse_n, delta = delta_n;
      float hb[RH], relw[W];
      f32x2 hb2[RH], relw2[PK2 ? W / 2 : 1];
#pragma unroll
      for (int r = 0; r < RH; ++r) {
        hb[r] = (valid && r * W < keys_valid) ? hb_n[r] - lse : -INFINITY;
        hb2[r] = pack_f2(hb[r], hb[r]);
      }
#pragma unroll
      for (int j = 0; j < W; ++j) relw[j] = relw_n[j];
      if constexpr (PK2) {
#pragma unroll
        for (int j = 0; j < W / 2; ++j) relw2[j] = pack_f2(relw[2 * j], relw[2 * j + 1]);
      }
      const f32x2 sc2 = pack_f2(sc, sc), nd2 = pack_f2(-delta, -delta);
      if (row == 0 && half == 0 && ab_tr) {
        // debug timeline only: force the operands of this tile to have arrived before the stamp
        float chk = lse + delta + hb[0] + relw[0] + relw[W - 1];
        asm volatile("" ::"f"(chk));
        AB_TRACE(1, 1, i, 6);
      }
      if (i + 1 < num_q) fetch(i + 1);
      if (row == 0 && half == 0) AB_TRACE(1, 1, i, 0);
      mbar_wait(bar_s + 8 * (i & 1), (i >> 1) & 1);
      if (row == 0 && half == 0) AB_TRACE(1, 1, i, 4);
      tc_fence_after();
      const int sbuf = (3 - i % 3) % 3, dbuf = (sbuf + 1) % 3;
      const uint32_t tS_h = tS + sbuf * 112 + lane_addr + cbase, tdP_h = tS + dbuf * 112 + lane_addr + cbase;
      const uint32_t sP_i = sP + (i & 1) * 32768, sdS_i = sdS;
      if (i >= 2) mbar_wait(bar_pe + 8 * (i & 1), ((i >> 1) - 1) & 1);  // dV(i-2) has drained this P buffer
      // ---- pass 1: p = exp2(scale * S + bias - lse) (fp32, kept in registers for pass 2), P -> smem as bf16 ----
      f32x2 pp[AB_KT / 4];   // 56 probabilities as 28 packed pairs
      {
        uint32_t v[2][8];   // 7 chunks of 8 columns, TMEM loads one chunk ahead (see kernel A)
        tmem_ld_x8(tS_h, v[0]);
#pragma unroll
        for (int ci = 0; ci < 7; ++ci) {
          const int c0 = ci * 8;
          tmem_wait_ld();
          if (ci + 1 < 7) tmem_ld_x8(tS_h + c0 + 8, v[(ci + 1) & 1]);
          uint32_t pb[4];
#pragma unroll
          for (int c = 0; c < 8; c += 2) {
            const int kc = c0 + c;
            const uint32_t v0 = v[ci & 1][c], v1 = v[ci & 1][c + 1];
            float p0, p1;
            if constexpr (PK2) {
              float t0, t1;
              unpack_f2(fma_f2(pack_u2(v0, v1), sc2, add_f2(hb2[kc / W], relw2[(kc % W) / 2])), t0, t1);
              exp2_pair<PK_EXP_POLY_MASK_DKV>(c >> 1, t0, t1, p0, p1);
            } else {
              const int k1 = kc + 1;
              p0 = fast_exp2(fmaf(__uint_as_float(v0), sc, hb[kc / W] + relw[kc % W]));
              p1 = fast_exp2(fmaf(__uint_as_float(v1), sc, hb[k1 / W] + relw[k1 % W]));
            }
            pp[kc / 2] = pack_f2(p0, p1);
            pb[c / 2] = pack_bf16x2(p0, p1);
          }
          const int g8 = (cbase + c0) >> 3;
          const uint32_t off = (g8 >> 3) * 16384 + row * 128 + (((g8 & 7) ^ (row & 7)) << 4);
          st_shared_v4(sP_i + off, pb[0], pb[1], pb[2], pb[3]);
        }
      }
      // S(i) is consumed: its TMEM buffer may take dP(i+1)
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_sc + 8 * (i & 1));
      // ---- pass 2: dS = p * (dP - delta) -> smem as bf16 ----
      mbar_wait((i & 1) ? bar_dp1 : bar_dp, (i >> 1) & 1);
      if (row == 0 && half == 0) AB_TRACE(1, 1, i, 1);
      tc_fence_after();
      if (i >= 1) mbar_wait(bar_dsf, (i - 1) & 1);   // the dK MMAs of tile i-1 have drained the dS buffer
      {
        uint32_t w[2][8];
        tmem_ld_x8(tdP_h, w[0]);
#pragma unroll
        for (int ci = 0; ci < 7; ++ci) {
          const int c0 = ci * 8;
          tmem_wait_ld();
          if (ci + 1 < 7) tmem_ld_x8(tdP_h + c0 + 8, w[(ci + 1) & 1]);
          uint32_t dsb[4];
#pragma unroll
          for (int c = 0; c < 8; c += 2) {
            const int kc = c0 + c;
            const uint32_t w0 = w[ci & 1][c], w1 = w[ci & 1][c + 1];
            float d0, d1;
            if constexpr (PK2) {
              unpack_f2(mul_f2(pp[kc / 2], add_f2(pack_u2(w0, w1), nd2)), d0, d1);
            } else {
              float p0, p1;
              unpack_f2(pp[kc / 2], p0, p1);
              d0 = p0 * (__uint_as_float(w0) - delta);
              d1 = p1 * (__uint_as_float(w1) - delta);
            }
            dsb[c / 2] = pack_bf16x2(d0, d1);
          }
          const int g8 = (cbase + c0) >> 3;
          const uint32_t off = (g8 >> 3) * 16384 + row * 128 + (((g8 & 7) ^ (row & 7)) << 4);
          st_shared_v4(sdS_i + off, dsb[0], dsb[1], dsb[2], dsb[3]);
        }
      }
      if (row == 0 && half == 0) AB_TRACE(1, 1, i, 2);
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive((i & 1) ? bar_p1 : bar_p0);
      if (row == 0 && half == 0) AB_TRACE(1, 1, i, 3);
    }
    // epilogue: accumulator row = key (jt*112 + row), rows >= 112 are padding; half 0 writes dK (x 1/8: dS is
    // stored unscaled), half 1 writes dV
    mbar_wait(bar_o, 0);
    tc_fence_after();
    const int u = jt * AB_KT + row;
    const bool kvalid = row < AB_KT && u < a.N;
    __nv_bfloat16* dst = a.dqkv + (static_cast<size_t>(b) * a.N + (kvalid ? u : 0)) * (3 * C) + C + head * 64 +
                         half * C;
    const uint32_t tacc = half == 0 ? tdK : tdV;
    const float osc = half == 0 ? 0.125f : 1.0f;
#pragma unroll
    for (int c0 = 0; c0 < 64; c0 += 16) {
      uint32_t o[16];
      tmem_ld_x16(tacc + lane_addr + c0, o);
      tmem_wait_ld();
      if (kvalid) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          uint4 uu;
          uu.x = pack_bf16x2(__uint_as_float(o[q * 8 + 0]) * osc, __uint_as_float(o[q * 8 + 1]) * osc);
          uu.y = pack_bf16x2(__uint_as_float(o[q * 8 + 2]) * osc, __uint_as_float(o[q * 8 + 3]) * osc);
          uu.z = pack_bf16x2(__uint_as_float(o[q * 8 + 4]) * osc, __uint_as_float(o[q * 8 + 5]) * osc);
          uu.w = pack_bf16x2(__uint_as_float(o[q * 8 + 6]) * osc, __uint_as_float(o[q * 8 + 7]) * osc);
          *reinterpret_cast<uint4*>(dst + c0 + q * 8) = uu;
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 9) tmem_dealloc(tmem, 512);
}

}  // namespace pk

using namespace pk;

static long long* g_attnb_trace = nullptr;
static int g_attnb_debug = 0;
extern "C" void pk_attn_bwd_debug(int flags) { g_attnb_debug = flags; }
// debug hook: device buffer of 2*2*16*8 int64 (clock64 timeline of CTA (0,0,0) of both backward kernels)
extern "C" void pk_attn_bwd_set_trace(void* buf) { g_attnb_trace = static_cast<long long*>(buf); }

// qkv / dqkv: bf16 [B*N, 3C];  O, dO: bf16 [B*N, C];  lse: fp32 [B*heads, N] from pk_attn_fwd
// scratch buffers (caller-allocated): delta [B*heads*N], relh_g [B*heads*Np*h], relw_g [B*heads*Np*w] fp32 with
// Np = N rounded up to a multiple of 128 (whole query tiles, row-innermost: see AttnBwdArgs)
// dt_ws: pk_attn_bwd_ws_floats(B, heads, h, w) fp32 (per-CTA partial table gradients)
// dTh [2h-1, 64], dTw [2w-1, 64]: fp32, ADDED to (caller zero-initialises or passes a running gradient)
extern "C" long long pk_attn_bwd_ws_floats(int B, int heads, int h, int w) {
  const long long ctas = static_cast<long long>((h * w + AB_BM - 1) / AB_BM) * heads * B;
  return ctas * (2 * h - 1 + 2 * w - 1) * 64;
}

// dT[r][c] += sum over CTA slices ws[cta][c][r] (table row innermost).  grid (64 columns, DT_STRIPES, row chunks), block
// (DT_RX, DT_RY): threadIdx.x walks the table rows (coalesced), the slices are strided over blockIdx.y / threadIdx.y
// with four loads in flight per thread, smem tree over threadIdx.y, one atomic per (row, column, stripe).
constexpr int DT_STRIPES = 4;
constexpr int DT_RX = 64, DT_RY = 16;
__global__ void __launch_bounds__(DT_RX * DT_RY)
attn_dt_reduce_kernel(const float* __restrict__ ws, int nctas, int rows, int rows_h, float* __restrict__ dTh,
                      float* __restrict__ dTw) {
  __shared__ float red[DT_RY][DT_RX];
  pdl_launch_dependents();
  pdl_wait();
  const int c = blockIdx.x;
  const size_t slice = static_cast<size_t>(rows) * 64;
  const int step = DT_STRIPES * DT_RY;
  {
    const int r = blockIdx.z * DT_RX + threadIdx.x;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    if (r < rows) {
      const float* p = ws + static_cast<size_t>(c) * rows + r;
      int i = blockIdx.y * DT_RY + threadIdx.y;
      for (; i + 3 * step < nctas; i += 4 * step) {
        s0 += p[static_cast<size_t>(i) * slice];
        s1 += p[static_cast<size_t>(i + step) * slice];
        s2 += p[static_cast<size_t>(i + 2 * step) * slice];
        s3 += p[static_cast<size_t>(i + 3 * step) * slice];
      }
      for (; i < nctas; i += step) s0 += p[static_cast<size_t>(i) * slice];
    }
    red[threadIdx.y][threadIdx.x] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (threadIdx.y == 0 && r < rows) {
      float s = 0.f;
#pragma unroll
      for (int y = 0; y < DT_RY; ++y) s += red[y][threadIdx.x];
      float* dst = r < rows_h ? dTh + static_cast<size_t>(r) * 64 + c : dTw + static_cast<size_t>(r - rows_h) * 64 + c;
      atomicAdd(dst, s);
    }
  }
}

// delta[b*heads + head][t] = sum_d O[b, t, head, d] * dO[b, t, head, d]: 8 lanes per (token, head) row of 64 bf16
// (one 16-byte load each from O and dO, fully coalesced), xor-shuffle tree, lane 0 of the group stores.
__global__ void __launch_bounds__(256)
attn_delta_kernel(const __nv_bfloat16* __restrict__ O, const __nv_bfloat16* __restrict__ dO,
                  float* __restrict__ delta, int B, int N, int heads) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  const size_t groups = static_cast<size_t>(B) * N * heads;
  const size_t g = idx >> 3;
  float acc = 0.f;
  if (g < groups) {
    const uint4 o = reinterpret_cast<const uint4*>(O)[idx], d = reinterpret_cast<const uint4*>(dO)[idx];
    const uint32_t ow[4] = {o.x, o.y, o.z, o.w}, dw[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      acc += __uint_as_float(ow[e] << 16) * __uint_as_float(dw[e] << 16);
      acc += __uint_as_float(ow[e] & 0xFFFF0000u) * __uint_as_float(dw[e] & 0xFFFF0000u);
    }
  }
  acc += __shfl_xor_sync(0xffffffffu, acc, 1);
  acc += __shfl_xor_sync(0xffffffffu, acc, 2);
  acc += __shfl_xor_sync(0xffffffffu, acc, 4);
  if (g < groups && (idx & 7) == 0) {
    const size_t tok = g / heads, head = g - tok * heads;
    const size_t b = tok / N, t = tok - b * N;
    delta[(b * heads + head) * N + t] = acc;
  }
}

static int attn_bwd_impl(const void* qkv, const void* O, const void* dO, const float* lse, const void* th,
                         const void* tw, void* dqkv, float* dTh, float* dTw, float* delta, float* relh_g,
                         float* relw_g, float* dt_ws, int B, int heads, int h, int w, int th_pad, int tw_pad,
                         int rel_ready, void* stream);

extern "C" int pk_attn_bwd(const void* qkv, const void* O, const void* dO, const float* lse, const void* th,
                           const void* tw, void* dqkv, float* dTh, float* dTw, float* delta, float* relh_g,
                           float* relw_g, float* dt_ws, int B, int heads, int h, int w, int th_pad, int tw_pad,
                           void* stream) {
  return attn_bwd_impl(qkv, O, dO, lse, th, tw, dqkv, dTh, dTw, delta, relh_g, relw_g, dt_ws, B, heads, h, w, th_pad,
                       tw_pad, 0, stream);
}
// relh_g / relw_g are INPUTS here: the bias rows stored by pk_attn_fwd_save on the same qkv / tables
extern "C" int pk_attn_bwd_saved(const void* qkv, const void* O, const void* dO, const float* lse, const void* th,
                                 const void* tw, void* dqkv, float* dTh, float* dTw, float* delta,
                                 const float* relh_g, const float* relw_g, float* dt_ws, int B, int heads, int h, int w,
                                 int th_pad, int tw_pad, void* stream) {
  return attn_bwd_impl(qkv, O, dO, lse, th, tw, dqkv, dTh, dTw, delta, const_cast<float*>(relh_g),
                       const_cast<float*>(relw_g), dt_ws, B, heads, h, w, th_pad, tw_pad, 1, stream);
}

static int attn_bwd_impl(const void* qkv, const void* O, const void* dO, const float* lse, const void* th,
                         const void* tw, void* dqkv, float* dTh, float* dTw, float* delta, float* relh_g,
                         float* relw_g, float* dt_ws, int B, int heads, int h, int w, int th_pad, int tw_pad,
                         int rel_ready, void* stream) {
  PK_CHECK(qkv && O && dO && lse && th && tw && dqkv && dTh && dTw && delta && relh_g && relw_g && dt_ws,
           "pk_attn_bwd: null pointer");
  PK_CHECK(th_pad % 16 == 0 && tw_pad % 16 == 0 && th_pad >= 2 * h - 1 && tw_pad >= 2 * w - 1 &&
               th_pad <= 224 && tw_pad <= 112,
           "pk_attn_bwd: bad table padding th_pad=%d tw_pad=%d (h=%d w=%d)", th_pad, tw_pad, h, w);
  // checked here, not only at the kernel switch below: the delta kernel is launched before it
  PK_CHECK(w == 2 || w == 4 || w == 7 || w == 8 || w == 14 || w == 28 || w == 56,
           "pk_attn_bwd: token-grid width %d unsupported (must divide 112)", w);
  const int N = h * w, C = heads * 64;
  AttnBwdArgs a;
  a.h = h; a.N = N; a.heads = heads; a.th_pad = th_pad; a.tw_pad = tw_pad;
  int relh_bytes = 128 * (h + 1) * 4;
  if (relh_bytes < 20480) relh_bytes = 20480;                        // 256 x 17 fp32 scratch rows (rel_w gather)
  if (relh_bytes < 128 * (w + 1) * 4) relh_bytes = 128 * (w + 1) * 4;  // Gw' exchange between the column halves
  relh_bytes = (relh_bytes + 15) & ~15;
  a.relh_bytes = relh_bytes;
  a.scale_log2 = 0.125f * AB_LOG2E;
  a.O = static_cast<const __nv_bfloat16*>(O);
  a.dO = static_cast<const __nv_bfloat16*>(dO);
  a.lse = lse; a.delta = delta; a.relh_g = relh_g; a.relw_g = relw_g;
  a.dqkv = static_cast<__nv_bfloat16*>(dqkv);
  a.dt_ws = dt_ws;
  a.rel_ready = rel_ready;
  a.trace = g_attnb_trace;
  a.debug = g_attnb_debug;

  CUtensorMap tmQ, tmKV, tmdO, tmTh, tmTw;
  {
    uint64_t dims[3] = {static_cast<uint64_t>(3 * C), static_cast<uint64_t>(N), static_cast<uint64_t>(B)};
    uint64_t strides[2] = {static_cast<uint64_t>(3 * C) * 2, static_cast<uint64_t>(N) * 3 * C * 2};
    uint32_t boxq[3] = {64, AB_BM, 1};
    uint32_t boxk[3] = {64, AB_KT, 1};
    if (!make_tmap_bf16(&tmQ, qkv, 3, dims, strides, boxq)) return 3;
    if (!make_tmap_bf16(&tmKV, qkv, 3, dims, strides, boxk)) return 3;
    uint64_t dimo[3] = {static_cast<uint64_t>(C), static_cast<uint64_t>(N), static_cast<uint64_t>(B)};
    uint64_t strideo[2] = {static_cast<uint64_t>(C) * 2, static_cast<uint64_t>(N) * C * 2};
    if (!make_tmap_bf16(&tmdO, dO, 3, dimo, strideo, boxq)) return 3;
    uint64_t d2[2] = {64, static_cast<uint64_t>(th_pad)};
    uint64_t s2[1] = {128};
    uint32_t b2[2] = {64, static_cast<uint32_t>(th_pad)};
    if (!make_tmap_bf16(&tmTh, th, 2, d2, s2, b2)) return 3;
    d2[1] = tw_pad;
    b2[1] = tw_pad;
    if (!make_tmap_bf16(&tmTw, tw, 2, d2, s2, b2)) return 3;
  }
  a.kv_stages = (1024 + A_SKV + 3 * 28672 + static_cast<size_t>(relh_bytes) + 192 <= 227 * 1024) ? 3 : 2;
  const size_t smemA = 1024 + A_SKV + static_cast<size_t>(a.kv_stages) * 28672 + relh_bytes + 192;
  const size_t smemB = 1024 + B_BARS + 192;
  PK_CHECK(smemA <= 227 * 1024, "pk_attn_bwd: h=%d needs %zu B of shared memory", h, smemA);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  {
    const size_t threads = static_cast<size_t>(B) * N * heads * 8;
    launch_pdl(attn_delta_kernel, dim3(static_cast<unsigned>((threads + 255) / 256)), dim3(256), 0, st,
               static_cast<const __nv_bfloat16*>(O), static_cast<const __nv_bfloat16*>(dO), delta, B, N, heads);
    PK_LAUNCH_CHECK("pk_attn_bwd(delta)");
  }
  dim3 gridA((N + AB_BM - 1) / AB_BM, heads, B);
  const int R = AB_KT / w;
  dim3 gridB((h + R - 1) / R, heads, B);
#define PK_ATTB_LAUNCH(WW)                                                                                     \
  case WW: {                                                                                                   \
    static bool attr = false;                                                                                  \
    if (!attr) {                                                                                               \
      cudaFuncSetAttribute(attn_bwd_dq_kernel<WW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);   \
      cudaFuncSetAttribute(attn_bwd_dkv_kernel<WW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);  \
      attr = true;                                                                                             \
    }                                                                                                          \
    if (!(a.debug & 4))                                                                                        \
      launch_pdl(attn_bwd_dq_kernel<WW>, gridA, dim3(AB_THREADS), smemA, st, tmQ, tmKV, tmdO, tmTh, tmTw, a);   \
    PK_LAUNCH_CHECK("pk_attn_bwd(dq)");                                                                        \
    if (!(a.debug & 8)) launch_pdl(attn_bwd_dkv_kernel<WW>, gridB, dim3(AB_THREADS), smemB, st, tmQ, tmKV, tmdO, a); \
    PK_LAUNCH_CHECK("pk_attn_bwd(dkv)");                                                                       \
  } break;
  switch (w) {
    PK_ATTB_LAUNCH(2)
    PK_ATTB_LAUNCH(4)
    PK_ATTB_LAUNCH(7)
    PK_ATTB_LAUNCH(8)
    PK_ATTB_LAUNCH(14)
    PK_ATTB_LAUNCH(28)
    PK_ATTB_LAUNCH(56)
    default:
      PK_CHECK(false, "pk_attn_bwd: token-grid width %d unsupported (must divide 112)", w);
  }
#undef PK_ATTB_LAUNCH
  {
    const int rows = 2 * h - 1 + 2 * w - 1;
    const int nctas = static_cast<int>(gridA.x * gridA.y * gridA.z);
    launch_pdl(attn_dt_reduce_kernel, dim3(64, DT_STRIPES, (rows + DT_RX - 1) / DT_RX), dim3(DT_RX, DT_RY), 0, st, static_cast<const float*>(dt_ws),
               nctas, rows, 2 * h - 1, dTh, dTw);
    PK_LAUNCH_CHECK("pk_attn_bwd(dT reduce)");
  }
  return 0;
}
