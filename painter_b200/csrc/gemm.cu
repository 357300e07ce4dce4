// painter_b200 — persistent, warp-specialised tcgen05 GEMM for sm_100a.
//
//   C[M,N] = A[M,K] . B[N,K]^T      bf16 operands, fp32 accumulation in TMEM
//
// One CTA per SM, 256 threads:
//   warps 0..3  epilogue       (tcgen05.ld 32x32b -> registers -> smem staging -> coalesced fused epilogue)
//   warp 4      TMA producer   (cp.async.bulk.tensor -> 128B-swizzled smem ring, mbarrier tx)
//   warp 5      MMA issuer     (one elected lane: tcgen05.mma 128 x BN x 16, commit -> mbarriers)
//   warp 6      TMEM allocator (2 accumulator stages of BN fp32 columns)
// (producer / MMA warps have the highest ids on purpose: the issue arbiter prefers higher warp ids, and a busy
//  epilogue warp must never delay the MMA issue)
// The accumulator is double-buffered in TMEM so the epilogue of tile i overlaps the MMAs of tile
// i+1.  Operands may be K-major (row-major [rows,K]) or MN-major (row-major [K,rows]); the latter is
// what the backward GEMMs (dgrad: B = W[out,in]; wgrad: A = dY[tokens,out], B = X[tokens,in]) need, so no
// transposed copies of weights or activations are ever materialised.
//
// Reference call sites replaced: every nn.Linear on the path (models_painter.py:60-61,76,87; timm Mlp
// fc1/fc2 via :201; decoder_embed :327,423) and autograd's mm backward for them.
#include "gemm_common.cuh"

namespace pk {


template <int KIND>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const GemmArgs g) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_base = smem_u32(smem_raw);
  const uint32_t base = (raw_base + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (base - raw_base);

  const int BN = g.BN;
  const int stages = g.stages;
  const uint32_t B_BYTES = static_cast<uint32_t>(BN) * 128u;
  const uint32_t sA = base;
  const uint32_t sB = base + stages * GEMM_A_BYTES;
  const uint32_t bar_base = sB + stages * B_BYTES;
  // barrier layout: full[stages], empty[stages], tfull[2], tempty[2], holder
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (stages + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * stages + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * stages + 2 + s); };
  const uint32_t holder = bar_base + 8u * (2 * stages + 4);
  volatile uint32_t* holder_gen =
      reinterpret_cast<volatile uint32_t*>(smem_gen + (holder - base));
  float* stg_gen = reinterpret_cast<float*>(smem_gen + (bar_base - base) + 256);  // 4 x [32][STG_LD] fp32

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_kb = (g.K + GEMM_BK - 1) / GEMM_BK;
  const int tiles_mn = g.num_m_tiles * g.num_n_tiles;
  const int total_tiles = tiles_mn * g.splits;
  const uint32_t tmem_cols = 2u * BN;

  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 9 && lane == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), GEMM_EPI_WARPS);
    }
    fence_barrier_init();
  }
  if (warp == 10) tmem_alloc(holder, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *holder_gen;

  if (warp == 8) {
    if (lane == 0) {
      // ------------------------------ TMA producer ------------------------------
      uint32_t s = 0, ph = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int mn = tile % tiles_mn, split = tile / tiles_mn;
        const int m_blk = mn % g.num_m_tiles, n_blk = mn / g.num_m_tiles;
        const int kb0 = split * g.kb_per_split;
        const int kb1 = min(num_kb, kb0 + g.kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(empty_bar(s), ph ^ 1u);
          mbar_expect_tx(full_bar(s), GEMM_A_BYTES + B_BYTES);
          const uint32_t a_dst = sA + s * GEMM_A_BYTES;
          const uint32_t b_dst = sB + s * B_BYTES;
          if (g.conv.mode == 1) {
            const int tx = m_blk % g.conv.tiles_x, r1 = m_blk / g.conv.tiles_x;
            const int ty = r1 % g.conv.tiles_y, bi = r1 / g.conv.tiles_y;
            const int dy = kb / 3, dx = kb - dy * 3;
            tma_load_4d(a_dst, &tmA, full_bar(s), 0, tx * g.conv.TW + dx - 1, ty * g.conv.TH + dy - 1, bi);
            tma_load_2d(b_dst, &tmB, full_bar(s), kb * GEMM_BK, n_blk * BN);
          } else if (g.conv.mode == 2) {
            const int tx = kb % g.conv.tiles_x, r1 = kb / g.conv.tiles_x;
            const int ty = r1 % g.conv.tiles_y, bi = r1 / g.conv.tiles_y;
#pragma unroll
            for (int gi = 0; gi < 2; ++gi) {
              const int tap = m_blk * 2 + gi;
              const int dy = tap / 3, dx = tap - dy * 3;
              // tap 9 does not exist: a far out-of-bounds box yields the zero rows of the last m-block
              const int yy = tap < 9 ? ty * g.conv.TH + dy - 1 : -(1 << 20);
              tma_load_4d(a_dst + gi * 8192, &tmA, full_bar(s), 0, tx * g.conv.TW + dx - 1, yy, bi);
            }
            tma_load_4d(b_dst, &tmB, full_bar(s), 0, tx * g.conv.TW, ty * g.conv.TH, bi);
          } else {
            if (!g.transA) {
              tma_load_2d(a_dst, &tmA, full_bar(s), kb * GEMM_BK, m_blk * GEMM_BM);
            } else {
              tma_load_2d(a_dst, &tmA, full_bar(s), m_blk * GEMM_BM, kb * GEMM_BK);
              tma_load_2d(a_dst + 8192, &tmA, full_bar(s), m_blk * GEMM_BM + 64, kb * GEMM_BK);
            }
            if (!g.transB) {
              tma_load_2d(b_dst, &tmB, full_bar(s), kb * GEMM_BK, n_blk * BN);
            } else {
              for (int gi = 0; gi < BN / 64; ++gi)
                tma_load_2d(b_dst + gi * 8192, &tmB, full_bar(s), n_blk * BN + gi * 64, kb * GEMM_BK);
            }
          }
          if (++s == static_cast<uint32_t>(stages)) {
            s = 0;
            ph ^= 1u;
          }
        }
      }
    }
  } else if (warp == 9) {
    {
      // ------------------------------- MMA issuer -------------------------------
      // warp-uniform control flow (descriptors stay in uniform registers); one elected lane issues tcgen05
      const uint32_t idesc = make_idesc_bf16(GEMM_BM, BN, g.transA != 0, g.transB != 0);
      uint32_t s = 0, ph = 0, it = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        const uint32_t as = it & 1u, aph = (it >> 1) & 1u;
        mbar_wait(tempty_bar(as), aph ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        const int split = tile / tiles_mn;
        const int kb0 = split * g.kb_per_split;
        const int kb1 = min(num_kb, kb0 + g.kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar(s), ph);
          tc_fence_after();
          const uint32_t a_addr = sA + s * GEMM_A_BYTES;
          const uint32_t b_addr = sB + s * B_BYTES;
          const uint64_t a0 = g.transA ? make_sdesc(a_addr, 8192, 1024) : make_sdesc(a_addr, 16, 1024);
          const uint64_t b0 = g.transB ? make_sdesc(b_addr, 8192, 1024) : make_sdesc(b_addr, 16, 1024);
          const uint32_t a_step = g.transA ? 2048u : 32u, b_step = g.transB ? 2048u : 32u;
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < GEMM_BK / 16; ++k)
              umma_ss(d_tmem, sdesc_add(a0, k * a_step), sdesc_add(b0, k * b_step), idesc,
                      (kb != kb0 || k != 0) ? 1u : 0u);
            umma_commit(empty_bar(s));
          }
          __syncwarp();
          if (++s == static_cast<uint32_t>(stages)) {
            s = 0;
            ph ^= 1u;
          }
        }
        if (elect_one()) umma_commit(tfull_bar(as));
        __syncwarp();
      }
    }
  } else if (warp < GEMM_EPI_WARPS) {
    // --------------------------------- epilogue ---------------------------------
    const int ew = warp & 3;   // TMEM lane quarter
    const int eg = warp >> 2;  // column group: this warp owns the 64-column blocks with (c0 / 64) % 2 == eg
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const int mn = tile % tiles_mn;
      const int m_blk = mn % g.num_m_tiles, n_blk = mn / g.num_m_tiles;
      const uint32_t as = it & 1u, aph = (it >> 1) & 1u;
      mbar_wait(tfull_bar(as), aph);
      tc_fence_after();
      const int rloc = ew * 32 + lane;
      const int row = m_blk * GEMM_BM + rloc;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + as * BN;
      if constexpr (KIND == EPI_HEAD || KIND == EPI_UNSHUF) {
        // pixel-row tile (64 columns: handled by column group 0; group 1 only signals): rloc -> (b, y, x)
        if (eg == 0) {
        const int tx = m_blk % g.conv.tiles_x, r1 = m_blk / g.conv.tiles_x;
        const int ty = r1 % g.conv.tiles_y, bi = r1 / g.conv.tiles_y;
        const int y = ty * g.conv.TH + rloc / g.conv.TW, x = tx * g.conv.TW + rloc % g.conv.TW;
        if constexpr (KIND == EPI_HEAD) {
          float c[64];
#pragma unroll
          for (int c0 = 0; c0 < 64; c0 += 32) {
            uint32_t v[32];
            tmem_ld_x32(taddr + c0, v);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 32; ++j) c[c0 + j] = __uint_as_float(v[j]);
          }
          head_epilogue_row(g, bi, y, x, c);
        } else {  // EPI_UNSHUF: token row m = (b, y/p, x/p), columns ((y%p)*p + x%p)*64 + c
          const int p = g.epi.ps_p;
          const size_t mtok = (static_cast<size_t>(bi) * (g.conv.H / p) + y / p) * (g.conv.W / p) + x / p;
          __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(g.epi.out) + mtok * g.epi.ldc +
                               ((y % p) * p + x % p) * 64 + n_blk * BN;
          for (int c0 = 0; c0 < BN; c0 += 32) {
            uint32_t v[32];
            tmem_ld_x32(taddr + c0, v);
            tmem_wait_ld();
            float xv[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) xv[j] = __uint_as_float(v[j]);
            store_bf16x32(dst + c0, xv);
          }
        }
        }
      } else {
        float* stg = stg_gen + warp * (32 * STG_LD);
        const int row0 = m_blk * GEMM_BM + ew * 32;
        EpiAux auxA, auxB;   // explicit ping-pong (BN is a multiple of 64): keeps both in registers
        if (eg * 64 < BN) gemm_epilogue_prefetch<KIND>(g.epi, row0, g.M, n_blk * BN + eg * 64, auxA);
        for (int c0 = eg * 64; c0 < BN; c0 += 128) {
          uint32_t v[32];
          tmem_ld_x32(taddr + c0, v);
          gemm_epilogue_prefetch<KIND>(g.epi, row0, g.M, n_blk * BN + c0 + 32, auxB);
          tmem_wait_ld();
          gemm_epilogue_chunk<KIND>(g.epi, stg, row0, g.M, n_blk * BN + c0, v, auxA);
          tmem_ld_x32(taddr + c0 + 32, v);
          if (c0 + 128 < BN) gemm_epilogue_prefetch<KIND>(g.epi, row0, g.M, n_blk * BN + c0 + 128, auxA);
          tmem_wait_ld();
          gemm_epilogue_chunk<KIND>(g.epi, stg, row0, g.M, n_blk * BN + c0 + 32, v, auxB);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(as));
    }
  }

  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 10) tmem_dealloc(tmem_base, tmem_cols);
}

int g_force_bn = 0;
int g_force_splits = 0;
int g_use_2cta = 1;  // 1 = CTA pairs (gemm2.cu) whenever the shape allows (default), 0 = 1-CTA kernel only

int launch_gemm2(const void* A, const void* B, int lda, int ldb, GemmArgs& g, cudaStream_t st);

static int launch_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, GemmArgs& g, cudaStream_t st,
                       const char* who) {
  const size_t smem = 1024 + static_cast<size_t>(g.stages) * (GEMM_A_BYTES + g.BN * 128) + 256 +
                      GEMM_EPI_WARPS * 32 * STG_LD * sizeof(float);
  const int total = g.num_m_tiles * g.num_n_tiles * g.splits;
  const int sms = sm_count();
  const int grid = total < sms ? total : sms;
#define PK_GEMM_CASE(KK)                                                                                       \
  case KK: {                                                                                                   \
    static bool attr_set = false;                                                                              \
    if (!attr_set) {                                                                                           \
      cudaError_t e = cudaFuncSetAttribute(gemm_bf16_kernel<KK>, cudaFuncAttributeMaxDynamicSharedMemorySize,  \
                                           227 * 1024);                                                        \
      PK_CHECK(e == cudaSuccess, "%s: cudaFuncSetAttribute: %s", who, cudaGetErrorString(e));                  \
      attr_set = true;                                                                                         \
    }                                                                                                          \
    gemm_bf16_kernel<KK><<<grid, GEMM_THREADS, smem, st>>>(tmA, tmB, g);                                       \
  } break;
  switch (g.epi.kind) {
    PK_GEMM_CASE(PK_EPI_BF16)
    PK_GEMM_CASE(PK_EPI_F32)
    PK_GEMM_CASE(PK_EPI_GELU)
    PK_GEMM_CASE(PK_EPI_RESID)
    PK_GEMM_CASE(PK_EPI_DGELU)
    PK_GEMM_CASE(PK_EPI_PIXSHUF)
    PK_GEMM_CASE(EPI_HEAD)
    PK_GEMM_CASE(EPI_UNSHUF)
    default:
      PK_CHECK(false, "%s: bad epilogue kind %d", who, g.epi.kind);
  }
#undef PK_GEMM_CASE
  PK_LAUNCH_CHECK(who);
  return 0;
}

}  // namespace pk

// test hooks: force the N tile (64/128/256) / the split-K factor; 0 restores the heuristics
extern "C" void pk_gemm_force_bn(int bn) { pk::g_force_bn = bn; }
extern "C" void pk_gemm_force_splits(int s) { pk::g_force_splits = s; }
extern "C" void pk_gemm_use_2cta(int on) { pk::g_use_2cta = on; }

// Tiling / scheduling decisions of one pk_gemm_bf16 call (host only; also reachable through pk_gemm_plan for the
// CPU-side schedule tests).  Returns the kernel arguments and which kernel (CTA pair or single CTA) runs them.
static void plan_gemm(int M, int N, int K, int transA, int transB, const PkEpilogue* epi, pk::GemmArgs& gout,
                      bool& two_cta) {
  using namespace pk;
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.M = M;
  g.N = N;
  g.K = K;
  g.transA = transA ? 1 : 0;
  g.transB = transB ? 1 : 0;
  g.epi = *epi;
  if (g.epi.alpha == 0.0f) g.epi.alpha = 1.0f;
  const int sms = sm_count();
  const int mt = (M + GEMM_BM - 1) / GEMM_BM;
  int BN = 64;
  const bool can_split = epi->kind == PK_EPI_F32 && epi->accumulate == 2;
  if (can_split) {
    // weight-gradient GEMMs (K = tokens): take the widest tile and fill the machine with split-K instead of
    // shrinking the tile
    BN = N % 256 == 0 ? 256 : (N % 128 == 0 ? 128 : 64);
  } else {
    if (N % 256 == 0 && static_cast<long long>(mt) * (N / 256) >= sms) BN = 256;
    else if (N % 128 == 0 && static_cast<long long>(mt) * (N / 128) >= sms / 2) BN = 128;
  }
  if (g_force_bn > 0 && N % g_force_bn == 0) BN = g_force_bn;
  g.BN = BN;
  g.stages = gemm_stages_for(GEMM_A_BYTES + BN * 128);
  g.num_m_tiles = mt;
  g.num_n_tiles = N / BN;
  // split-K: only for plain fp32 outputs whose tile count cannot fill the machine (wgrad GEMMs);
  // accumulate == 2 means "out is zero-initialised, add atomically".
  const int num_kb = (K + GEMM_BK - 1) / GEMM_BK;
  g.splits = 1;
  if (epi->kind == PK_EPI_F32 && epi->accumulate == 2) {
    int want = sms / (g.num_m_tiles * g.num_n_tiles);
    if (want > 1) {
      if (want > num_kb / 8) want = num_kb / 8 > 0 ? num_kb / 8 : 1;
      g.splits = want;
    }
    if (g_force_splits > 0) g.splits = g_force_splits < num_kb ? g_force_splits : num_kb;
  }
  g.kb_per_split = (num_kb + g.splits - 1) / g.splits;
  g.splits = (num_kb + g.kb_per_split - 1) / g.kb_per_split;
  if (g.splits == 1 && g.epi.kind == PK_EPI_F32 && g.epi.accumulate == 2) g.epi.accumulate = 1;

  // CTA-pair kernel (256 x BN tiles): needs a pair-tile count that can feed 74 clusters
  two_cta = g_use_2cta && (BN == 256 || BN == 128) && M >= 256;
  if (two_cta) {
    GemmArgs g2 = g;
    g2.num_m_tiles = (M + 255) / 256;
    g2.stages = gemm_stages_for(GEMM_A_BYTES + (BN / 2) * 128);
    if (g2.epi.kind == PK_EPI_F32 && epi->accumulate == 2) {
      // zero-initialised fp32 output (weight gradients): stream-K.  The tiles_mn * num_kb k-block units are cut
      // into one equal range per cluster; a tile that straddles ranges is finished with fp32 atomics.
      g2.epi.accumulate = 2;
      g2.splits = 1;
      g2.kb_per_split = num_kb;
      const int clusters = sms / 2;
      const int tiles2 = g2.num_m_tiles * g2.num_n_tiles;
      const long long units = static_cast<long long>(tiles2) * num_kb;
      if (g_force_splits > 0) {
        const int want = g_force_splits < num_kb ? g_force_splits : num_kb;
        g2.kb_per_split = (num_kb + want - 1) / want;
        g2.splits = (num_kb + g2.kb_per_split - 1) / g2.kb_per_split;
        if (g2.splits == 1) g2.epi.accumulate = 1;
      } else if (tiles2 % clusters == 0 || units < 4ll * clusters) {
        g2.epi.accumulate = 1;   // already balanced (or too small to matter): plain data-parallel tiles
      } else {
        int per = static_cast<int>((units + clusters - 1) / clusters);
        if (per < 4) per = 4;
        g2.streamk_units = per;
      }
    }
    // rasterisation: keep B L2-resident when it fits, otherwise sweep the columns inside groups of 8 row blocks
    // (stream-K calls with a large B keep the row-fastest order: measured 1006 vs 918 TF/s on the decoder wgrad)
    g2.group_m = (static_cast<long long>(N) * K * 2 <= (40ll << 20)) ? 1 : (g2.streamk_units > 0 ? 0 : 8);
    gout = g2;
    return;
  }
  gout = g;
}

// Host-side views of the scheduler (no device work): the plan of a call, and the (row block, column block, k-block
// range) items one cluster / CTA walks - the same GemmSched / gemm_tile_coords code the kernels run.
extern "C" int pk_gemm_plan(int M, int N, int K, int kind, int accumulate, int* out9) {
  using namespace pk;
  PK_CHECK(out9 && M > 0 && N > 0 && K > 0 && N % 64 == 0, "pk_gemm_plan: bad arguments");
  PkEpilogue e;
  memset(&e, 0, sizeof(e));
  e.kind = kind;
  e.accumulate = accumulate;
  GemmArgs g;
  bool two = false;
  plan_gemm(M, N, K, 0, 0, &e, g, two);
  const int num_kb = (K + GEMM_BK - 1) / GEMM_BK;
  const int tiles = g.num_m_tiles * g.num_n_tiles;
  int workers;
  if (two) {
    workers = sm_count() / 2;
    if (g.streamk_units > 0) workers = (tiles * num_kb + g.streamk_units - 1) / g.streamk_units;
    else if (workers > tiles * g.splits) workers = tiles * g.splits;
  } else {
    workers = sm_count() < tiles * g.splits ? sm_count() : tiles * g.splits;
  }
  const int vals[9] = {two ? 1 : 0, g.BN, g.num_m_tiles, g.num_n_tiles, g.splits, g.kb_per_split, g.streamk_units,
                       g.group_m, workers};
  for (int i = 0; i < 9; ++i) out9[i] = vals[i];
  return 0;
}

extern "C" int pk_gemm_plan_walk(int M, int N, int K, int kind, int accumulate, int worker, int* out4, int max_items) {
  using namespace pk;
  PK_CHECK(out4 && max_items > 0, "pk_gemm_plan_walk: bad arguments");
  int plan[9];
  if (pk_gemm_plan(M, N, K, kind, accumulate, plan)) return 2;
  PkEpilogue e;
  memset(&e, 0, sizeof(e));
  e.kind = kind;
  e.accumulate = accumulate;
  GemmArgs g;
  bool two = false;
  plan_gemm(M, N, K, 0, 0, &e, g, two);
  const int num_kb = (K + GEMM_BK - 1) / GEMM_BK;
  const int tiles = g.num_m_tiles * g.num_n_tiles;
  int n = 0;
  if (two) {
    GemmSched sch;
    sch.init(g, tiles, num_kb, worker, plan[8]);
    int mn, kb0, kb1;
    while (sch.next(mn, kb0, kb1) && n < max_items) {
      int mb, nb;
      gemm_tile_coords(g, mn, mb, nb);
      out4[4 * n] = mb; out4[4 * n + 1] = nb; out4[4 * n + 2] = kb0; out4[4 * n + 3] = kb1;
      ++n;
    }
  } else {
    for (int tile = worker; tile < tiles * g.splits && n < max_items; tile += plan[8]) {
      const int mn = tile % tiles, split = tile / tiles;
      const int kb0 = split * g.kb_per_split;
      const int kb1 = num_kb < kb0 + g.kb_per_split ? num_kb : kb0 + g.kb_per_split;
      out4[4 * n] = mn % g.num_m_tiles; out4[4 * n + 1] = mn / g.num_m_tiles; out4[4 * n + 2] = kb0; out4[4 * n + 3] = kb1;
      ++n;
    }
  }
  return -n;   // number of items, negated (0 and positive values are the usual status codes)
}

extern "C" int pk_gemm_bf16(const void* A, const void* B, int M, int N, int K, int lda, int ldb,
                            int transA, int transB, const PkEpilogue* epi, void* stream) {
  using namespace pk;
  PK_CHECK(A && B && epi && epi->out, "pk_gemm_bf16: null pointer");
  PK_CHECK(M > 0 && N > 0 && K > 0, "pk_gemm_bf16: bad shape M=%d N=%d K=%d", M, N, K);
  PK_CHECK(N % 64 == 0, "pk_gemm_bf16: N=%d must be a multiple of 64", N);
  PK_CHECK(lda % 8 == 0 && ldb % 8 == 0, "pk_gemm_bf16: lda/ldb must be multiples of 8 (16 B)");
  PK_CHECK((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(B) & 15) == 0,
           "pk_gemm_bf16: operands must be 16-byte aligned");
  PK_CHECK(epi->kind >= PK_EPI_BF16 && epi->kind <= PK_EPI_PIXSHUF, "pk_gemm_bf16: bad epilogue %d",
           epi->kind);
  if (epi->kind != PK_EPI_PIXSHUF)
    PK_CHECK(epi->ldc % 8 == 0 && epi->ldc >= N, "pk_gemm_bf16: bad ldc %d", epi->ldc);
  if (epi->kind == PK_EPI_RESID || epi->kind == PK_EPI_DGELU)
    PK_CHECK(epi->aux && epi->ld_aux % 8 == 0, "pk_gemm_bf16: epilogue %d needs aux", epi->kind);
  if (epi->kind == PK_EPI_GELU) PK_CHECK(epi->out2, "pk_gemm_bf16: GELU epilogue needs out2");
  if (epi->kind == PK_EPI_RESID && epi->rowscale)
    PK_CHECK(epi->rows_per_group > 0, "pk_gemm_bf16: rows_per_group must be > 0");
  if (epi->kind == PK_EPI_PIXSHUF)
    PK_CHECK(epi->ps_c % 32 == 0 && epi->ps_h * epi->ps_w > 0 && M % (epi->ps_h * epi->ps_w) == 0 &&
                 N == epi->ps_p * epi->ps_p * epi->ps_c,
             "pk_gemm_bf16: bad pixel-shuffle geometry");

  GemmArgs g;
  bool two_cta = false;
  plan_gemm(M, N, K, transA, transB, epi, g, two_cta);
  if (two_cta) return launch_gemm2(A, B, lda, ldb, g, static_cast<cudaStream_t>(stream));

  CUtensorMap tmA, tmB;
  {
    uint64_t dims[2], strides[1];
    uint32_t box[2];
    if (!g.transA) {
      dims[0] = K; dims[1] = M; box[0] = 64; box[1] = 128;
    } else {
      dims[0] = M; dims[1] = K; box[0] = 64; box[1] = 64;
    }
    strides[0] = static_cast<uint64_t>(lda) * 2;
    if (!make_tmap_bf16(&tmA, A, 2, dims, strides, box)) return 3;
    if (!g.transB) {
      dims[0] = K; dims[1] = N; box[0] = 64; box[1] = static_cast<uint32_t>(g.BN);
    } else {
      dims[0] = N; dims[1] = K; box[0] = 64; box[1] = 64;
    }
    strides[0] = static_cast<uint64_t>(ldb) * 2;
    if (!make_tmap_bf16(&tmB, B, 2, dims, strides, box)) return 3;
  }
  return launch_gemm(tmA, tmB, g, static_cast<cudaStream_t>(stream), "pk_gemm_bf16");
}

// ------------------------------------------------------------------------------------------------
// Decoder 3x3 convolution (64 -> 64, pad 1) as implicit GEMM over NHWC bf16 (models_painter.py:328-333)
// ------------------------------------------------------------------------------------------------
static int conv_common(const void* img_nhwc, const void* wmat, int B, int H, int W, pk::GemmArgs& g,
                       void* stream, const char* who) {
  using namespace pk;
  int TW, TH;
  PK_CHECK(conv_tile_geometry(H, W, 128, &TW, &TH), "%s: unsupported image size %dx%d", who, H, W);
  g.M = B * H * W;
  g.N = 64;
  g.K = 576;
  g.BN = 64;
  g.stages = gemm_stages_for(GEMM_A_BYTES + 64 * 128);
  g.transA = g.transB = 0;
  g.splits = 1;
  g.kb_per_split = 9;
  g.conv.mode = 1;
  g.conv.H = H; g.conv.W = W; g.conv.TW = TW; g.conv.TH = TH;
  g.conv.tiles_x = W / TW; g.conv.tiles_y = H / TH;
  g.num_m_tiles = B * g.conv.tiles_x * g.conv.tiles_y;
  g.num_n_tiles = 1;
  CUtensorMap tmA, tmB;
  uint64_t dims[4] = {64, static_cast<uint64_t>(W), static_cast<uint64_t>(H), static_cast<uint64_t>(B)};
  uint64_t strides[3] = {128, static_cast<uint64_t>(W) * 128, static_cast<uint64_t>(H) * W * 128};
  uint32_t box[4] = {64, static_cast<uint32_t>(TW), static_cast<uint32_t>(TH), 1};
  if (!make_tmap_bf16(&tmA, img_nhwc, 4, dims, strides, box)) return 3;
  uint64_t d2[2] = {576, 64};
  uint64_t s2[1] = {576 * 2};
  uint32_t b2[2] = {64, 64};
  if (!make_tmap_bf16(&tmB, wmat, 2, d2, s2, b2)) return 3;
  return launch_gemm(tmA, tmB, g, static_cast<cudaStream_t>(stream), who);
}

extern "C" int pk_decoder_head_fwd(const void* g_nhwc, const void* wmat, const float* head_params,
                                   const float* tgts, const uint8_t* mask, int maskB, const float* valid,
                                   void* c1_out, float* patch_out, float* num, int B, int H, int W, int p,
                                   int loss_kind, void* stream) {
  using namespace pk;
  PK_CHECK(g_nhwc && wmat && head_params && tgts && mask && valid && c1_out && patch_out && num,
           "pk_decoder_head_fwd: null pointer");
  PK_CHECK(H % p == 0 && W % p == 0 && maskB >= 1, "pk_decoder_head_fwd: bad geometry");
  // the head parameters ride in constant memory (operands of the epilogue's FFMAs): every call takes the next of
  // HEAD_SLOTS copies, uploaded on the call's stream just ahead of its kernel
  static std::atomic<unsigned> next_slot{0};
  const int slot = static_cast<int>(next_slot.fetch_add(1, std::memory_order_relaxed) % HEAD_SLOTS);
  cudaError_t e = cudaMemcpyToSymbolAsync(c_head_all, head_params, 387 * sizeof(float), slot * 392 * sizeof(float),
                                          cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream));
  PK_CHECK(e == cudaSuccess, "pk_decoder_head_fwd: constant upload: %s", cudaGetErrorString(e));
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.head.slot = slot;
  g.epi.kind = EPI_HEAD;
  g.epi.alpha = 1.0f;
  g.head.tgts = tgts; g.head.mask = mask; g.head.valid = valid; g.head.maskB = maskB;
  g.head.c1_out = static_cast<__nv_bfloat16*>(c1_out);
  g.head.patch_out = patch_out; g.head.num = num; g.head.p = p; g.head.loss_kind = loss_kind;
  return conv_common(g_nhwc, wmat, B, H, W, g, stream, "pk_decoder_head_fwd");
}

// dG (inverse pixel shuffle) [B*h*w, p*p*64] = conv3x3^T(dC1); wmat_t = dgrad weight matrix (flipped taps)
extern "C" int pk_conv3x3_dgrad_unshuffle(const void* dc1_nhwc, const void* wmat_t, void* out_tok, int B, int H,
                                          int W, int p, void* stream) {
  using namespace pk;
  PK_CHECK(dc1_nhwc && wmat_t && out_tok && H % p == 0 && W % p == 0, "pk_conv3x3_dgrad_unshuffle: bad args");
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.epi.kind = EPI_UNSHUF;
  g.epi.alpha = 1.0f;
  g.epi.out = out_tok;
  g.epi.ldc = p * p * 64;
  g.epi.ps_p = p;
  return conv_common(dc1_nhwc, wmat_t, B, H, W, g, stream, "pk_conv3x3_dgrad_unshuffle");
}

// wgrad: out[(tap*64 + c), o] += sum_pix G[pix + tap, c] * dC1[pix, o]   (out fp32 [576(+pad to 640), 64], zeroed)
extern "C" int pk_conv3x3_wgrad(const void* g_nhwc, const void* dc1_nhwc, float* out, int B, int H, int W,
                                void* stream) {
  using namespace pk;
  PK_CHECK(g_nhwc && dc1_nhwc && out, "pk_conv3x3_wgrad: null pointer");
  int TW, TH;
  PK_CHECK(conv_tile_geometry(H, W, 64, &TW, &TH), "pk_conv3x3_wgrad: unsupported image size %dx%d", H, W);
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.M = 576; g.N = 64; g.K = B * H * W;
  g.BN = 64; g.stages = gemm_stages_for(GEMM_A_BYTES + 64 * 128);
  g.transA = g.transB = 1;
  g.conv.mode = 2;
  g.conv.H = H; g.conv.W = W; g.conv.TW = TW; g.conv.TH = TH;
  g.conv.tiles_x = W / TW; g.conv.tiles_y = H / TH;
  g.num_m_tiles = 5; g.num_n_tiles = 1;
  const int num_kb = B * g.conv.tiles_x * g.conv.tiles_y;
  int splits = sm_count() / 5;
  if (splits > num_kb) splits = num_kb;
  if (splits < 1) splits = 1;
  g.kb_per_split = (num_kb + splits - 1) / splits;
  g.splits = (num_kb + g.kb_per_split - 1) / g.kb_per_split;
  g.epi.kind = PK_EPI_F32;
  g.epi.out = out;
  g.epi.ldc = 64;
  g.epi.alpha = 1.0f;
  g.epi.accumulate = 2;
  CUtensorMap tmA, tmB;
  uint64_t dims[4] = {64, static_cast<uint64_t>(W), static_cast<uint64_t>(H), static_cast<uint64_t>(B)};
  uint64_t strides[3] = {128, static_cast<uint64_t>(W) * 128, static_cast<uint64_t>(H) * W * 128};
  uint32_t box[4] = {64, static_cast<uint32_t>(TW), static_cast<uint32_t>(TH), 1};
  if (!make_tmap_bf16(&tmA, g_nhwc, 4, dims, strides, box)) return 3;
  if (!make_tmap_bf16(&tmB, dc1_nhwc, 4, dims, strides, box)) return 3;
  return launch_gemm(tmA, tmB, g, static_cast<cudaStream_t>(stream), "pk_conv3x3_wgrad");
}
