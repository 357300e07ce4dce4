// painter_b200 — decoder-side helper kernels: conv weight packing, loss bookkeeping and the backward of
// the fused head (LayerNorm2D + GELU + 1x1 conv + masked smooth-L1).  The 3x3 convolution itself runs as
// an implicit GEMM on tcgen05 (gemm.cu, conv modes).
//
// Reference: Painter/models_painter.py:328-333 (decoder_pred), util/vitdet_utils.py:189-209 (LayerNorm2D),
// models_painter.py:433-462 (forward_loss), SegGPT variant models_seggpt.py:448-469.
#include "common.cuh"
#include "host_common.h"
#include "../../include/painter_b200.h"

namespace pk {

// ---------------------------------------------------------------------------------------------
// Conv weight [O=64, C=64, 3, 3] fp32  ->  bf16 GEMM operands
//   fwd  : Wf[o, tap*64 + c]  = W[o, c, dy, dx]            tap = dy*3 + dx
//   dgrad: Wd[c, tap*64 + o]  = W[o, c, 2-dy, 2-dx]
// ---------------------------------------------------------------------------------------------
__global__ void conv_pack_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wf,
                                 __nv_bfloat16* __restrict__ wd) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 64 * 576) return;
  const int o = idx / 576, k = idx % 576, tap = k / 64, c = k % 64;
  const int dy = tap / 3, dx = tap % 3;
  wf[idx] = __float2bfloat16_rn(w[((o * 64 + c) * 3 + dy) * 3 + dx]);
  // here (o, c) play (row = input channel c', column channel o'): row index "o" is the dgrad output channel
  wd[idx] = __float2bfloat16_rn(w[((c * 64 + o) * 3 + (2 - dy)) * 3 + (2 - dx)]);
}

// wgrad GEMM result acc[(tap*64 + c), o]  ->  dW[o, c, dy, dx]
__global__ void conv_wgrad_unpack_kernel(const float* __restrict__ acc, float* __restrict__ dw) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 64 * 64 * 9) return;
  const int o = idx / 576, r = idx % 576, c = r / 9, tap = r % 9;
  dw[idx] = acc[(tap * 64 + c) * 64 + o];
}

// ---------------------------------------------------------------------------------------------
// Loss bookkeeping (forward_loss): per-sample
//   stats[b][0] = sum_{c,y,x} (tgt*std_c + mean_c) * (1 - M)      ("is the unmasked target black?")
//   stats[b][1] = sum_{c,y,x} M * valid
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
loss_prep_kernel(const float* __restrict__ tgts, const uint8_t* __restrict__ mask, int maskB,
                 const float* __restrict__ valid, float* __restrict__ stats, int H, int W, int p) {
  const int b = blockIdx.y;
  const int wt = W / p, Ntok = (H / p) * wt;
  const size_t plane = static_cast<size_t>(H) * W;
  const float mean[3] = {0.485f, 0.456f, 0.406f}, stdv[3] = {0.229f, 0.224f, 0.225f};
  float s0 = 0.f, s1 = 0.f;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < plane;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int y = static_cast<int>(i / W), x = static_cast<int>(i % W);
    const float m = mask[static_cast<size_t>(b % maskB) * Ntok + (y / p) * wt + x / p] ? 1.f : 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const size_t o = (static_cast<size_t>(b) * 3 + c) * plane + i;
      s0 += (tgts[o] * stdv[c] + mean[c]) * (1.f - m);
      s1 += m * valid[o];
    }
  }
  __shared__ float r0[8], r1[8];
  s0 = warp_sum(s0);
  s1 = warp_sum(s1);
  if ((threadIdx.x & 31) == 0) {
    r0[threadIdx.x >> 5] = s0;
    r1[threadIdx.x >> 5] = s1;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, c = 0.f;
    for (int w = 0; w < 8; ++w) {
      a += r0[w];
      c += r1[w];
    }
    atomicAdd(stats + 2 * b, a);
    atomicAdd(stats + 2 * b + 1, c);
  }
}

// loss = sum_b keep_b num_b / (sum_b keep_b den_b + eps);  coef[b] = keep_b / (that denominator)
__global__ void loss_finalize_kernel(const float* __restrict__ stats, const float* __restrict__ num,
                                     float* __restrict__ loss, float* __restrict__ coef, int B, int seggpt) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  float n = 0.f, d = 0.f;
  for (int b = 0; b < B; ++b) {
    const float keep = (seggpt || !(stats[2 * b] < 300.f)) ? 1.f : 0.f;
    n += keep * num[b];
    d += keep * stats[2 * b + 1];
  }
  const float den = seggpt ? d : d + 1e-2f;
  loss[0] = n / den;
  for (int b = 0; b < B; ++b) {
    const float keep = (seggpt || !(stats[2 * b] < 300.f)) ? 1.f : 0.f;
    coef[b] = keep / den;
  }
}

// ---------------------------------------------------------------------------------------------
// Backward of the fused head, one warp per pixel (lane owns channels 2*lane, 2*lane+1).
//   recompute: xh = (c1 - mu) rstd; ln = g*xh + b; ge = gelu(ln); pred = W1 ge + b1
//   dpred_c = gscale * coef[b] * M * valid_c * dloss/dpred;   back through 1x1, GELU, LN2D -> dC1 (bf16)
//   param grads accumulate in registers, one atomic per lane per block at the end.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
head_bwd_kernel(const __nv_bfloat16* __restrict__ c1, const float* __restrict__ tgts,
                const uint8_t* __restrict__ mask, int maskB, const float* __restrict__ valid,
                const float* __restrict__ coef, const float* __restrict__ gscale,
                const float* __restrict__ hp /* head params, 387 floats */, __nv_bfloat16* __restrict__ dc1,
                float* __restrict__ dhp /* grads of [gamma 64 | beta 64 | w 192 | b 3] at offsets 64.. */,
                int B, int H, int W, int p, int loss_kind) {
  const int lane = threadIdx.x & 31;
  const int warps_total = gridDim.x * (blockDim.x >> 5);
  const int gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int k0 = 2 * lane, k1 = 2 * lane + 1;
  const float ga0 = hp[64 + k0], ga1 = hp[64 + k1], be0 = hp[128 + k0], be1 = hp[128 + k1];
  float w0[3], w1[3], b1[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    w0[c] = hp[192 + c * 64 + k0];
    w1[c] = hp[192 + c * 64 + k1];
    b1[c] = hp[384 + c];
  }
  const float gs = gscale ? gscale[0] : 1.f;
  const int wt = W / p, Ntok = (H / p) * wt;
  const size_t plane = static_cast<size_t>(H) * W;
  const size_t npix = static_cast<size_t>(B) * plane;
  float dga0 = 0, dga1 = 0, dbe0 = 0, dbe1 = 0, dw0[3] = {0, 0, 0}, dw1[3] = {0, 0, 0}, db1[3] = {0, 0, 0};
  // PP pixels per warp iteration: the seven shuffle reductions of a pixel form one long dependent chain, so
  // several independent pixels are interleaved to keep the issue slots busy.
  constexpr int PP = 4;
  // 32-bit index math (npix < 2^31 is checked on the host); W % PP == 0 keeps the PP pixels in one row, so the
  // divisions happen once per group.
  const uint32_t npix32 = static_cast<uint32_t>(npix), plane32 = static_cast<uint32_t>(plane);
  for (uint32_t pix0 = static_cast<uint32_t>(gw) * PP; pix0 < npix32; pix0 += static_cast<uint32_t>(warps_total) * PP) {
    float x0[PP], x1[PP], mean[PP], rstd[PP], xh0[PP], xh1[PP], ln0[PP], ln1[PP], ge0[PP], ge1[PP], mk[PP];
    float dg0[PP], dg1[PP];
    uint32_t yx[PP];
    uint32_t raw[PP];
    constexpr bool live[PP] = {true, true, true, true};
    const uint32_t bq = pix0 / plane32, yx0 = pix0 - bq * plane32;
    const uint32_t yq = yx0 / static_cast<uint32_t>(W), xq = yx0 - yq * static_cast<uint32_t>(W);
    const uint8_t* mrow = mask + static_cast<size_t>(bq % maskB) * Ntok + (yq / p) * wt;
    const int bb[PP] = {static_cast<int>(bq), static_cast<int>(bq), static_cast<int>(bq), static_cast<int>(bq)};
#pragma unroll
    for (int u = 0; u < PP; ++u) {
      yx[u] = yx0 + u;
      raw[u] = reinterpret_cast<const uint32_t*>(c1)[static_cast<size_t>(pix0 + u) * 32 + lane];
    }
#pragma unroll
    for (int u = 0; u < PP; ++u) {
      x0[u] = __uint_as_float(raw[u] << 16);
      x1[u] = __uint_as_float(raw[u] & 0xFFFF0000u);
      mk[u] = mrow[(xq + u) / p] ? 1.f : 0.f;
    }
#pragma unroll
    for (int u = 0; u < PP; ++u) mean[u] = x0[u] + x1[u];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int u = 0; u < PP; ++u) mean[u] += __shfl_xor_sync(0xffffffffu, mean[u], o);
#pragma unroll
    for (int u = 0; u < PP; ++u) {
      mean[u] *= (1.f / 64);
      const float d0 = x0[u] - mean[u], d1 = x1[u] - mean[u];
      xh0[u] = d0;
      xh1[u] = d1;
      rstd[u] = d0 * d0 + d1 * d1;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int u = 0; u < PP; ++u) rstd[u] += __shfl_xor_sync(0xffffffffu, rstd[u], o);
#pragma unroll
    for (int u = 0; u < PP; ++u) {
      rstd[u] = rsqrtf(rstd[u] * (1.f / 64) + 1e-6f);
      xh0[u] *= rstd[u];
      xh1[u] *= rstd[u];
      ln0[u] = ga0 * xh0[u] + be0;
      ln1[u] = ga1 * xh1[u] + be1;
      ge0[u] = gelu_erf(ln0[u]);
      ge1[u] = gelu_erf(ln1[u]);
      dg0[u] = 0.f;
      dg1[u] = 0.f;
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float pr[PP];
#pragma unroll
      for (int u = 0; u < PP; ++u) pr[u] = w0[c] * ge0[u] + w1[c] * ge1[u];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1)
#pragma unroll
        for (int u = 0; u < PP; ++u) pr[u] += __shfl_xor_sync(0xffffffffu, pr[u], o);
#pragma unroll
      for (int u = 0; u < PP; ++u) {
        const size_t o = (static_cast<size_t>(bb[u]) * 3 + c) * plane + yx[u];
        const float d = pr[u] + b1[c] - tgts[o];
        float dl;
        if (loss_kind == 0) dl = fminf(fmaxf(d * 100.f, -1.f), 1.f);
        else if (loss_kind == 1) dl = d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f);
        else if (loss_kind == 2) dl = 2.f * d;
        else dl = 0.5f * ((d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f)) + 2.f * d);
        const float dp = live[u] ? gs * coef[bb[u]] * mk[u] * valid[o] * dl : 0.f;
        dw0[c] += dp * ge0[u];
        dw1[c] += dp * ge1[u];
        db1[c] += dp;
        dg0[u] += dp * w0[c];
        dg1[u] += dp * w1[c];
      }
    }
    float dx0[PP], dx1[PP], c1m[PP], c2m[PP];
#pragma unroll
    for (int u = 0; u < PP; ++u) {
      const float dln0 = dg0[u] * gelu_erf_grad(ln0[u]), dln1 = dg1[u] * gelu_erf_grad(ln1[u]);
      dga0 += dln0 * xh0[u]; dga1 += dln1 * xh1[u];
      dbe0 += dln0; dbe1 += dln1;
      dx0[u] = dln0 * ga0;
      dx1[u] = dln1 * ga1;
      c1m[u] = dx0[u] + dx1[u];
      c2m[u] = dx0[u] * xh0[u] + dx1[u] * xh1[u];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int u = 0; u < PP; ++u) {
        c1m[u] += __shfl_xor_sync(0xffffffffu, c1m[u], o);
        c2m[u] += __shfl_xor_sync(0xffffffffu, c2m[u], o);
      }
#pragma unroll
    for (int u = 0; u < PP; ++u) {
      if (!live[u]) continue;
      const float a1 = c1m[u] * (1.f / 64), a2 = c2m[u] * (1.f / 64);
      const float o0 = rstd[u] * (dx0[u] - a1 - xh0[u] * a2), o1 = rstd[u] * (dx1[u] - a1 - xh1[u] * a2);
      reinterpret_cast<uint32_t*>(dc1)[static_cast<size_t>(pix0 + u) * 32 + lane] = pack_bf16x2(o0, o1);
    }
  }
  // block reduction through shared memory, then atomics
  __shared__ float red[8][323];
  const int wq = threadIdx.x >> 5;
  red[wq][k0] = dga0; red[wq][k1] = dga1;
  red[wq][64 + k0] = dbe0; red[wq][64 + k1] = dbe1;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    red[wq][128 + c * 64 + k0] = dw0[c];
    red[wq][128 + c * 64 + k1] = dw1[c];
  }
  if (lane == 0) {
    // db1 is identical across lanes (dp is warp-uniform)
    red[wq][320] = db1[0]; red[wq][321] = db1[1]; red[wq][322] = db1[2];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 323; i += blockDim.x) {
    float s = 0.f;
    for (int w = 0; w < 8; ++w) s += red[w][i];
    atomicAdd(dhp + 64 + i, s);
  }
}

// ---------------------------------------------------------------------------------------------
// head_bwd2_kernel: the same math with a LANE PAIR per pixel (each lane owns 32 of the pixel's 64 channels in
// registers: LayerNorm statistics, the 1x1 convolution and its transpose cost 7 pair-shuffles per pixel instead of 35
// warp-wide ones) and the per-channel parameter gradients reduced over the 16 pixels of a warp with a butterfly
// transpose-reduce (30 shuffles per quantity: afterwards lane l holds channels 32 (l & 1) + 2 (l >> 1) + {0, 1} summed
// over the warp's pixels).  Head parameters are staged once per block in shared memory as {gamma, beta, w0, w1}, {w2}
// records (two broadcast LDS.128 per channel); no global or __constant__ state.
// ---------------------------------------------------------------------------------------------
// v[32] per lane, reduced over the 16 lanes of equal parity; result v[0], v[1] (see above)
__device__ __forceinline__ void transpose_reduce_pairs(float (&v)[32], int lane) {
#pragma unroll
  for (int s = 16; s >= 2; s >>= 1) {
    const bool up = (lane & s) != 0;
#pragma unroll
    for (int i = 0; i < s; ++i) {
      const float send = up ? v[i] : v[i + s];
      const float keep = up ? v[i + s] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
    }
  }
}
__device__ __forceinline__ float pair_sum(float v) { return v + __shfl_xor_sync(0xffffffffu, v, 1); }
// volatile shared-memory load of one parameter record: keeps ptxas from hoisting all 64 records of a pass into
// registers (which cost 160 registers and spills); the loads are warp-uniform broadcasts, two per channel
__device__ __forceinline__ float4 lds_v4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float lds_f(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}

__global__ void __launch_bounds__(128, 2)
head_bwd2_kernel(const __nv_bfloat16* __restrict__ c1, const float* __restrict__ tgts,
                 const uint8_t* __restrict__ mask, int maskB, const float* __restrict__ valid,
                 const float* __restrict__ coef, const float* __restrict__ gscale, const float* __restrict__ hp,
                 __nv_bfloat16* __restrict__ dc1, float* __restrict__ dhp, int B, int H, int W, int p, int loss_kind,
                 int pix_per_warp) {
  __shared__ float4 prm[64][2];     // [k] = {gamma, beta, w0, w1}, {w2, -, -, -}
  __shared__ float red[4][323];
  const int lane = threadIdx.x & 31, wq = threadIdx.x >> 5;
  const int hsel = lane & 1, kb = hsel * 32;
  for (int k = threadIdx.x; k < 64; k += blockDim.x) {
    prm[k][0] = make_float4(hp[64 + k], hp[128 + k], hp[192 + k], hp[256 + k]);
    prm[k][1] = make_float4(hp[320 + k], 0.f, 0.f, 0.f);
  }
  __syncthreads();
  const float b1_0 = hp[384], b1_1 = hp[385], b1_2 = hp[386];
  const uint32_t prm_s = smem_u32(&prm[0][0]) + static_cast<uint32_t>(kb) * 32u;   // this lane's 32 records
  const float gs = gscale ? gscale[0] : 1.f;
  const int wt = W / p, Ntok = (H / p) * wt;
  const uint32_t plane = static_cast<uint32_t>(H) * W;
  const uint32_t npix = static_cast<uint32_t>(B) * plane;
  float acc[5][2] = {{0, 0}, {0, 0}, {0, 0}, {0, 0}, {0, 0}};   // dgamma, dbeta, dW0, dW1, dW2 of this lane's channels
  float db0 = 0.f, db1v = 0.f, db2 = 0.f;
  const uint32_t warp_global = blockIdx.x * (blockDim.x >> 5) + wq;
  const uint32_t base0 = warp_global * static_cast<uint32_t>(pix_per_warp);
  for (int it = 0; it < pix_per_warp; it += 16) {
    const uint32_t pix = base0 + it + (lane >> 1);
    const bool live = pix < npix;
    const uint32_t pc = live ? pix : npix - 1;
    uint32_t raw[16];
    const uint4* src = reinterpret_cast<const uint4*>(c1 + static_cast<size_t>(pc) * 64 + kb);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint4 u = src[q];
      raw[4 * q] = u.x; raw[4 * q + 1] = u.y; raw[4 * q + 2] = u.z; raw[4 * q + 3] = u.w;
    }
    const uint32_t bq = pc / plane, yx = pc - bq * plane;
    const uint32_t yq = yx / static_cast<uint32_t>(W), xq = yx - yq * static_cast<uint32_t>(W);
    const float mk = mask[static_cast<size_t>(bq % maskB) * Ntok + (yq / p) * wt + xq / p] ? 1.f : 0.f;
    float tg[3], vl[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const size_t o = (static_cast<size_t>(bq) * 3 + c) * plane + yx;
      tg[c] = tgts[o];
      vl[c] = valid[o];
    }
    const float cf = live ? gs * coef[bq] * mk : 0.f;
#define HB2_X(j) (((j) & 1) ? __uint_as_float(raw[(j) >> 1] & 0xFFFF0000u) : __uint_as_float(raw[(j) >> 1] << 16))
    // ---- statistics over the pixel's 64 channels (32 here + 32 in the partner lane)
    float mean = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) mean += HB2_X(j);
    mean = pair_sum(mean) * (1.f / 64);
    float var = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float a = HB2_X(j) - mean;
      var += a * a;
    }
    const float rstd = rsqrtf(pair_sum(var) * (1.f / 64) + 1e-6f);
    // ---- forward: gelu(ln) of this lane's channels, pred_c
    float ge[32];
    float pr0 = 0.f, pr1 = 0.f, pr2 = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float4 p0 = lds_v4(prm_s + j * 32);
      const float w2 = lds_f(prm_s + j * 32 + 16);
      const float g = gelu_erf(p0.x * ((HB2_X(j) - mean) * rstd) + p0.y);
      ge[j] = g;
      pr0 += p0.z * g;
      pr1 += p0.w * g;
      pr2 += w2 * g;
    }
    float dp[3];
    {
      const float prd[3] = {pair_sum(pr0) + b1_0, pair_sum(pr1) + b1_1, pair_sum(pr2) + b1_2};
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float d = prd[c] - tg[c];
        float dl;
        if (loss_kind == 0) dl = fminf(fmaxf(d * 100.f, -1.f), 1.f);
        else if (loss_kind == 1) dl = d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f);
        else if (loss_kind == 2) dl = 2.f * d;
        else dl = 0.5f * ((d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f)) + 2.f * d);
        dp[c] = cf * vl[c] * dl;
      }
    }
    if (hsel == 0) {
      db0 += dp[0];
      db1v += dp[1];
      db2 += dp[2];
    }
    // ---- backward through 1x1, GELU, LayerNorm2D
    float t[32];
#pragma unroll
    for (int c = 0; c < 3; ++c) {      // dW_c[k] += dp_c * gelu(ln_k)
#pragma unroll
      for (int j = 0; j < 32; ++j) t[j] = ge[j] * dp[c];
      transpose_reduce_pairs(t, lane);
      acc[2 + c][0] += t[0];
      acc[2 + c][1] += t[1];
    }
    float dln[32];
    float a1 = 0.f, a2 = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float4 p0 = lds_v4(prm_s + j * 32);
      const float w2 = lds_f(prm_s + j * 32 + 16);
      const float xh = (HB2_X(j) - mean) * rstd;
      const float d = (dp[0] * p0.z + dp[1] * p0.w + dp[2] * w2) * gelu_erf_grad(p0.x * xh + p0.y);
      dln[j] = d;
      const float dx = d * p0.x;
      a1 += dx;
      a2 += dx * xh;
      t[j] = d * xh;
    }
    transpose_reduce_pairs(t, lane);    // dgamma
    acc[0][0] += t[0];
    acc[0][1] += t[1];
#pragma unroll
    for (int j = 0; j < 32; ++j) t[j] = dln[j];
    transpose_reduce_pairs(t, lane);    // dbeta
    acc[1][0] += t[0];
    acc[1][1] += t[1];
    a1 = pair_sum(a1) * (1.f / 64);
    a2 = pair_sum(a2) * (1.f / 64);
    if (live) {
      uint4* dst = reinterpret_cast<uint4*>(dc1 + static_cast<size_t>(pix) * 64 + kb);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint32_t o[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int j = q * 8 + e * 2;
          const float x0 = (HB2_X(j) - mean) * rstd, x1 = (HB2_X(j + 1) - mean) * rstd;
          o[e] = pack_bf16x2(rstd * (dln[j] * lds_f(prm_s + j * 32) - a1 - x0 * a2),
                             rstd * (dln[j + 1] * lds_f(prm_s + (j + 1) * 32) - a1 - x1 * a2));
        }
        dst[q] = make_uint4(o[0], o[1], o[2], o[3]);
      }
    }
#undef HB2_X
  }
  db0 = warp_sum(db0);
  db1v = warp_sum(db1v);
  db2 = warp_sum(db2);
  {
    const int k0 = kb + 2 * (lane >> 1);
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      red[wq][k0 + e] = acc[0][e];
      red[wq][64 + k0 + e] = acc[1][e];
#pragma unroll
      for (int c = 0; c < 3; ++c) red[wq][128 + c * 64 + k0 + e] = acc[2 + c][e];
    }
  }
  if (lane == 0) {
    red[wq][320] = db0; red[wq][321] = db1v; red[wq][322] = db2;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 323; i += blockDim.x) {
    float s = 0.f;
    for (int w = 0; w < 4; ++w) s += red[w][i];
    atomicAdd(dhp + 64 + i, s);
  }
}

// conv bias gradient: db[o] = sum_pix dC1[pix, o]  (bf16 [npix, 64])  -> reuse the generic column sum
}  // namespace pk

using namespace pk;

extern "C" int pk_conv3x3_pack(const float* w, void* wf_bf16, void* wd_bf16, void* stream) {
  PK_CHECK(w && wf_bf16 && wd_bf16, "pk_conv3x3_pack: null pointer");
  conv_pack_kernel<<<(64 * 576 + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      w, static_cast<__nv_bfloat16*>(wf_bf16), static_cast<__nv_bfloat16*>(wd_bf16));
  PK_LAUNCH_CHECK("pk_conv3x3_pack");
  return 0;
}
extern "C" int pk_conv3x3_wgrad_unpack(const float* acc, float* dw, void* stream) {
  PK_CHECK(acc && dw, "pk_conv3x3_wgrad_unpack: null pointer");
  conv_wgrad_unpack_kernel<<<(64 * 576 + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(acc, dw);
  PK_LAUNCH_CHECK("pk_conv3x3_wgrad_unpack");
  return 0;
}
extern "C" int pk_loss_prep(const float* tgts, const uint8_t* mask, int maskB, const float* valid,
                            float* stats_zeroed, int B, int H, int W, int p, void* stream) {
  PK_CHECK(tgts && mask && valid && stats_zeroed && maskB >= 1, "pk_loss_prep: bad args");
  dim3 grid(64, B);
  loss_prep_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(tgts, mask, maskB, valid, stats_zeroed,
                                                                        H, W, p);
  PK_LAUNCH_CHECK("pk_loss_prep");
  return 0;
}
extern "C" int pk_loss_finalize(const float* stats, const float* num, float* loss, float* coef, int B,
                                int seggpt, void* stream) {
  PK_CHECK(stats && num && loss && coef, "pk_loss_finalize: null pointer");
  loss_finalize_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(stats, num, loss, coef, B, seggpt);
  PK_LAUNCH_CHECK("pk_loss_finalize");
  return 0;
}
static int g_head_bwd_legacy = 0;
// test hook: 1 = the warp-per-pixel kernel of round 1 (kept as an independent implementation to cross-check)
extern "C" void pk_head_bwd_legacy(int on) { g_head_bwd_legacy = on; }
extern "C" int pk_decoder_head_bwd(const void* c1, const float* tgts, const uint8_t* mask, int maskB,
                                   const float* valid, const float* coef, const float* gscale,
                                   const float* head_params, void* dc1, float* dhead_params_zeroed, int B,
                                   int H, int W, int p, int loss_kind, void* stream) {
  PK_CHECK(c1 && tgts && mask && valid && coef && head_params && dc1 && dhead_params_zeroed,
           "pk_decoder_head_bwd: null pointer");
  PK_CHECK(W % 4 == 0 && static_cast<long long>(B) * H * W < (1ll << 31),
           "pk_decoder_head_bwd: W must be a multiple of 4 and B*H*W < 2^31");
  int TW, TH;   // the image sizes the forward (pk_decoder_head_fwd) accepts
  PK_CHECK(conv_tile_geometry(H, W, 128, &TW, &TH), "pk_decoder_head_bwd: unsupported image size %dx%d", H, W);
  if (g_head_bwd_legacy) {
    const int grid = sm_count() * 4;
    head_bwd_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __nv_bfloat16*>(c1), tgts, mask, maskB, valid, coef, gscale, head_params,
        static_cast<__nv_bfloat16*>(dc1), dhead_params_zeroed, B, H, W, p, loss_kind);
  } else {
    // a lane pair per pixel; every warp walks `ppw` consecutive pixels (a multiple of 16) so that the block-level
    // parameter-gradient atomics stay ~4 per SM-resident block
    const long long npix = static_cast<long long>(B) * H * W;
    const long long warps_target = static_cast<long long>(sm_count()) * 16;
    long long ppw = (npix + warps_target - 1) / warps_target;
    ppw = (ppw + 15) / 16 * 16;
    const long long warps = (npix + ppw - 1) / ppw;
    const int grid = static_cast<int>((warps + 3) / 4);
    head_bwd2_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __nv_bfloat16*>(c1), tgts, mask, maskB, valid, coef, gscale, head_params,
        static_cast<__nv_bfloat16*>(dc1), dhead_params_zeroed, B, H, W, p, loss_kind, static_cast<int>(ppw));
  }
  PK_LAUNCH_CHECK("pk_decoder_head_bwd");
  return 0;
}
