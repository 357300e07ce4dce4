/* painter_b200 — C ABI of the B200-native Painter/SegGPT hot path.
 *
 * The reference (baaivision/Painter) has no FFI layer: its hot path is the Python module
 * Painter/models_painter.py (+ SegGPT/SegGPT_inference/models_seggpt.py, util/vitdet_utils.py), every
 * arithmetic step being a torch op.  Each entry point below replaces one group of those torch call
 * sites (cited per function) with a hand-written sm_100a kernel.  The host-side mirror of the
 * reference nn.Module API (painter_b200/models_painter.py, models_seggpt.py) calls these through
 * ctypes; see INTEGRATION.md for the binding.
 *
 * Conventions
 *  - all pointers are DEVICE pointers owned by the caller (PyTorch's caching allocator); the library
 *    never allocates device memory and keeps no pointer past return;
 *  - `stream` is a cudaStream_t passed as void*; kernels are enqueued asynchronously on it;
 *  - return value 0 = ok; otherwise pk_last_error() describes the failure (thread-local);
 *  - bf16 = raw 16-bit bfloat16, f32 = IEEE float. "tokens" are rows of [B*h*w, C] matrices.
 */
#ifndef PAINTER_B200_H
#define PAINTER_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

int pk_version(void);
const char* pk_last_error(void);
/* number of kernel launches issued by this library since load (bench.py's gpu_launches claim) */
long long pk_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Dense contraction on tcgen05 tensor cores:  C[M,N] = A[M,K] . B[N,K]^T   (bf16 x bf16 -> fp32)
 * Replaces every nn.Linear / F.linear on the path (models_painter.py:60-61,76,87 qkv/proj; timm Mlp
 * fc1/fc2 used at :201; decoder_embed :327,423) and their autograd backward (dgrad / wgrad GEMMs).
 *   transA = 0: A stored [M,K] row-major (lda = row stride, elements)   transA = 1: stored [K,M]
 *   transB = 0: B stored [N,K] row-major (ldb)                          transB = 1: stored [K,N]
 * Epilogues (PkEpilogue.kind):
 */
enum {
  PK_EPI_BF16 = 0,    /* out(bf16)[m,n] = alpha*acc + bias[n]                                     */
  PK_EPI_F32 = 1,     /* out(f32)[m,n]  = alpha*acc + bias[n] (+ out[m,n] when accumulate != 0)    */
  PK_EPI_GELU = 2,    /* out(bf16) = z = acc + bias ; out2(bf16) = gelu_erf(bf16(z))  (Mlp fc1+act) */
  PK_EPI_RESID = 3,   /* out(f32) = aux_f32[m,n] + rowscale[m / rows_per_group] * (acc + bias[n])
                         (residual add + DropPath scale, models_painter.py:229-230)               */
  PK_EPI_DGELU = 4,   /* out(bf16) = acc * gelu'(aux_bf16[m,n])        (backward through GELU)     */
  PK_EPI_PIXSHUF = 5, /* out(bf16) NHWC [B, h*p, w*p, c]: decoder_embed + 'nhwpqc->nchpwq' pixel
                         shuffle (models_painter.py:423-428), rows m=(b,i,j), cols n=(r,s,c)       */
};
typedef struct {
  int kind;
  void* out;
  void* out2;
  const float* bias;
  const void* aux;
  const float* rowscale;
  int ldc;            /* row stride of out/out2 (elements) */
  int ld_aux;         /* row stride of aux (elements) */
  int rows_per_group; /* rows sharing one rowscale entry */
  int accumulate;     /* PK_EPI_F32: 0 overwrite, 1 out += , 2 out zero-initialised, split-K atomics */
  float alpha;        /* scales acc (alpha == 0 is taken as 1, so a zero-initialised struct computes acc) */
  int ps_h, ps_w, ps_p, ps_c; /* pixel shuffle geometry: token grid h x w, patch p, channels c */
} PkEpilogue;

int pk_gemm_bf16(const void* A, const void* B, int M, int N, int K, int lda, int ldb, int transA,
                 int transB, const PkEpilogue* epi, void* stream);

/* test hooks: force the GEMM N-tile (64/128/256) or split-K factor; 0 restores the heuristics */
void pk_gemm_force_bn(int bn);
void pk_gemm_force_splits(int s);
/* Host-only views of the GEMM scheduler (schedule tests; no device work).  pk_gemm_plan: out9 = {cta_pair_kernel,
 * BN, row blocks, column blocks, splits, k-blocks per split, stream-K units per cluster, raster group, workers}.
 * pk_gemm_plan_walk: the (row block, column block, kb0, kb1) items worker `worker` processes, 4 ints each; returns
 * minus the item count. */
int pk_gemm_plan(int M, int N, int K, int kind, int accumulate, int* out9);
int pk_gemm_plan_walk(int M, int N, int K, int kind, int accumulate, int worker, int* out4, int max_items);
/* 0 = single-CTA tiles (128 x BN), 1 = CTA pairs / cta_group::2 (256 x BN) whenever the shape allows */
void pk_gemm_use_2cta(int on);

/* ------------------------------------------------------------------------------------------------
 * LayerNorm over channels (nn.LayerNorm(eps=1e-6): models_painter.py:193,200 norm1/norm2, :315,:417 final norm).
 * x fp32 [M, C] (row stride ldx) -> out (bf16 if out_is_bf16 else fp32; row stride ldo, so it can be a column
 * slice of the [M, 4C] decoder input, models_painter.py:422); mean/rstd [M] saved for backward (nullable).
 * bwd: dx = LN'(dy) (+ dres); dgamma/dbeta += column sums (caller initialises; deterministic two-stage
 * reduction through `workspace`).                                                                         */
int pk_layernorm_fwd(const float* x, int ldx, const float* gamma, const float* beta, float eps, void* out,
                     int ldo, int out_is_bf16, float* mean, float* rstd, int M, int C, void* stream);
long long pk_layernorm_bwd_ws_floats(int M, int C); /* fp32 elements of `workspace` (per-block partial sums) */
/* pk_layernorm_bwd fused with pk_scale_cast_colsum of its result (the backward of `x + drop_path(attn(norm1(x)))`
 * feeds norm2's input gradient, DropPath-scaled and cast to bf16, straight into the proj GEMMs; models_painter.py:
 * 216-235): also writes dx_bf16 = bf16(rowscale[row / rows_per_group] * dx) and adds its column sums to colsum[C]. */
int pk_layernorm_bwd_cast(const void* dy, int dy_is_bf16, int lddy, const float* x, int ldx, const float* mean, const float* rstd,
                          const float* gamma, const float* dres, float* dx, float* dgamma, float* dbeta,
                          float* workspace, const float* rowscale, int rows_per_group, void* dx_bf16, float* colsum,
                          int M, int C, void* stream);
int pk_layernorm_bwd(const void* dy, int dy_is_bf16, int lddy, const float* x, int ldx, const float* mean, const float* rstd,
                     const float* gamma, const float* dres, float* dx, float* dgamma, float* dbeta,
                     float* workspace, int M, int C, void* stream);

/* PatchEmbed lowering (util/vitdet_utils.py:178-186, models_painter.py:387-388): rows of (c,r,s)-ordered
 * patches of imgs then tgts, bf16 [2*B*h*w, Cin*p*p]; the conv itself is pk_gemm_bf16 on these rows.       */
int pk_im2col_patch(const float* imgs, const float* tgts, void* out_bf16, int B, int Cin, int H, int W, int p,
                    void* stream);

/* Token assembly (models_painter.py:392-409; SegGPT type tokens models_seggpt.py:414-420) and its backward.
 * E fp32 [2B*N, C] (x rows then y rows); mask uint8 [maskB, N] (maskB = 1 broadcasts); pos fp32 [N, C];
 * type_emb fp32 [B, C] or NULL.  bwd: dE bf16 (y rows gated by 1-mask), dpos [N,C], dseg/dmask_token [C]
 * (atomically accumulated, caller zero-initialises).                                                      */
int pk_assemble_tokens(const float* E, const uint8_t* mask, int maskB, const float* mask_token,
                       const float* seg_x, const float* seg_y, const float* pos, const float* type_emb,
                       float* out, int B, int N, int C, void* stream);
int pk_assemble_tokens_bwd(const float* dZ, const uint8_t* mask, int maskB, void* dE_bf16, float* dpos,
                           float* dseg_x, float* dseg_y, float* dmask_token, int B, int N, int C, void* stream);

/* get_abs_pos (util/vitdet_utils.py:141-157): F.interpolate(bicubic, align_corners=False), NHWC [sh,sw,C] ->
 * [h,w,C]; bwd scatters atomically into a zero-initialised [sh,sw,C].                                      */
int pk_bicubic_fwd(const float* src, float* dst, int sh, int sw, int h, int w, int C, void* stream);
int pk_bicubic_bwd(const float* ddst, float* dsrc_accum, int sh, int sw, int h, int w, int C, void* stream);

/* Early merge (models_painter.py:414-415): out = 0.5*(z[:half] + z[half:]); bwd duplicates 0.5*d.          */
int pk_merge_halves(const float* z, float* out, long long half_elems, void* stream);
int pk_merge_halves_bwd(const float* d, float* out, long long half_elems, void* stream);

/* fp32 -> bf16 operand casts; optional per-row-group scale (DropPath backward, timm drop_path) and fused
 * column sums (bias gradients).                                                                           */
int pk_cast_bf16(const float* in, void* out_bf16, long long n, void* stream);
int pk_scale_cast_colsum(const float* in, int ldin, const float* rowscale, int rows_per_group, void* out_bf16,
                         float* colsum, int M, int C, void* stream);
int pk_colsum_bf16(const void* in_bf16, int ldin, float* colsum, int M, int C, void* stream);

/* Window attention plumbing (util/vitdet_utils.py:16-60 window_partition / window_unpartition; reachable only
 * through Painter(window_block_indexes=[...]), models_painter.py:220-227): zero-padded bf16 partition of the
 * [B,H,W,C] token grid into [B*nWh*nWw, ws, ws, C]; inverse: out = (resid or 0) + rowscale[b] * window value.   */
int pk_window_partition_bf16(const void* in, void* out, int B, int H, int W, int C, int ws, void* stream);
int pk_window_unpartition(const float* win, const float* resid, const float* rowscale, float* out, int B, int H,
                          int W, int C, int ws, void* stream);

/* SegGPT multi-prompt feature ensemble + residual (models_seggpt.py:220-231,:233): a, z, out fp32 [G*P, N, C]. */
int pk_ensemble_resid(const float* a, const float* z, float* out, int G, int P, int N, int C, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused attention with decomposed relative-position bias (models_painter.py:73-86 + util/vitdet_utils.py:
 * 63-125).  qkv bf16 [B*h*w, 3*heads*64] with columns (3, head, 64); th/tw = pk_relpos_table_bf16 outputs
 * (bf16, zero-padded to th_pad/tw_pad rows, multiples of 16); w must divide 112 (2,4,7,8,14,28,56).
 * Limits: fwd th_pad <= 256 (h <= 128), bwd th_pad <= 224 (h <= 112), both tw_pad <= 112 (w <= 56); a forward at
 * 112 < h <= 128 runs, its backward is refused.  Shapes past the limits are refused before any launch.
 * fwd: out bf16 [B*N, heads*64], lse fp32 [B*heads, N] (log2 domain, nullable).
 * bwd: dqkv bf16 like qkv; dTh [2h-1,64], dTw [2w-1,64] fp32, added to (zero-initialise);
 *      scratch: delta [B*heads*N], relh_g [B*heads*Np*h], relw_g [B*heads*Np*w] (Np = N rounded up to 128), dt_ws
 *      [pk_attn_bwd_ws_floats(B, heads, h, w)] fp32 (per-CTA partial table gradients, reduced by a
 *      second kernel instead of same-address atomics).                                                     */
int pk_relpos_table_bf16(const float* table, void* out_bf16, int L, int Lpad, void* stream);
int pk_attn_fwd(const void* qkv, const void* th, const void* tw, void* out, float* lse, int B, int heads, int h,
                int w, int th_pad, int tw_pad, void* stream);
int pk_attn_bwd(const void* qkv, const void* O, const void* dO, const float* lse, const void* th, const void* tw,
                void* dqkv, float* dTh, float* dTw, float* delta, float* relh_g, float* relw_g, float* dt_ws,
                int B, int heads, int h, int w, int th_pad, int tw_pad, void* stream);
long long pk_attn_bwd_ws_floats(int B, int heads, int h, int w);
/* Training pair: pk_attn_fwd_save additionally stores every query's log2e-scaled bias rows (rel_h / rel_w of
 * vitdet_utils.py:113-123) in relh_g / relw_g (B*heads*Np*h resp. B*heads*Np*w floats, Np = N rounded up to 128; per
 * 128-query tile, query row innermost); pk_attn_bwd_saved takes them as INPUTS, so its dQ kernel starts from coalesced
 * loads instead of recomputing the two bias GEMMs and Toeplitz gathers.  Results are identical to pk_attn_fwd /
 * pk_attn_bwd.                                                                                                  */
int pk_attn_fwd_save(const void* qkv, const void* th, const void* tw, void* out, float* lse, float* relh_g,
                     float* relw_g, int B, int heads, int h, int w, int th_pad, int tw_pad, void* stream);
int pk_attn_bwd_saved(const void* qkv, const void* O, const void* dO, const float* lse, const void* th, const void* tw,
                      void* dqkv, float* dTh, float* dTw, float* delta, const float* relh_g, const float* relw_g,
                      float* dt_ws, int B, int heads, int h, int w, int th_pad, int tw_pad, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Decoder head (models_painter.py:328-333,430 decoder_pred = conv3x3 -> LayerNorm2D -> GELU -> conv1x1;
 * util/vitdet_utils.py:189-209) fused with forward_loss (:433-462) and patchify (:355-368).
 * g_nhwc: bf16 [B, H, W, 64] (output of the PK_EPI_PIXSHUF GEMM). wmat/wmat_t: pk_conv3x3_pack outputs.
 * Image sizes: the conv runs on tiles of 128 pixels (wgrad: 64), min(W, 64) wide, which must tile the image: W a
 * multiple of 64 with H even, or W < 64 dividing 64 with H a multiple of 128 / W.  Every decoder entry point
 * refuses other sizes (W = 48 or 96, for example) before any launch.
 * head_params: fp32 [387] = conv3x3 bias[64] | LN2D weight[64] | LN2D bias[64] | conv1x1 weight[3][64] | bias[3].
 * fwd writes c1 (bf16 conv output, NHWC), patch_out fp32 [B, N, p*p*3] (= patchify(pred)), num[B] += sum
 * loss*mask*valid.  loss_kind: 0 smoothl1(beta .01), 1 l1, 2 l2, 3 l1l2.
 * pk_loss_prep: stats[b] = {sum (tgt*std+mean)*(1-M), sum M*valid};  pk_loss_finalize: loss + per-sample
 * coefficient keep_b/den (the `inds_ign` rule of :446-448; seggpt != 0 selects models_seggpt.py:457-468).      */
int pk_conv3x3_pack(const float* w, void* wf_bf16, void* wd_bf16, void* stream);
int pk_loss_prep(const float* tgts, const uint8_t* mask, int maskB, const float* valid, float* stats_zeroed,
                 int B, int H, int W, int p, void* stream);
int pk_decoder_head_fwd(const void* g_nhwc, const void* wmat, const float* head_params, const float* tgts,
                        const uint8_t* mask, int maskB, const float* valid, void* c1_out, float* patch_out,
                        float* num, int B, int H, int W, int p, int loss_kind, void* stream);
int pk_loss_finalize(const float* stats, const float* num, float* loss, float* coef, int B, int seggpt,
                     void* stream);
int pk_decoder_head_bwd(const void* c1, const float* tgts, const uint8_t* mask, int maskB, const float* valid,
                        const float* coef, const float* gscale, const float* head_params, void* dc1,
                        float* dhead_params_zeroed, int B, int H, int W, int p, int loss_kind, void* stream);
int pk_conv3x3_dgrad_unshuffle(const void* dc1_nhwc, const void* wmat_t, void* out_tok, int B, int H, int W,
                               int p, void* stream);
int pk_conv3x3_wgrad(const void* g_nhwc, const void* dc1_nhwc, float* out, int B, int H, int W, void* stream);
int pk_conv3x3_wgrad_unpack(const float* acc, float* dw, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Optimizer step (SURVEY §8 f.1): fused multi-tensor AdamW with per-tensor lr / weight decay (the groups of
 * Painter/util/lr_decay.py:param_groups_lrd, main_train.py:344-348) and the global gradient norm of
 * util/misc.py:252-278.  `tensors_dev`: device array of PkOptTensor; `chunks_dev`: device array of int pairs
 * (tensor index, chunk index) - one CUDA block per chunk of pk_opt_chunk_elems() elements.  gscale (nullable device
 * scalar) multiplies every gradient (1 / loss scale, clip coefficient); gscale_cap > 0 clamps it from above
 * (clip coefficient min(1, .)).  pk_grad_sumsq adds sum(g^2) over all tensors to out_zeroed[0].
 * pk_droppath_scales: timm DropPath (0.3.2 layers/drop.py; models_painter.py:199,229-230) for a whole step in one
 * launch: out[i] = floor(round_to_dtype(keep[i] + r[i])) / keep[i], r = the torch.rand draws (dtype code 0 fp32,
 * 1 bf16, 2 fp16: the reference adds in the branch output's dtype).                                             */
typedef struct PkOptTensor {
  float* p;
  float* g;
  float* m;
  float* v;
  void* w16;      /* optional bf16 copy of p refreshed by the step (the tensor-core operand), or NULL */
  long long n;
  float lr, wd;
} PkOptTensor;
int pk_opt_chunk_elems(void);
/* zero_grad != 0: every gradient element is overwritten with 0 after it has been consumed (the flat gradient
 * arena is left clean for the next backward); found_inf (nullable device scalar): non-zero => the whole step is a
 * no-op (torch.cuda.amp.GradScaler.step semantics, util/misc.py:266). */
int pk_adamw_step(const PkOptTensor* tensors_dev, const int* chunks_dev, int nchunks, double beta1, double beta2,
                  double eps, int step, const float* gscale, float gscale_cap, int zero_grad,
                  const float* found_inf, void* stream);
/* pk_adamw_step for a CUDA-graph-captured training step (painter_b200.train_utils.GraphedTrainStep): the bias
   corrections 1 / (1 - beta1^t), 1 / sqrt(1 - beta2^t) are read from bc_dev[0..1] at run time. */
int pk_adamw_step_graph(const PkOptTensor* tensors_dev, const int* chunks_dev, int nchunks, double beta1,
                        double beta2, double eps, const float* bc_dev, const float* gscale, float gscale_cap,
                        int zero_grad, const float* found_inf, void* stream);
int pk_grad_sumsq(const PkOptTensor* tensors_dev, const int* chunks_dev, int nchunks, float* out_zeroed, void* stream);
int pk_droppath_scales(const void* r, int dtype_code, const float* keep, float* out, int n, void* stream);
/* Persistent kernels (the tcgen05 GEMMs) use at most `n` SMs (0 = all): leaves room for a concurrent NCCL kernel
 * so that statically partitioned tiles never run as a second wave (multi-GPU backward).  Returns the old value. */
int pk_set_sm_budget(int n);
/* Programmatic dependent launch of the library's hot kernels (default on; PK_PDL=0 in the environment or
   pk_set_pdl(0) turns the launch attribute off).  Returns the previous setting. */
int pk_set_pdl(int on);

/* ------------------------------------------------------------------------------------------------
 * Inference pre/post-processing on the device (SURVEY §8 f.2).  Replaces the numpy / torch-CPU arithmetic around the
 * forward in SegGPT/SegGPT_inference/seggpt_engine.py:26-53 (run_one_image), :56-103 (inference_image), :106-181
 * (inference_video) and Painter/eval/ade20k_semantic/painter_inference_segm.py:67-93 (run_one_image).
 * dtype codes of image sources: 0 = uint8 (divided by 255.), 1 = fp32 in [0,1], 2 = fp64 in [0,1].
 *  pk_stitch_normalize  canvas[p,c,y,x] fp32 NCHW [P,3,2S,S] = ((top|bottom)[p][y%S,x,c] - mean_c) / std_c in fp64
 *                       (:75-91 stitch + ImageNet normalisation, :29-34 nhwc->nchw .float()); host arrays of P device
 *                       pointers
 *  pk_nhwc_to_nchw_f32  torch.einsum('nhwc->nchw', x).float() of an already normalised fp64/fp32 batch (:29-34)
 *  pk_seg_postprocess   out fp64 [h*p/2, w*p, 3] = clip((unpatchify(patch)[0, bottom half] * std + mean) * 255, 0, 255)
 *                       (:48-52); bin (nullable) fp32 [h*p/2, w*p] = mean_c(out) > 128 (:164-169, video cache)
 *  pk_nearest_blend     dst uint8 [OH,OW,3] = uint8(image * (0.6 * nearest(seg) / 255 + 0.4)) (:93-102)
 *  pk_bilinear_u8       dst uint8 [OH,OW,3] = uint8(int(bilinear(seg))) (painter_inference_segm.py:89-92)        */
int pk_stitch_normalize(const void* const* top, const int* top_dtype, const void* const* bottom,
                        const int* bottom_dtype, float* out, int P, int S, void* stream);
int pk_nhwc_to_nchw_f32(const void* in, int in_is_f64, float* out, int n, int H, int W, void* stream);
int pk_seg_postprocess(const float* patch, double* out, float* bin_or_null, int h, int w, int p, void* stream);
int pk_nearest_blend(const double* seg, int SH, int SW, const uint8_t* image, uint8_t* dst, int OH, int OW,
                     void* stream);
int pk_bilinear_u8(const double* seg, int SH, int SW, uint8_t* dst, int OH, int OW, void* stream);

/* ------------------------------------------------------------------------------------------------
 * fp32-accurate forward mode (north star: within 1e-5 of the reference's fp32 forward, the way
 * seggpt_engine.run_one_image calls the model, seggpt_engine.py:47).  Every fp32 GEMM operand is split into three
 * bf16 terms (h, m, l) and the six significant cross products are evaluated by ONE pk_gemm_bf16 call over operands
 * concatenated along K: A' = [l|m|h|m|h|h], B' = [h|m|l|h|m|h] (K' = 6K, fp32 accumulation in TMEM).
 *  pk_split3                 out bf16 [M, 6K] from x fp32 [M, K] (side_b: 0 = A-side, 1 = B-side order); gelu != 0
 *                            applies the exact erf GELU (timm Mlp act, models_painter.py:201) first
 *  pk_split3_heads           q / k / v of qkv fp32 [B*N, 3C] -> per-(b, head) operands of the attention GEMMs
 *                            (which: 0 q [B*heads, N, 384]; 1 k [B*heads, Npad, 384]; 2 v [B*heads, 6*Npad, 64])
 *  pk_softmax_relpos_split3  P' = split(softmax(scale * S + rel_h + rel_w)) (models_painter.py:80-86,
 *                            vitdet_utils.py:113-123) from S fp32 [BH, N, Npad], Gh = q.T_h^T, Gw = q.T_w^T
 *  pk_im2col_patch_split3    PatchEmbed im2col of imgs and tgts (vitdet_utils.py:178-186) as split A operand
 *  pk_dec_im2col_split3      pixel shuffle + 3x3 im2col of decoder_embed's output (models_painter.py:424-430)
 *  pk_head_f32               LayerNorm2D + exact GELU + conv1x1 + masked loss terms + patchify, fp32, from the fp32
 *                            conv3x3 output [B*H*W, 64]; num accumulates in fp64 (num_zeroed) and is emitted as fp32  */
int pk_split3(const float* x, int ldx, void* out_bf16, int M, int K, int side_b, int gelu, void* stream);
int pk_split3_heads(const float* qkv, void* out_bf16, int B, int heads, int N, int Npad, int which, void* stream);
int pk_softmax_relpos_split3(const float* S, const float* Gh, int ldgh, const float* Gw, int ldgw, void* P_bf16,
                             int BH, int N, int Npad, int h, int w, float scale, void* stream);
int pk_im2col_patch_split3(const float* imgs, const float* tgts, void* out_bf16, int B, int Cin, int H, int W, int p,
                           void* stream);
int pk_dec_im2col_split3(const float* D, void* out_bf16, int B, int h, int w, int p, int dd, void* stream);
int pk_head_f32(const float* c1, const float* head_params, const float* tgts, const uint8_t* mask, int maskB,
                const float* valid, float* patch, double* num_zeroed, float* num_out, int B, int H, int W, int p,
                int loss_kind, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Training data path, per-sample device work (SURVEY §8 f.4).
 *  pk_block_masks  BEiT block masks, one warp per sample: Painter/util/masking_generator.py:15-93 (blocks of random
 *                  area / log-uniform aspect ratio until num_masking cells are covered, then an exact-count fix-up) and
 *                  the half-mask alternative of Painter/data/pairdataset.py:149,183-186.  out int32 [B, H, W].
 *  pk_valid_maps   the per-task loss-weight maps of pairdataset.py:154-181.  rule[b]: 0 all ones; 1 valid[t < thr] = 0
 *                  (depth / semantic / panoptic-semantic); 2 valid[t > thr] = 10 and all 0 when fewer than 300
 *                  foreground values (pose); 3 all 0 when fewer than 300 foreground values (panoptic instances).
 *                  thr: fp32 [B, 3] normalised thresholds; fg_zeroed: int32 [B] scratch.                          */
int pk_block_masks(int* out, int B, int H, int W, int num_masking, int min_patches, int max_patches, float log_ar_lo,
                   float log_ar_hi, float half_mask_ratio, unsigned long long seed, void* stream);
int pk_valid_maps(const float* targets, const int* rule_dev, const float* thr_dev, int* fg_zeroed, float* valid, int B,
                  int H, int W, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PAINTER_B200_H */
