/*
 * mvoc_b200.h — C-ABI of the B200-native MVOC composition hot path.
 *
 * Every entry point takes raw device pointers, explicit shapes/strides and a
 * cudaStream_t (passed as void*).  No call allocates, synchronises or falls
 * back to another implementation: an unsupported shape/dtype returns a
 * negative error code and the text is available from mvoc_last_error().
 * sm_100a only.
 *
 * Threading / devices: the library is built for one process per GPU (the deployment model of this repo).
 * Calls may come from any host thread but not concurrently; launches go to the current device, and the
 * one-time per-kernel attributes (dynamic shared-memory size) are set for the device of the first call, so
 * a process must stay on one device.  mvoc_last_error() is thread-local.
 *
 * Each function cites the reference interface it replaces (paths relative to
 * the SobeyMIL/MVOC tree).  The reference is Python on diffusers; the
 * binding a maintainer would add is a ctypes stub — see INTEGRATION.md.
 *
 * Batch-slot convention (i2vgen-xl/pipelines/pipeline_i2vgen_xl.py:1675-1677):
 *   slot 0 = background, slots 1..n_obj = objects, slot n_obj+1 = uncond
 *   composite, slot n_obj+2 = cond composite.  n_branches = n_obj + 3.
 */
#ifndef MVOC_B200_H
#define MVOC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MVOC_MAX_OBJECTS 8

/* return codes */
#define MVOC_OK 0
#define MVOC_ERR_INVALID_ARG (-1)
#define MVOC_ERR_UNSUPPORTED (-2)
#define MVOC_ERR_CUDA (-3)
#define MVOC_ERR_DRIVER (-4)

/* storage dtypes */
#define MVOC_BF16 0
#define MVOC_F16 1
#define MVOC_F32 2

/* mask kinds for the blends */
#define MVOC_MASK_U8 0  /* binary select, bit exact  */
#define MVOC_MASK_F32 1 /* soft mask, fp32 lerp, rounded once */

/* modes of mvoc_attn_inject_fwd */
#define MVOC_INJECT_SPATIAL 0  /* attention over the pixels of each (branch, frame) */
#define MVOC_INJECT_TEMPORAL 1 /* attention over the frames of each (branch, pixel) */

const char* mvoc_version(void);
const char* mvoc_last_error(void);
/* 0 if `device` is compute capability 10.x, MVOC_ERR_UNSUPPORTED otherwise. */
int mvoc_device_check(int device);

/*
 * Dense non-causal attention forward, O = softmax(Q K^T * scale) V.
 * Replaces F.scaled_dot_product_attention at i2vgen-xl/pnp_utils.py:684-686
 * (injected spatial attn1) and the same call inside diffusers'
 * AttnProcessor2_0 for every spatial self-attention and cross-attention
 * (reached through attention_forward, i2vgen-xl/pnp_utils.py:348-385).
 *
 * q,o: [B, Nq, H, D]   k,v: [B, Nk, H, D]   D innermost and contiguous, D == 64.
 * Strides are in ELEMENTS for (batch, token, head).  Tensor-core path
 * (tcgen05.mma, accumulators in TMEM, operands staged by TMA); bf16 or fp16 (P is rounded to the storage type).
 * Requirements: base pointers 16-byte aligned, strides non-negative multiples of 8, and positive along every
 * dimension of extent > 1 (q, k and v are read through TMA, which cannot broadcast: a zero stride there returns
 * MVOC_ERR_UNSUPPORTED).
 * variant: 0 = default (currently 4).  1, 2 = all exp2 on the MUFU; 3 / 4 / 5 = 2 / 3 / 4 of every
 *          8 exp2 pairs evaluated by a degree-3 polynomial on the FMA pipe.  Same results up to the exp2
 *          approximation (<= 1e-4 relative, below the 16-bit rounding of P); the tests run all of them.
 */
int mvoc_attn_fwd(const void* q, const void* k, const void* v, void* o,
                  int B, int H, int Nq, int Nk, int D,
                  int64_t q_sb, int64_t q_sn, int64_t q_sh,
                  int64_t k_sb, int64_t k_sn, int64_t k_sh,
                  int64_t v_sb, int64_t v_sn, int64_t v_sh,
                  int64_t o_sb, int64_t o_sn, int64_t o_sh,
                  float scale, int dtype, int variant, void* stream);

/*
 * Attention of a PAIR of branches that share Q and K: O[b] = softmax(Q[b] K[b]^T scale) V[b] and
 * O[b + pair_batches] = (the same softmax) V[b + pair_batches], b < B.  One softmax, two P.V products per CTA —
 * half the exponentials, which are what bounds a head_dim-64 attention on this chip.
 * This is the structure MVOC creates and the reference ignores: ModifiedSpaAttnProcessor writes the SAME blended
 * Q', K' into the uncond and the cond composite chunk (i2vgen-xl/pnp_utils.py:664-668) and then runs SDPA on
 * both (:684).  q, k: [B, N, H, D]; v, o: [B + pair_batches, N, H, D]; other arguments and the stride
 * requirements as mvoc_attn_fwd.  pair_batches >= B (MVOC_ERR_INVALID_ARG otherwise): with fewer, output batch
 * b + pair_batches < B would be written by two CTAs.  Output batches in [B, pair_batches) are not written.
 */
int mvoc_attn_pair_fwd(const void* q, const void* k, const void* v, void* o,
                       int B, int H, int Nq, int Nk, int D,
                       int64_t q_sb, int64_t q_sn, int64_t q_sh,
                       int64_t k_sb, int64_t k_sn, int64_t k_sh,
                       int64_t v_sb, int64_t v_sn, int64_t v_sh,
                       int64_t o_sb, int64_t o_sn, int64_t o_sh,
                       int pair_batches, float scale, int dtype, int variant, void* stream);

/*
 * Causal attention forward at head_dim 64: O[r] = softmax(Q[r] K[0..r]^T * scale) V[0..r] for query row r.
 * Replaces the self-attention of transformers' CLIPAttention with the causal mask in the CLIP text tower (16 heads of
 * 64 over 77 tokens), reached from I2VGenXLPipeline.encode_prompt (diffusers 0.27.2) for the prompt, the negative
 * prompt and the inversion prompt (no attention mask is passed: the pad positions are encoded too).
 *
 * Arguments and strides as mvoc_attn_fwd: q,o [B, Nq, H, D], k,v [B, Nk, H, D], D == 64 innermost and contiguous,
 * strides in ELEMENTS for (batch, token, head), so q/k/v may be the three column slices of one fused QKV projection
 * output [B*N, 3*H*64].  Nq == Nk (top-left and bottom-right alignment are then the same and no row is empty;
 * MVOC_ERR_UNSUPPORTED otherwise), any N >= 1.  Key blocks above the diagonal are skipped, so the work is about half
 * that of mvoc_attn_fwd at long N.  Tensor-core path; bf16 or fp16 (P is rounded to the storage type); the exp2 split
 * of mvoc_attn_fwd's default variant.  Requirements and error codes as mvoc_attn_fwd: base pointers 16-byte aligned,
 * strides non-negative multiples of 8, and positive along every dimension of extent > 1 (MVOC_ERR_UNSUPPORTED).
 */
int mvoc_attn_causal_fwd(const void* q, const void* k, const void* v, void* o,
                         int B, int H, int Nq, int Nk, int D,
                         int64_t q_sb, int64_t q_sn, int64_t q_sh,
                         int64_t k_sb, int64_t k_sn, int64_t k_sh,
                         int64_t v_sb, int64_t v_sn, int64_t v_sh,
                         int64_t o_sb, int64_t o_sn, int64_t o_sh,
                         float scale, int dtype, void* stream);

/*
 * Diagnostics: mvoc_attn_fwd (pair_batches == 0) or mvoc_attn_pair_fwd with clock64() time stamps of CTA (0,0,0)
 * written to trace[key block * 8 + event] (device memory, int64): 0 softmax starts waiting for S, 1 S ready,
 * 2 row maximum known, 3 exponentials done, 4 P buffer free, 5 P published; 6 Q K^T issued, 7 P V issued.
 * strides12: the twelve element strides of mvoc_attn_fwd in order.  tools/attn_trace.py prints the phase times.
 */
int mvoc_attn_fwd_trace(const void* q, const void* k, const void* v, void* o, int B, int H, int Nq, int Nk, int D,
                        const int64_t* strides12, int pair_batches, float scale, int dtype, int variant,
                        long long* trace, void* stream);

/*
 * Single-head attention of width 512, O = softmax(Q K^T * scale) V.
 * Replaces the mid-block Attention of the AutoencoderKL decoder (one head over the 512 channels of the latent-
 * resolution map, diffusers' Attention with group_norm and residual_connection), reached from decode_latents,
 * i2vgen-xl/pipelines/pipeline_i2vgen_xl.py:771-791.
 *
 * q,k,v,o: [B, N, D], D == 512 innermost and contiguous; strides in ELEMENTS for (batch, token), so q/k/v may be
 * the three column slices of one fused QKV projection output [B*N, 1536].  Any N >= 1 (no multiple of 128 needed).
 * Tensor-core path (tcgen05.mma, accumulators in TMEM, operands staged by TMA); bf16 or fp16 (P is rounded to the
 * storage type).  Requirements: base pointers 16-byte aligned, strides non-negative multiples of 8, and positive
 * along every dimension of extent > 1 (a zero q / k / v stride there returns MVOC_ERR_UNSUPPORTED).
 */
int mvoc_attn_d512_fwd(const void* q, const void* k, const void* v, void* o, int B, int N, int D,
                       int64_t q_sb, int64_t q_sn, int64_t k_sb, int64_t k_sn,
                       int64_t v_sb, int64_t v_sn, int64_t o_sb, int64_t o_sn,
                       float scale, int dtype, void* stream);

/*
 * Dense non-causal attention forward at head_dim 80, O = softmax(Q K^T * scale) V.
 * Replaces the self-attention of transformers' CLIPAttention in the CLIP image tower (ViT-H/14: 16 heads of 80 over
 * 257 tokens), reached from I2VGenXLPipeline._encode_image, i2vgen-xl/pipelines/pipeline_i2vgen_xl.py:1391-1541
 * (the per-branch, per-frame image embeddings).
 *
 * Arguments and strides as mvoc_attn_fwd: q,o [B, Nq, H, D], k,v [B, Nk, H, D], D == 80 innermost and contiguous,
 * strides in ELEMENTS for (batch, token, head), so q/k/v may be the three column slices of one fused QKV projection
 * output [B*N, 3*H*80].  Any Nq, Nk >= 1.  Tensor-core path (tcgen05.mma, accumulators in TMEM, operands staged by
 * TMA); bf16 or fp16 (P is rounded to the storage type).  Requirements: base pointers 16-byte aligned, strides
 * non-negative multiples of 8, and positive along every dimension of extent > 1 (MVOC_ERR_UNSUPPORTED otherwise).
 */
int mvoc_attn_d80_fwd(const void* q, const void* k, const void* v, void* o,
                      int B, int H, int Nq, int Nk, int D,
                      int64_t q_sb, int64_t q_sn, int64_t q_sh,
                      int64_t k_sb, int64_t k_sn, int64_t k_sh,
                      int64_t v_sb, int64_t v_sn, int64_t v_sh,
                      int64_t o_sb, int64_t o_sn, int64_t o_sh,
                      float scale, int dtype, void* stream);

/*
 * Short-sequence attention (tokens = frames), one warp per (pixel, head).
 * Replaces F.scaled_dot_product_attention at i2vgen-xl/pnp_utils.py:862-864
 * (injected temporal attn1) and the stock processor on the temporal attn2,
 * transformer_in (i2vgen-xl/pnp_utils.py:170-220 drives them).
 *
 * q,k,v,o: [P, T, H, D], D == 64 contiguous, 1 <= T <= 32 (16 and 32 are the unmasked fast paths);
 * strides in elements for (problem, token, head).  HBM-bound; bf16 only.
 */
int mvoc_attn_temporal_fwd(const void* q, const void* k, const void* v, void* o,
                           int64_t P, int T, int H, int D,
                           int64_t q_sp, int64_t q_st, int64_t q_sh,
                           int64_t k_sp, int64_t k_st, int64_t k_sh,
                           int64_t v_sp, int64_t v_st, int64_t v_sh,
                           int64_t o_sp, int64_t o_st, int64_t o_sh,
                           float scale, int dtype, void* stream);

/*
 * Same kernel with a two-level problem index (problem = outer * P_inner + inner), so that temporal
 * attention reads channels-last activations [B, T, HW, C] in place — problem (b, pixel) starts at
 * b*s_outer + pixel*s_inner and its frames are s_token apart — and the [(b t), c, h, w] ->
 * [(b h w), t, c] permutes of i2vgen-xl/pnp_utils.py:189 and :207-213 are never materialised.
 * strides16: element strides (outer, inner, token, head) for q, k, v, o in that order.
 */
int mvoc_attn_temporal_strided_fwd(const void* q, const void* k, const void* v, void* o,
                                   int64_t P_outer, int64_t P_inner, int T, int H, int D,
                                   const int64_t* strides16, float scale, int dtype, void* stream);

/*
 * Q/K mask-blend injection, in place.
 * Replaces i2vgen-xl/pnp_utils.py:628-672 (spatial, binary mask) and
 * :782-850 (temporal, float mask).
 *
 * x0, x1 (x1 may be NULL): [n_branches, tokens, C] contiguous — Q and K of one
 * layer viewed with the branch slot outermost (spatial: tokens = T*h*w in
 * (frame, pixel) order; temporal: tokens = h*w*T in (pixel, frame) order).
 * mask: [n_obj, tokens] in the SAME token order, u8 (MVOC_MASK_U8: nonzero
 * selects the object) or f32 (MVOC_MASK_F32: base*(1-m)+obj*m in fp32).
 * base_slot: n_obj+2 (cond; inject_background False) or 0 (background).
 * Result is written to slots n_obj+1 and n_obj+2.  C % 8 == 0.
 */
int mvoc_qk_blend(void* x0, void* x1, int n_obj, int64_t tokens, int C,
                  const void* mask, int mask_kind, int base_slot,
                  int dtype, void* stream);
/* Same with a row stride `ld` (elements, >= C): x0 / x1 may be column slices of a wider row-major buffer, e.g. the
 * Q and K thirds of a fused QKV projection.  single != 0 writes the blend to slot n_obj+1 only. */
int mvoc_qk_blend_strided(void* x0, void* x1, int n_obj, int64_t tokens, int C, int64_t ld,
                          const void* mask, int mask_kind, int base_slot, int single,
                          int dtype, void* stream);

/*
 * Injected self-attention in one call: the Q/K mask blend followed by the attention of ALL branches on `stream`.
 * Replaces what ModifiedSpaAttnProcessor.__call__ does between the q/k/v projections and to_out
 * (i2vgen-xl/pnp_utils.py:624-686; mode MVOC_INJECT_SPATIAL, binary mask) and what
 * ModifiedTmpAttnProcessor.__call__ does there (:778-864; mode MVOC_INJECT_TEMPORAL, float mask).
 *
 * q, k, v, o: [(n_obj+3)*frames, pixels, H*D] with row strides ld_q / ld_k / ld_v / ld_o (elements; rows of a
 * branch-major, frame-major, pixel-minor token list) — q, k, v may be the three column slices of ONE fused QKV
 * projection output, so the injected layers keep the single projection GEMM.  Rows are in (branch, frame, pixel)
 * order in BOTH modes (the temporal mode reads the frames of a pixel through strides; the [(b h w), T, C] permute
 * of :189 is not needed).  q and k are modified in place (slot n_obj+1, and slot n_obj+2 unless share_p).
 * mask: [n_obj, frames*pixels] in (frame, pixel) order, kind as for mvoc_qk_blend.
 * share_p (spatial mode): the uncond and cond composite branches receive the same blended Q', K' (:664-668), so
 * their attention runs as ONE softmax with two P.V products (mvoc_attn_pair_fwd) and the blend writes one copy.
 * Restrictions of the attention kernels apply (D == 64, bf16 / fp16; temporal: frames <= 32, share_p == 0).
 */
int mvoc_attn_inject_fwd(void* q, void* k, const void* v, void* o,
                         int64_t ld_q, int64_t ld_k, int64_t ld_v, int64_t ld_o,
                         int n_obj, int frames, int64_t pixels, int H, int D,
                         const void* mask, int mask_kind, int base_slot, int mode,
                         int share_p, float scale, int dtype, int variant, void* stream);

/*
 * Hidden-state mask-blend after resnet conv2 / temporal conv / conv_out.
 * Replaces i2vgen-xl/pnp_utils.py:970-1004, :1059-1082, :1114-1146.
 *
 * x: [n_branches*T, C, HW] contiguous (NCHW, frames fastest inside a slot),
 * mask: [n_obj, T, HW] u8 (binary at full latent resolution).  base = slot 0
 * always; result written to slots n_obj+1 and n_obj+2 in place.  Bit exact.
 */
int mvoc_feature_blend(void* x, int n_obj, int T, int C, int64_t HW,
                       const void* mask, int dtype, void* stream);

/*
 * GroupNorm (+ optional SiLU) over [N, C, S] with G groups; statistics are
 * shared by `frames_per_stat` consecutive n (1 = spatial GroupNorm on
 * [B*T,C,H,W]; T = the 5-D GroupNorm on [B,C,T,H,W] stored frame-major).
 * Replaces norm1/norm2 + nonlinearity at i2vgen-xl/pnp_utils.py:909-910,
 * :953-965, the GN→SiLU heads of TemporalConvLayer.conv1..4 (:1048-1051),
 * Transformer2DModel.norm (:430), TransformerTemporalModel.norm (:185-188) and
 * conv_norm_out + conv_act (pipelines/pipeline_i2vgen_xl.py:351-352).
 *
 * gamma/beta: [C] in `dtype`.  y may alias x.  workspace: at least
 * mvoc_groupnorm_workspace_bytes(N, G) bytes of device memory.
 */
int64_t mvoc_groupnorm_workspace_bytes(int64_t N, int G);
int mvoc_groupnorm_silu(const void* x, void* y, const void* gamma, const void* beta,
                        int64_t N, int C, int64_t S, int G, int frames_per_stat,
                        float eps, int silu, int dtype, void* workspace, void* stream);

/*
 * Channels-last GroupNorm (+SiLU, + fused per-(n, channel) add) on [N, S, C]: the same reference call
 * sites as mvoc_groupnorm_silu, for the NHWC host path; `add` [N, C] (nullable) fuses the resnet's
 * `hidden_states + temb` (i2vgen-xl/pnp_utils.py:941-953) into the normalisation.
 * Three launches so that the statistics of pixel shards can be merged across GPUs in between:
 *   stats    -> partial [N, G, chunks] float2 (mean, M2); chunks from mvoc_groupnorm_nhwc_geometry
 *   finalize -> stat [N / frames_per_stat, G] float2 (mean, rstd); merges `sets` partial arrays laid out
 *               [sets, N, G, chunks] with element counts counts[sets, chunks] (float)
 *   apply    -> y = silu?((x + add - mean) * rstd * gamma + beta); y may alias x
 */
int64_t mvoc_groupnorm_nhwc_partial_count(int64_t N, int G);
int mvoc_groupnorm_nhwc_geometry(int64_t S, int C, int dtype, int* chunks, int64_t* tokens_per_chunk);
int mvoc_groupnorm_nhwc_stats(const void* x, const void* add, void* partial, int64_t N, int64_t S, int C,
                              int G, int dtype, void* stream);
int mvoc_groupnorm_nhwc_finalize(const void* partial, const void* counts, void* stat, int64_t N, int G,
                                 int chunks, int frames_per_stat, int sets, float eps, void* stream);
int mvoc_groupnorm_nhwc_apply(const void* x, void* y, const void* gamma, const void* beta, const void* add,
                              const void* stat, int64_t N, int64_t S, int C, int G, int frames_per_stat,
                              int silu, int dtype, void* stream);

/*
 * Row-wise LayerNorm over [M, C] (affine, eps): norm1 / norm2 / norm3 of BasicTransformerBlock
 * (i2vgen-xl/pnp_utils.py:249-250, :295-296, :322).  One warp per row, one read + one write.  C % 8 == 0,
 * C <= 2048.  y may alias x.
 */
int mvoc_layernorm(const void* x, void* y, const void* gamma, const void* beta, int64_t M, int C,
                   float eps, int dtype, void* stream);

/*
 * Fused GEGLU gate: y[m, j] = x[m, j] * gelu(x[m, F + j]) (exact erf GELU), x [M, 2F] -> y [M, F].
 * Replaces the chunk + F.gelu + multiply of diffusers' GEGLU inside `model.ff`
 * (i2vgen-xl/pnp_utils.py:335).  F % 8 == 0.
 */
int mvoc_geglu(const void* x, void* y, int64_t M, int F, int dtype, void* stream);

/*
 * Nearest-neighbour 2x upsampling of a channels-last activation x [N, H, W, C] -> y [N, 2H, 2W, C]: the
 * F.interpolate(scale_factor=2.0, mode="nearest") of diffusers' Upsample2D in the up blocks
 * (i2vgen-xl/pipelines/pipeline_i2vgen_xl.py:318-350 -> UpBlock3D / CrossAttnUpBlock3D upsamplers).  C % 8 == 0.
 */
int mvoc_upsample_nearest2x_nhwc(const void* x, void* y, int64_t N, int H, int W, int C, int dtype, void* stream);

/*
 * Channel concatenation of two channels-last activations a [rows, CA], b [rows, CB] -> y [rows, CA + CB]: the
 * skip-connection torch.cat before every resnet of the up blocks (diffusers UNet3D up blocks, reached from
 * i2vgen-xl/pipelines/pipeline_i2vgen_xl.py:318-350).  A copy, bit-identical to torch.cat.  CA, CB % 8 == 0.
 */
int mvoc_concat_lastdim(const void* a, const void* b, void* y, int64_t rows, int CA, int CB, int dtype, void* stream);

/*
 * ---- dense work on tcgen05 tensor cores (csrc/gemm_tc.cu) ------------------------------------------------
 * One persistent implicit-GEMM kernel: 128-row activation tiles are TMA boxes of the channels-last tensor
 * (shifted per filter tap, zero-filled outside = the padding), weights are K-major [tap, Cout, Cin], fp32
 * accumulation in TMEM (two buffers), epilogue fuses bias / residual / GEGLU and leaves through TMA stores.
 * bf16 or fp16 storage (MVOC_BF16 / MVOC_F16); channel counts multiples of 64; pointers 16-byte aligned.
 * variant: bit 0 = run as CTA pairs (tcgen05 cta_group::2, 256-row tiles); bits 8..16 = tile width override
 * (256 / 192 / 160 / 128 / 64; 0 = widest that divides Cout).  Outputs may not alias inputs.
 */

/*
 * 3x3 convolution, stride 1, padding 1, channels-last: out[N,H,W,Cout] = conv(x[N,H,W,Cin], w) + bias
 * (+ x2[N,H,W,Cin2] . w2[Cout,Cin2], the resnet's 1x1 shortcut conv accumulated in the same tile)
 * (+ residual[N,H,W,Cout]).  w_taps: [9, Cout, Cin] (tap = kh*3+kw), i.e. conv.weight.permute(2,3,0,1).
 * Replaces conv1 / conv2 / conv_shortcut + the skip add of the resnet closure, i2vgen-xl/pnp_utils.py:939,
 * :968, :1011-1018, and the same calls inside diffusers' stock ResnetBlock2D / Upsample2D.
 */
/*
 * Host-side tile plan of the GEMM kernel for `rows` output rows x N output columns on a chip of `sms` SMs (no device
 * call; `variant` as in the compute entries): the column-tile width, whether CTA pairs are used, and the width of
 * the narrower last column tile (0 = the width divides N).  What the compute entries choose internally.
 */
int mvoc_gemm_plan(int64_t rows, int64_t N, int geglu, int variant, int sms, int* tile_cols, int* cta_pair,
                   int* tail_cols);

int mvoc_conv3x3_nhwc(const void* x, const void* w_taps, const void* bias, const void* residual,
                      const void* x2, const void* w2, int Cin2, void* out,
                      int N, int H, int W, int Cin, int Cout, int dtype, int variant, void* stream);

/*
 * 3x3 convolution, stride 2, channels-last: out[N,Ho,Wo,Cout] = conv(x[N,H,W,Cin], w) + bias, with pad_begin zero
 * rows / columns before and pad_end after the input, each 0 or 1: Ho = (H + pad_begin + pad_end - 3) / 2 + 1, Wo
 * likewise.  w_taps: [9, Cout, Cin] as for mvoc_conv3x3_nhwc; bias optional.  Replaces the Conv2d of the VAE
 * encoder's Downsample2D, which pads (0, 1, 0, 1) and runs a stride-2 conv without padding (pads (0, 1);
 * i2vgen-xl/pipelines/pipeline_i2vgen_xl.py:893-920 and :860-890 reach it through vae.encode).  torch's
 * padding=1, as in the UNet's downsamplers, is pads (1, 1).  Cin, Cout multiples of 64; checked before any CUDA call.
 */
int mvoc_conv3x3_s2_nhwc(const void* x, const void* w_taps, const void* bias, void* out,
                         int N, int H, int W, int Cin, int Cout, int pad_begin, int pad_end,
                         int dtype, int variant, void* stream);

/*
 * Temporal convolution Conv3d(kernel (3,1,1), padding (1,0,0)) on frame-major channels-last rows:
 * x [B, T, S, Cin] -> out [B, T, S, Cout] (+ bias, + residual), w_taps [3, Cout, Cin] (tap = frame offset + 1).
 * Replaces the Conv3d of TemporalConvLayer.conv1..4 and the identity add, i2vgen-xl/pnp_utils.py:1048-1053;
 * the [(b t) c h w] <-> [b c t h w] permutes of :1044-1046, :1055-1057 are never materialised.
 */
int mvoc_temporal_conv3(const void* x, const void* w_taps, const void* bias, const void* residual, void* out,
                        int B, int T, int64_t S, int Cin, int Cout, int dtype, int variant, void* stream);

/*
 * Linear / 1x1 conv: out[M, N] = x[M, K] . w[N, K]^T (+ bias[N]) (+ residual[M, N]); row strides ldx / ldr /
 * ldo in elements (multiples of 8).  Replaces to_q / to_k / to_v / to_out[0] (i2vgen-xl/pnp_utils.py:604-612,
 * :692 — bias + the block's residual add :283/:315 in the epilogue), proj_in / proj_out (:191, :206, :432,
 * :503-508), ff.net[2] (:335-342) and the K/V projections of the cross-attention.
 */
int mvoc_linear(const void* x, const void* w, const void* bias, const void* residual, void* out,
                int64_t M, int K, int N, int64_t ldx, int64_t ldr, int64_t ldo,
                int dtype, int variant, void* stream);

/*
 * GEGLU projection with the gate in the epilogue: out[M, F] = (x . w[:F]^T + b[:F]) * gelu(x . w[F:]^T + b[F:])
 * (exact erf GELU); w [2F, K], bias [2F].  The [M, 2F] intermediate of diffusers' GEGLU
 * (i2vgen-xl/pnp_utils.py:335: proj, chunk, gelu, multiply) never reaches HBM.  F % 64 == 0.
 */
int mvoc_linear_geglu(const void* x, const void* w, const void* bias, void* out, int64_t M, int K, int F,
                      int dtype, int variant, void* stream);

/*
 * Linear with the exact (erf) GELU in the epilogue: out[M, N] = gelu(x[M, K] . w[N, K]^T + bias[N]); row strides
 * ldx / ldo in elements (multiples of 8); bias may be null.  The erf GELU is the GEGLU epilogue's.  Replaces mlp.fc1 +
 * activation_fn ("gelu") of every CLIPEncoderLayer of the CLIP image tower (transformers' CLIPMLP), reached from
 * I2VGenXLPipeline._encode_image, i2vgen-xl/pipelines/pipeline_i2vgen_xl.py:1391-1541.  K, N multiples of 64.
 */
int mvoc_linear_gelu(const void* x, const void* w, const void* bias, void* out, int64_t M, int K, int N,
                     int64_t ldx, int64_t ldo, int dtype, int variant, void* stream);

/*
 * ---- frame-shard <-> pixel-shard exchange over NVLink peer memory (csrc/exchange.cu) ----------------------
 * The multi-GPU partition keeps T/P frames of every branch on each rank; the temporal operators
 * (TemporalConvLayer, the temporal transformers: i2vgen-xl/pnp_utils.py:1042-1057, :170-220) need all frames of a
 * pixel, so the activation is re-laid out around them — what the single-GPU reference expresses as the permutes at
 * :189, :207-213, :1044-1046, :1055-1057.  Each rank owns an ARENA (cudaMalloc + CUDA IPC handle, opened by every
 * peer); ranks allocate from their arenas in lockstep, so a destination buffer has the same offset everywhere.
 * A put kernel reads the local shard once and stores every 16-byte vector at its final position in the destination
 * rank's buffer (pack + transfer + unpack in one pass), then publishes a per-site epoch in every peer's flag row;
 * mvoc_exchange_wait spins until all sources have published.  Epochs live in device memory: CUDA-graph safe.
 * `site`: index of the exchange within one forward (each site owns a flag row), < mvoc_exchange_max_sites().
 * `site | MVOC_EXCHANGE_WAIT_FUSED`: the put kernel itself also waits for the peers (its last CTA spins on this
 * rank's flag row after publishing), so that no separate mvoc_exchange_wait launch is needed for the site.
 * peer_bases: HOST array of `world` device pointers (the arenas as mapped into THIS process; entry `rank` is the
 * local arena).  dst_offset: byte offset of the destination buffer inside every arena (>= header bytes).
 */
#define MVOC_EXCHANGE_WAIT_FUSED (1 << 30)
int64_t mvoc_exchange_header_bytes(void);
int mvoc_exchange_max_sites(void);
int mvoc_exchange_arena_create(int64_t bytes, void** base, void* ipc_handle64);
int mvoc_exchange_arena_open(const void* ipc_handle64, void** peer_base);
int mvoc_exchange_arena_close(void* peer_base);
int mvoc_exchange_arena_destroy(void* base);
/* x [b, frames_local, S, C] (this rank's frames) -> every rank d: [b, frames_local * world, S / world, C] */
int mvoc_exchange_to_pixel_shards(const void* x, void* const* peer_bases, int64_t dst_offset, int rank, int world,
                                  int b, int frames_local, int64_t S, int C, int dtype, int site, void* stream);
/* y [b, frames_total, S_local, C] (this rank's pixels) -> every rank d: [b, frames_total / world, S_local * world, C] */
int mvoc_exchange_to_frame_shards(const void* y, void* const* peer_bases, int64_t dst_offset, int rank, int world,
                                  int b, int frames_total, int64_t S_local, int C, int dtype, int site, void* stream);
/* `bytes` of src -> slot `rank` of every rank's [world, bytes] buffer (GroupNorm partial statistics of pixel shards) */
int mvoc_exchange_allgather(const void* src, int64_t bytes, void* const* peer_bases, int64_t dst_offset, int rank,
                            int world, int site, void* stream);
int mvoc_exchange_wait(const void* my_base, int world, int site, void* stream);

/*
 * Latent compositing ("noise fusion") fused with the UNet input concat.
 * Replaces pipelines/pipeline_i2vgen_xl.py:1644-1663 and the torch.cat at
 * :1675-1677.
 *
 * z [E] (in/out, E = 4*T*h*w laid out [4,T,h,w]), bg [E], objs [n_obj,E],
 * mask [n_obj, T*h*w] f32 (broadcast over the 4 channels).
 * do_fusion: z = r*z + (1-r)*bg; then per object
 *   z = z*(1-M) + obj*M                       (obj_noise_fusion == 0)
 *   z = z*(1-M) + r*z*M + (1-r)*obj*M         (obj_noise_fusion != 0)
 * unet_in (nullable): [n_obj+3, E] receives [bg, objs..., z, z] in
 * `in_dtype`; latents themselves are `lat_dtype`.
 */
int mvoc_latent_composite(void* z, const void* bg, const void* objs, const void* mask,
                          void* unet_in, int n_obj, int64_t E, int64_t THW,
                          float ratio, int do_fusion, int obj_noise_fusion,
                          int lat_dtype, int in_dtype, void* stream);

/*
 * Classifier-free guidance + v-prediction DDIM update (eta = 0).
 * Replaces pipelines/pipeline_i2vgen_xl.py:1713-1731 and diffusers
 * DDIMScheduler.step.   v = u + g*(c-u);
 *   x0 = sqrt(a_t) x - sqrt(1-a_t) v;  eps = sqrt(a_t) v + sqrt(1-a_t) x;
 *   x_prev = sqrt(a_prev) x0 + sqrt(1-a_prev) eps.
 * pred_cond may be NULL (no guidance: v = pred_uncond).
 */
int mvoc_cfg_ddim_step(const void* pred_uncond, const void* pred_cond, void* x,
                       int64_t E, float guidance, double alpha_t, double alpha_prev,
                       int pred_dtype, int lat_dtype, void* stream);

/*
 * Inverse DDIM step (pipelines/pipeline_i2vgen_xl.py:1967-1984 and diffusers
 * DDIMInverseScheduler.step): same algebra, from level alpha_src to alpha_dst.
 */
int mvoc_ddim_inverse_step(const void* pred_uncond, const void* pred_cond, void* x,
                           int64_t E, float guidance, double alpha_src, double alpha_dst,
                           int pred_dtype, int lat_dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MVOC_B200_H */
