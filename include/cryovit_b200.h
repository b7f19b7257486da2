/*
 * cryovit_b200 C ABI  --  the drop-in boundary of the B200-native CryoVIT hot path.
 *
 * The reference (VivianDLi/CryoVIT) is pure Python and has no FFI of its own; its seams for this path are
 * Python call sites (SURVEY.md 8b, B1-B6).  This header is seam B7: the operator-level C ABI that the
 * Python host mirror (cryovit_b200/vit.py, head.py, extract.py) binds with ctypes, and that any other host
 * (C++, a torch custom op, a napari plugin) can bind the same way.  Each entry point names the reference
 * computation it replaces (file:line under /root/reference/src/cryovit, or the un-vendored upstream
 * facebookresearch/dinov2 cross-checked against transformers' Dinov2WithRegisters, "HF:").
 *
 * Contract for every function:
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless named host_*;
 *   - the caller owns every buffer; nothing is allocated, nothing is freed, no hidden synchronisation;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream);
 *   - returns 0 on success or a negative CVIT_ERR_* code; cvit_last_error() gives the message for the
 *     calling thread.  No exceptions cross the boundary;
 *   - re-entrant per (device, stream).  sm_100a only: there is no CPU or other-architecture fallback.
 *
 * Layout vocabulary: a "slice" is one z-plane of a tomogram; "tokens" are the ViT tokens of one slice
 * (1 cls + R registers + Np patches); a "feature volume" is fp16 (C, D, h, w); the head works on
 * channels-last (D, H, W, C) bf16 volumes ("ndhwc").
 */
#ifndef CRYOVIT_B200_H
#define CRYOVIT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CVIT_OK 0
#define CVIT_ERR_INVALID (-1)
#define CVIT_ERR_CUDA (-2)
#define CVIT_ERR_DRIVER (-3)
#define CVIT_ERR_UNSUPPORTED (-4)

/* Library identity / diagnostics. */
int cvit_abi_version(void);
const char* cvit_last_error(void);
/* Process-wide switch of the GEMM family: 1 (default) = plain-rows GEMMs with 256-wide N tiles run as CTA pairs
 * (tcgen05 cta_group::2, 256 x 256 output tile per TPC), 0 = single-CTA kernel everywhere. Returns the previous
 * value. Exists for A/B measurement only; results are bit-identical in both modes. */
int cvit_set_gemm_pair(int enable);

/* ---------------------------------------------------------------------------------------------------------
 * Slice pre-processing + patchify.
 * Replaces VITDataset._load_tomogram + _dino_transform (datasets/vit_dataset.py:71-123): uint8 -> /255
 * (src_is_u8 != 0) or float32 pass-through, edge-pad H,W to multiples of 16, bicubic x14/16 (A=-0.75,
 * align_corners=False, borders clamped), cut into 14x14 patches.  The reference replicates the single
 * channel three times; here ONE channel is produced (host pre-sums the patch-embed weight over its 3 input
 * channels).  Output: bf16 [D * Np, Kp], column i*14+j for pixel (i,j) of the patch, columns 196..Kp-1 zero;
 * Np = (ceil16(H)*14/16/14) * (ceil16(W)*14/16/14).  Kp is a multiple of 64, >= 196.
 */
int cvit_preproc_patchify(const void* src, int src_is_u8, void* patches_bf16, int64_t D, int64_t H, int64_t W,
                          int64_t Kp, void* stream);

/* The same pre-processing written in the reference's own layout: f32 [D, 3, ceil16(H)*14/16, ceil16(W)*14/16]
 * with three identical channels -- what VITDataset.__getitem__ returns (datasets/vit_dataset.py:90-123). */
int cvit_preproc_resize_f32_3ch(const void* src, int src_is_u8, float* out, int64_t D, int64_t H, int64_t W,
                                void* stream);

/* Patchify for the reference-facing model call forward_features(x: f32[B,3,H',W']) (run/dino_features.py:58;
 * upstream PatchEmbed, HF:42-73).  Output bf16 [B * Np, Kp], column c*196 + i*14 + j, zero padded to Kp
 * (multiple of 64, >= 588). */
int cvit_patchify_f32_3ch(const float* src, void* patches_bf16, int64_t B, int64_t OH, int64_t OW, int64_t Kp,
                          void* stream);

/* The two patchify entry points above with fp32 output rounded to TF32 (nearest, ties away from zero; the 13 low
 * mantissa bits zero): the patch rows of the TF32 patch embedding (cvit_patch_embed_gemm_fmt with
 * CVIT_FMT_OPERANDS_TF32), which keeps the 10-bit-exact pixels the reference embeds in TF32
 * (run/dino_features.py:24, set_float32_matmul_precision("high")) where bf16 would keep 8 bits. */
int cvit_preproc_patchify_tf32(const void* src, int src_is_u8, float* patches, int64_t D, int64_t H, int64_t W,
                               int64_t Kp, void* stream);
int cvit_patchify_f32_3ch_tf32(const float* src, float* patches, int64_t B, int64_t OH, int64_t OW, int64_t Kp,
                               void* stream);

/* Patch-embed GEMM: x[b, first_patch_token + p, :] = patches[b*Np + p, :] @ W^T + pos_bias_table[p, :].
 * Replaces upstream PatchEmbed.proj (conv 14/14 as a GEMM) + the pos-embed add of prepare_tokens_with_masks
 * (HF:61-71,147-173).  W: bf16 [N, K] row-major; table: fp32 [Np, N] = interpolated pos-embed + conv bias;
 * x: fp32 [n_slices * tokens_per_slice, ldx]. */
int cvit_patch_embed_gemm(const void* patches, int64_t lda, const void* W, const float* pos_bias_table, float* x,
                          int64_t ldx, int64_t n_slices, int64_t n_patches, int64_t tokens_per_slice,
                          int64_t first_patch_token, int64_t N, int64_t K, void* stream);
/* The same GEMM by format flags: fmt = 0 (bf16 patches and W, = cvit_patch_embed_gemm) or CVIT_FMT_OPERANDS_TF32
 * (patches and W fp32 holding TF32 values: the reference's TF32 conv, run/dino_features.py:24; lda and K in fp32
 * elements).  Other flags return CVIT_ERR_UNSUPPORTED. */
int cvit_patch_embed_gemm_fmt(const void* patches, int64_t lda, const void* W, const float* pos_bias_table, float* x,
                              int64_t ldx, int64_t n_slices, int64_t n_patches, int64_t tokens_per_slice,
                              int64_t first_patch_token, int64_t N, int64_t K, int fmt, void* stream);

/* x[b, s, :] = special[s, :] for s < S (cls + pos[0], then the register tokens; HF:147-173). */
int cvit_assemble_special_tokens(float* x, const float* special, int64_t B, int64_t T, int64_t C, int64_t S,
                                 void* stream);

/* LayerNorm over the last dim: out_bf16 = (x - mean) * rsqrt(var + eps) * gamma + beta.  Replaces
 * Block.norm1 / norm2 (upstream block.py; HF:370,377).  x fp32 [M, ldx]; C in {384, 768, 1024, 1536}. */
int cvit_layernorm_f32_bf16(const float* x, int64_t ldx, const float* gamma, const float* beta, void* out,
                            int64_t ldo, int64_t M, int64_t C, float eps, void* stream);

/* Same with an IEEE fp16 result: the A operand of the fp16-operand linears below (CVIT_FMT_OPERANDS_F16). */
int cvit_layernorm_f32_f16(const float* x, int64_t ldx, const float* gamma, const float* beta, void* out,
                           int64_t ldo, int64_t M, int64_t C, float eps, void* stream);

/* Same with fp32 output: the final model.norm when the caller wants x_norm_* tensors (HF:477-503) rather than
 * the fused fp16 write-out below. */
int cvit_layernorm_f32_f32(const float* x, int64_t ldx, const float* gamma, const float* beta, float* out,
                           int64_t ldo, int64_t M, int64_t C, float eps, void* stream);

/* Same with fp32 output rounded to TF32 (nearest, ties away from zero; the 13 low mantissa bits zero): Block.norm1 /
 * norm2 as the A operand of the TF32 linears (CVIT_FMT_OPERANDS_TF32), which the reference runs in TF32
 * (run/dino_features.py:24). */
int cvit_layernorm_f32_tf32(const float* x, int64_t ldx, const float* gamma, const float* beta, float* out,
                            int64_t ldo, int64_t M, int64_t C, float eps, void* stream);

/* out_bf16[M, N] = A[M, K] @ W[N, K]^T + bias, optionally followed by exact-erf GELU.  Replaces attn.qkv
 * (HF:219-221) and, with gelu=1, Mlp.fc1 + GELU of ViT-S/B/L and the head's 1x1x1 Conv3d + GELU
 * (models/cryovit.py:19-22).  bf16 operands, fp32 accumulation in TMEM. */
int cvit_linear_bias_bf16(const void* A, int64_t lda, const void* W, const float* bias, void* out, int64_t ldo,
                          int64_t M, int64_t N, int64_t K, int gelu, void* stream);

/* SwiGLU FFN input half: out_bf16[M, N2/2] = silu(A @ W1^T + b1) * (A @ W2^T + b2).  Replaces
 * SwiGLUFFNFused.w12 + silu(x1)*x2 (upstream swiglu_ffn.py; HF:354-360).  W12i / bias12i are the w12
 * parameters with rows re-ordered per 256-row tile as [128 rows of w1 | the matching 128 rows of w2]
 * (cryovit_b200.vit.interleave_w12 does this at load time).  N2 = 2 * hidden, multiple of 256. */
int cvit_linear_swiglu_bf16(const void* A, int64_t lda, const void* W12i, const float* bias12i, void* out,
                            int64_t ldo, int64_t M, int64_t N2, int64_t K, void* stream);

/* x_f32[M, N] += gamma * (A @ W^T + bias).  Replaces attn.proj + ls1 + residual and w3/fc2 + ls2 + residual
 * (upstream block.py, layer_scale.py; HF:257-300,355-361,386-404). */
int cvit_linear_scale_residual_f32(const void* A, int64_t lda, const void* W, const float* bias, const float* gamma,
                                   float* x, int64_t ldx, int64_t M, int64_t N, int64_t K, void* stream);

/* 16-bit operand formats of the three linears above.  The reference runs these GEMMs in TF32 (10 mantissa bits,
 * run/dino_features.py:24 set_float32_matmul_precision("high")); IEEE fp16 keeps the same 10 bits for operands whose
 * range is bounded (LayerNorm output, q/k/v, attention output, and the weights they meet), bf16 (7 bits) stays the
 * choice where range matters (the FFN hidden activations).  `fmt` is a combination of:
 *   CVIT_FMT_OPERANDS_F16  A and W hold IEEE fp16 instead of bf16 (always both: a tcgen05 kind::f16 MMA takes one
 *                          16-bit type for both operands);
 *   CVIT_FMT_OUT_F16       the 16-bit output of linear_bias / linear_swiglu is stored as fp16 instead of bf16;
 *   CVIT_FMT_OPERANDS_TF32 A and W are fp32 holding TF32 values (tcgen05 kind::tf32, half the kind::f16 rate): the
 *                          reference's own matmul precision (run/dino_features.py:24).  lda and K in fp32 elements,
 *                          multiples of 4, K >= 32;
 *   CVIT_FMT_OUT_F32       with CVIT_FMT_OPERANDS_TF32, and required there by linear_bias with gelu = 1 and by
 *                          linear_swiglu: the output is fp32 rounded to TF32, the A operand of the next TF32 linear.
 *                          linear_bias without GELU (qkv) keeps its 16-bit output under TF32 operands.
 * Combinations without an instantiated kernel (TF32 with fp16 operands, CVIT_FMT_OUT_F32 without TF32 operands or
 * on the 16-bit outputs) return CVIT_ERR_UNSUPPORTED.  fmt = 0 is exactly the *_bf16 / *_f32 entry point of the
 * same name. */
#define CVIT_FMT_OPERANDS_F16 1
#define CVIT_FMT_OUT_F16 2
#define CVIT_FMT_OPERANDS_TF32 4
#define CVIT_FMT_OUT_F32 8
int cvit_linear_bias_fmt(const void* A, int64_t lda, const void* W, const float* bias, void* out, int64_t ldo,
                         int64_t M, int64_t N, int64_t K, int gelu, int fmt, void* stream);
int cvit_linear_swiglu_fmt(const void* A, int64_t lda, const void* W12i, const float* bias12i, void* out,
                           int64_t ldo, int64_t M, int64_t N2, int64_t K, int fmt, void* stream);
int cvit_linear_scale_residual_fmt(const void* A, int64_t lda, const void* W, const float* bias, const float* gamma,
                                   float* x, int64_t ldx, int64_t M, int64_t N, int64_t K, int fmt, void* stream);

/* out_bf16[M, N] = At[K, M]^T @ W[N, K]^T + bias (+ exact-erf GELU): the same linear with A read from its TRANSPOSED
 * storage (row k of At holds the M values of input channel k, M contiguous, ldat elements apart) as an MN-major
 * tensor-core operand.  At and W are IEEE fp16.  Replaces, in one kernel, the head's input permute
 * (models/cryovit.py:38-41, datamodules/utils.py collate: (C, D, h, w) features -> channels-last) AND layers[0]
 * Conv3d 1x1x1 + GELU (models/cryovit.py:19-22): the on-disk fp16 feature volume is the A operand as it lies, no
 * channels-last copy is written.  M, ldat multiples of 8; K >= 64; N multiple of 128. */
int cvit_linear_bias_cfirst_f16(const void* At, int64_t ldat, const void* W, const float* bias, void* out, int64_t ldo,
                                int64_t M, int64_t N, int64_t K, int gelu, void* stream);

/* Multi-head self-attention of every slice: out[b, t, h*64 + d] = softmax(q k^T / 8) v with
 * q,k,v = qkv[b, t, {0,1,2}, h, :].  Replaces MemEffAttention / xformers memory_efficient_attention
 * (upstream attention.py; HF:202-256).  qkv bf16 [n_slices * tokens, 3 * heads * 64]; head_dim must be 64. */
int cvit_attention_fwd_bf16(const void* qkv, void* out, int64_t n_slices, int64_t tokens, int64_t heads,
                            int64_t head_dim, void* stream);
/* Same kernel with IEEE fp16 q/k/v, probabilities and output (fp32 scores, softmax and accumulation as above). */
int cvit_attention_fwd_f16(const void* qkv, void* out, int64_t n_slices, int64_t tokens, int64_t heads,
                           int64_t head_dim, void* stream);
/* The same kernel by format flags: fmt = 0 (all bf16), CVIT_FMT_OUT_F16 (bf16 q/k/v and probabilities, fp16 output:
 * the default ViT path -- the format of q/k/v/P does not move the end-to-end error, the format of the output that
 * meets the projection weights does), CVIT_FMT_OPERANDS_F16 | CVIT_FMT_OUT_F16 (= cvit_attention_fwd_f16), or
 * CVIT_FMT_OUT_F32 (bf16 q/k/v and probabilities, output fp32 rounded to TF32 for a TF32 projection).  Other flags
 * return CVIT_ERR_UNSUPPORTED. */
int cvit_attention_fwd_fmt(const void* qkv, void* out, int64_t n_slices, int64_t tokens, int64_t heads,
                           int64_t head_dim, int fmt, void* stream);
/* Same contract on the legacy warp-level mma.sync path: kept only as an A/B comparison kernel for profiles. */
int cvit_attention_fwd_bf16_mma_sync(const void* qkv, void* out, int64_t n_slices, int64_t tokens, int64_t heads,
                                     int64_t head_dim, void* stream);

/* Final LayerNorm + patch-token slice + (B, Np, C) -> (C, D, Np) transpose + fp16 cast, written into the
 * tomogram-wide feature volume at depth offset d0.  Replaces model.norm + x_norm_patchtokens (HF:477-503) and
 * run/dino_features.py:58-64 (reshape, permute([3,0,1,2]).contiguous(), .half(), concatenate(axis=1)). */
int cvit_final_norm_writeout_f16(const float* x, const float* gamma, const float* beta, void* features_f16,
                                 int64_t n_slices, int64_t tokens_per_slice, int64_t first_patch_token,
                                 int64_t n_patches, int64_t C, int64_t D_total, int64_t d0, float eps, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * CryoVIT 3-D head (models/cryovit.py:10-83), channels-last bf16 volumes.
 */

/* fp16 feature volume (C, D, h, w) -> bf16 channels-last (D, h, w, C): the head's input permute
 * (models/cryovit.py:45-46, datamodules/utils.py:105-107) fused with the dtype change. */
int cvit_features_to_ndhwc_bf16(const void* features_f16, void* out_bf16, int64_t C, int64_t DHW, void* stream);
/* Same from the fp32 (C, D, h, w) volume the reference's collate_fn hands to forward_volume. */
int cvit_features_f32_to_ndhwc_bf16(const float* features_f32, void* out_bf16, int64_t C, int64_t DHW, void* stream);

/* GroupNorm(G groups, eps) over a channels-last bf16 volume [DHW, C], statistics over (C/G) * DHW per group,
 * in fp32 (models/cryovit.py:69).  stats is a caller-provided fp32 scratch of 2*G floats (zeroed here). */
int cvit_groupnorm_ndhwc_bf16(const void* x, void* out, const float* gamma, const float* beta, float* stats,
                              int64_t DHW, int64_t C, int64_t G, float eps, void* stream);

/* GroupNorm FOLDED into its neighbours (head inference; models/cryovit.py:56-62 GroupNorm -> Conv3d of a SynthesisBlock).
 * Instead of a statistics pass and a normalise pass over the volume:
 *   producer  cvit_linear_bias_cfirst_f16_gn / cvit_linear_bias_gelu_bf16_gn (layers[0] + GELU) and
 *             cvit_convT_1x2x2_ndhwc_gn (the previous block's ConvTranspose3d + GELU) are the plain kernels of the same name
 *             that ALSO write gn_partials: fp32 [rows32][N / gn_cpg][2] = (sum, sum of squares) of the stored values per
 *             32-row block and per group of gn_cpg (4 or 8) consecutive output columns. rows32 must cover
 *             ceil(M / 1024) * 32 row blocks (tiles may overhang M); entries past ceil(M / 32) are not defined.
 *   fold      cvit_groupnorm_fold reduces the first rows32 = ceil(M / 32) row blocks in a fixed order to the per-channel
 *             scale a_c = gamma_c * rstd_g and shift b_c = beta_c - mean_g * a_c (ab: fp32 [2][channels]; partial_cols =
 *             N / gn_cpg = reps * groups; n_per_group = values per group), then writes w_out = bf16(w32 * a_ci) in the
 *             consumer's operand layout (layout 0: cvit_conv3d_dilated_ndhwc's [27 * cout_pad][cin]; layout 1:
 *             cvit_conv3d_halo_ndhwc's image, cin a multiple of 16; n_elems = 27 * cin * cout_pad; w32 is the fp32 original in
 *             the same layout) and table: fp32 [64][cout_pad], row (dm*4 + hm)*4 + wm = bias + sum over the taps that the
 *             2-bit masks (bit 0: the -1 tap, bit 1: the +1 tap along depth / height / width is inside the volume) admit
 *             of sum_ci w32[tap][co][ci] * b_ci -- zero padding pads the NORMALISED tensor, so a border voxel must not
 *             receive the shift through taps that fall outside.
 *   consumer  cvit_conv3d_dilated_ndhwc_tab / cvit_conv3d_halo_ndhwc_tab convolve the un-normalised volume with the folded
 *             weights and add each voxel's table row (+ GELU). */
int cvit_linear_bias_cfirst_f16_gn(const void* At, int64_t ldat, const void* W, const float* bias, void* out, int64_t ldo,
                                   int64_t M, int64_t N, int64_t K, int gelu, float* gn_partials, int64_t gn_cpg, void* stream);
int cvit_linear_bias_gelu_bf16_gn(const void* A, int64_t lda, const void* W, const float* bias, void* out, int64_t ldo,
                                  int64_t M, int64_t N, int64_t K, float* gn_partials, int64_t gn_cpg, void* stream);
int cvit_convT_1x2x2_ndhwc_gn(const void* x, const void* w_sub, const float* bias4, void* out, int64_t D, int64_t H,
                              int64_t W, int64_t Cin, int64_t Cout, float* gn_partials, int64_t gn_cpg, void* stream);
/* Layout of the statistics that cvit_convT_1x2x2_ndhwc_gn writes: with 32 output channels in groups of 4 every epilogue thread
 * keeps its group sums in registers for the whole kernel and writes one row [8 groups][2]: this returns that row count (fold
 * with rows32 = rows, partial columns = 8; the buffer must hold rows * 16 floats). 0: the per-32-voxel layout described above. */
int64_t cvit_convT_gn_partial_rows(int64_t Cout, int64_t gn_cpg);
 /* ab must hold cvit_groupnorm_fold_ab_elems(channels, groups) floats (scale / shift first, then the reduction's
  * scratch), 16-byte aligned, ZERO-FILLED once before its first use (the kernels leave the scratch as they found it). */
int64_t cvit_groupnorm_fold_ab_elems(int64_t channels, int64_t groups);
int cvit_groupnorm_fold(const float* partials, int64_t rows32, int64_t partial_cols, int64_t groups, int64_t channels,
                        double n_per_group, const float* gamma, const float* beta, float eps, float* ab,
                        const float* w32, void* w_out, int64_t n_elems, int64_t cin, int64_t cout_pad, int layout,
                        const float* bias, float* table, void* stream);
int cvit_conv3d_dilated_ndhwc_tab(const void* x, const void* w_taps, const float* bias_table, void* out, int64_t D,
                                  int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t Cout_valid, int64_t dil,
                                  void* stream);
int cvit_conv3d_halo_ndhwc_tab(const void* x, const void* w_img, const float* bias_table, void* out, int64_t D, int64_t H,
                               int64_t W, int64_t Cin, int64_t Cout_pad, int64_t Cout_valid, int64_t dil, void* stream);

/* The same narrow-layer convolution (Conv3d 3x3x3, dilation (dil,1,1), "same", + bias + GELU; models/cryovit.py:68-78) with
 * P consecutive output voxels along W packed into one tensor-core row (csrc/conv_wpackn.cu): (Cin, Cout_pad) = (32,16) and
 * (32,32) with P = 2, (16,16) with P = 4; W must be a multiple of P.  cvit_conv3d_wpackn_group returns P (0: no such kernel),
 * cvit_conv3d_wpackn_weight_bytes the size of the banded weight image [kd*3+kh][K step][2][j_out * Cout_pad + co][8] that
 * cryovit_b200.head.wpackn_weight_image builds (layout 2 of cvit_groupnorm_fold).  bias_table: fp32 [64][Cout_pad] as for the
 * *_tab kernels (64 equal rows for a plain bias).  act: 1 = GELU, 0 = store the pre-activation. */
int64_t cvit_conv3d_wpackn_group(int64_t Cin, int64_t Cout_pad);
int64_t cvit_conv3d_wpackn_weight_bytes(int64_t Cin, int64_t Cout_pad);
int cvit_conv3d_wpackn_ndhwc(const void* x, const void* w_img, const float* bias_table, void* out, int64_t D, int64_t H,
                             int64_t W, int64_t Cin, int64_t Cout_pad, int64_t Cout_valid, int64_t dil, int act, void* stream);

/* Conv3d(Cin -> Cout, kernel 3, padding "same", dilation (dil,1,1)) + bias + GELU as an implicit GEMM
 * (models/cryovit.py:70-73).  x bf16 [D,H,W,Cin]; w_taps bf16 [27 * Cout, Cin] with tap = (kd*3+kh)*3+kw
 * (Cout may be zero-padded to a multiple of 32, Cout_valid = real channel count = row pitch of out). */
int cvit_conv3d_dilated_ndhwc(const void* x, const void* w_taps, const float* bias, void* out, int64_t D,
                              int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t Cout_valid, int64_t dil,
                              void* stream);

/* The same convolution for the NARROW layers (Cin in {8, 16, 32}; SynthesisBlocks 3-4 and output_layer.0,
 * models/cryovit.py:26-33,68-78) from a shared-memory halo tile: each input voxel is staged once per depth tap
 * instead of once per tap. w_img is the host-arranged shared-memory image of the weights (bf16,
 * cvit_conv3d_halo_weight_bytes(Cin, Cout_pad) bytes; cryovit_b200.head.halo_weight_image builds it); Cout_pad in
 * {16, 32} is the MMA N, Cout_valid (multiple of 8) the stored channel count = row pitch of out. */
int64_t cvit_conv3d_halo_weight_bytes(int64_t Cin, int64_t Cout_pad);
int cvit_conv3d_halo_ndhwc(const void* x, const void* w_img, const float* bias, void* out, int64_t D, int64_t H,
                           int64_t W, int64_t Cin, int64_t Cout_pad, int64_t Cout_valid, int64_t dil, void* stream);

/* The two 8-channel full-resolution convolutions of output_layer (models/cryovit.py:30-34) with P consecutive output
 * voxels of a row packed into the MMA N dimension (banded weight matrix; csrc/conv_wpack.cu). x is bf16 [D,H,W,8], W a
 * multiple of P (8 resp. 16), dilation 1. w_img is the host-arranged banded image (bf16,
 * cvit_conv3d_wpack_weight_bytes(P, Cout) bytes; cryovit_b200.head.wpack_weight_image), bias_n the bias repeated per
 * packed voxel ([P * Cout] fp32).
 *   cvit_conv3d_wpack8_gelu : output_layer.0 (8 -> 8) + bias + GELU (act = 1) -> bf16 [D,H,W,8]
 *   cvit_conv3d_wpack8_final: output_layer.2 (8 -> 1) + bias + clip(-5, 5) -> logits fp32 [D,H,W] and/or
 *                             sigmoid of them -> probs (cryovit.py:39,49); either pointer may be null. */
int64_t cvit_conv3d_wpack_weight_bytes(int64_t P, int64_t Cout);
int cvit_conv3d_wpack8_gelu(const void* x, const void* w_img, const float* bias_n, void* out, int64_t D, int64_t H,
                            int64_t W, int act, void* stream);
int cvit_conv3d_wpack8_final(const void* x, const void* w_img, const float* bias_n, float* logits, float* probs,
                             int64_t D, int64_t H, int64_t W, void* stream);

/* output_layer.0 (8 -> 8 channels, 3x3x3, dilation 1; models/cryovit.py:30-32) with ONE VOXEL PER MMA ROW and the channels-last
 * volume as the operand as it lies (csrc/conv_rows8.cu): a row of voxels at its 16-byte pitch is a K-major operand whose K
 * chunks -- the three column taps -- are the same bytes one voxel further on; the nine (plane, row) partial sums of an
 * output voxel meet in sliding windows of tensor memory. x, out (and aux) bf16 [D,H,W,8], W a multiple of 8; bias fp32 [8];
 * w_img bf16, cvit_conv3d_rows8_weight_bytes() bytes (cryovit_b200.head.rows8_weight_image);
 * act: 0 none, 1 GELU, 2 out = pre-activation and aux = GELU of it, 3 out = result * gelu'(aux) (an input-gradient convolution
 * handing on the gradient of the pre-activation aux; the z values are prefetched before the accumulator wait) with
 * db (fp32 [8], may be null) += the column sums of what is stored: the bias gradient of the layer below. */
int64_t cvit_conv3d_rows8_weight_bytes(void);
int cvit_conv3d_rows8(const void* x, const void* w_img, const float* bias, void* out, int64_t D, int64_t H, int64_t W,
                      int act, void* aux, float* db, void* stream);
/* output_layer.2 (8 -> 1) the same way (w_img: the image of the [1,8,3,3,3] weight, bias fp32 [1]) + clip(-5, 5) -> logits
 * fp32 [D,H,W] and/or their sigmoid -> probs (cryovit.py:39,49); either pointer may be null. */
int cvit_conv3d_rows8_final(const void* x, const void* w_img, const float* bias, float* logits, float* probs, int64_t D,
                            int64_t H, int64_t W, void* stream);
/* ... scored instead of stored (a validation pass): the same MMAs, clip and sigmoid, and an epilogue that reads the voxel's
 * int8 label (labels [D,H,W], -1 = ignore) and accumulates the eight masked sums of cvit_seg_stats with threshold; out8 fp64 [8]
 * is overwritten. Each CTA writes one fp64 row of 8 into partials (cvit_conv3d_rows8_score_partials(D, H, W) doubles the caller
 * provides), a one-block kernel adds the rows in a fixed order: counts (sums 1, 3..7) are exact, and two runs give
 * bit-identical sums. W % 8 != 0: CVIT_ERR_UNSUPPORTED; null labels / partials / out8: CVIT_ERR_INVALID. */
int64_t cvit_conv3d_rows8_score_partials(int64_t D, int64_t H, int64_t W);
int cvit_conv3d_rows8_score(const void* x, const void* w_img, const float* bias, const int8_t* labels, int64_t D, int64_t H,
                            int64_t W, float threshold, double* partials, double* out8, void* stream);

/* The 16- / 32-channel depth-dilated convolutions of SynthesisBlocks 3-4 the same way (csrc/conv_rows.cu): 8-channel chunk arrays
 * of the input rows as K-major operands (column taps = 16-byte shifts), a 144-column accumulator window per input row sliding
 * through tensor memory, the planes of one dilation residue class walked like a dilation-1 stack. Cin, Cout in {16, 32};
 * x bf16 [D,H,W,Cin], out (aux) bf16 [D,H,W,Cout]; bias_table fp32 [64][Cout] (the *_tab layout; a plain bias = 64 equal rows);
 * w_img: Cout / 16 images of cvit_conv3d_rows_weight_bytes(Cin) bytes (cryovit_b200.head.rowsn_weight_image);
 * act / aux / db as cvit_conv3d_rows8 (db fp32 [Cout]). */
int64_t cvit_conv3d_rows_weight_bytes(int64_t Cin);
int cvit_conv3d_rows_ndhwc(const void* x, const void* w_img, const float* bias_table, void* out, int64_t D, int64_t H,
                           int64_t W, int64_t Cin, int64_t Cout, int64_t dil, int act, void* aux, float* db, void* stream);

/* ConvTranspose3d(Cin -> Cout, kernel (1,2,2), stride (1,2,2)) + bias + GELU (models/cryovit.py:74-77) as a
 * per-voxel GEMM with a pixel-shuffle store.  w_sub bf16 [4 * Cout, Cin], row (i*2+j)*Cout + co;
 * bias4 fp32 [4 * Cout] (the bias repeated per sub-pixel); out bf16 [D, 2H, 2W, Cout]. */
int cvit_convT_1x2x2_ndhwc(const void* x, const void* w_sub, const float* bias4, void* out, int64_t D, int64_t H,
                           int64_t W, int64_t Cin, int64_t Cout, void* stream);

/* Head tail: Conv3d(8->8,k3) + GELU + Conv3d(8->1,k3) + clip(-5,5) [+ sigmoid] (models/cryovit.py:30-49).
 * x bf16 [D,H,W,8]; w1 fp32 [27][8 out][8 in]; w2 fp32 [27][8]; logits/probs fp32 [D,H,W] (either may be
 * NULL); scratch_bf16 holds the 8-channel intermediate, [D,H,W,8] bf16. */
int cvit_head_tail_fused(const void* x, const float* w1, const float* b1, const float* w2, const float* b2,
                         float* logits, float* probs, void* scratch_bf16, int64_t D, int64_t H, int64_t W,
                         void* stream);

/* The last convolution alone: Conv3d(8->1,k3) + clip(-5,5) [+ sigmoid], fp32 on the CUDA cores
 * (models/cryovit.py:33,39,49); x bf16 [D,H,W,8] is the GELU output of output_layer.0, which runs on tensor cores
 * through cvit_conv3d_halo_ndhwc. w2 fp32 [27][8]; logits / probs fp32 [D,H,W] (either may be NULL). */
int cvit_head_out_conv(const void* x, const float* w2, const float* b2, float* logits, float* probs, int64_t D, int64_t H,
                       int64_t W, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Head TRAINING (BASELINE config 5; models/base_model.py:58-63,91-164, models/losses.py:17-32,
 * configs/trainer/fit.yaml). Forward runs the inference kernels with act = 0 (pre-activations are kept) followed by
 * cvit_gelu_fwd_bf16; input gradients are the same convolution kernels on flipped / transposed weights (act = 0);
 * weight gradients are split-K GEMMs over channels-first, zero-padded copies of the activations.
 */

/* The three convolution entry points with an explicit activation switch: act = 1 GELU after the bias (the
 * inference entry points above), act = 0 none. */
int cvit_conv3d_dilated_ndhwc_act(const void* x, const void* w_taps, const float* bias, void* out, int64_t D,
                                  int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t Cout_valid, int64_t dil,
                                  int act, void* stream);
int cvit_conv3d_halo_ndhwc_act(const void* x, const void* w_img, const float* bias, void* out, int64_t D, int64_t H,
                               int64_t W, int64_t Cin, int64_t Cout_pad, int64_t Cout_valid, int64_t dil, int act,
                               void* stream);
int cvit_convT_1x2x2_ndhwc_act(const void* x, const void* w_sub, const float* bias4, void* out, int64_t D, int64_t H,
                               int64_t W, int64_t Cin, int64_t Cout, int act, void* stream);

/* Fused element-wise passes of the training step (reference: nn.GELU() between the layers of models/cryovit.py:19-37,
 * 68-78 and its autograd backward). The *_aux entry points are the kernels above with a second bf16 tensor `aux` of
 * the output's shape and indexing, and act one of
 *     0  out = y                          1  out = gelu(y)
 *     2  out = y, aux = gelu(y)           (training forward: the pre-activation is kept for the backward pass)
 *     3  out = y * gelu'(aux)             (input-gradient convolution; aux = saved pre-activation of the layer below)
 * y = the convolution / GEMM result plus bias. act 0 / 1 ignore aux (may be null); act 3 is not offered by the
 * transposed convolution and the channels-first linear. aux must be 16-byte aligned. */
int cvit_conv3d_dilated_ndhwc_aux(const void* x, const void* w_taps, const float* bias, void* out, int64_t D,
                                  int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t Cout_valid, int64_t dil,
                                  int act, void* aux, void* stream);
int cvit_conv3d_halo_ndhwc_aux(const void* x, const void* w_img, const float* bias, void* out, int64_t D, int64_t H,
                               int64_t W, int64_t Cin, int64_t Cout_pad, int64_t Cout_valid, int64_t dil, int act,
                               void* aux, void* stream);
int cvit_conv3d_wpackn_ndhwc_aux(const void* x, const void* w_img, const float* bias_table, void* out, int64_t D, int64_t H,
                                 int64_t W, int64_t Cin, int64_t Cout_pad, int64_t Cout_valid, int64_t dil, int act,
                                 void* aux, void* stream);
int cvit_conv3d_wpack8_aux(const void* x, const void* w_img, const float* bias_n, void* out, int64_t D, int64_t H,
                           int64_t W, int act, void* aux, void* stream);
int cvit_convT_1x2x2_ndhwc_aux(const void* x, const void* w_sub, const float* bias4, void* out, int64_t D, int64_t H,
                               int64_t W, int64_t Cin, int64_t Cout, int act, void* aux, void* stream);
int cvit_linear_bias_cfirst_f16_aux(const void* At, int64_t ldat, const void* W, const float* bias, void* out, int64_t ldo,
                                    int64_t M, int64_t N, int64_t K, int act, void* aux, void* stream);
/* act 0 or 3 only; aux bf16 [M, n_valid] with row pitch ldo. */
int cvit_linear_bias_bf16_nvalid_aux(const void* A, int64_t lda, const void* W, const float* bias, void* out, int64_t ldo,
                                     int64_t M, int64_t N, int64_t K, int64_t n_valid, int act, const void* aux, void* stream);

/* cvit_linear_bias_bf16 (no GELU) for an output narrower than the zero-row-padded weight: columns >= n_valid are not
 * stored and ldo is the true row pitch (input gradient of the 16-channel transposed convolution). */
int cvit_linear_bias_bf16_nvalid(const void* A, int64_t lda, const void* W, const float* bias, void* out, int64_t ldo,
                                 int64_t M, int64_t N, int64_t K, int64_t n_valid, void* stream);

/* a = gelu(z) and dz = da * gelu'(z) (exact erf form, nn.GELU() default), bf16, n a multiple of 8. */
int cvit_gelu_fwd_bf16(const void* z, void* a, int64_t n, void* stream);
int cvit_gelu_bwd_bf16(const void* da, const void* z, void* dz, int64_t n, void* stream);
/* The same over a bf16 [R, C] matrix with the bias gradient on the way: db[c] += sum_r dz[r, c] (fp32 [C], caller zeroes;
 * C % 8 == 0, C <= 2048) -- what autograd's conv bias gradient reduces, without a second pass over dz. */
int cvit_gelu_bwd_colsum_bf16(const void* da, const void* z, void* dz, float* db, int64_t R, int64_t C, void* stream);
/* The same over a bf16 [D, H2, W2, C] volume (H2, W2 even) with dz stored PIXEL-UNSHUFFLED, [D, H2/2, W2/2, (i, j, C)]:
 * the row layout the transposed convolution's input- and weight-gradient GEMMs read (saves the separate
 * cvit_pixel_unshuffle_1x2x2_bf16 pass over the step's largest gradient volumes). */
int cvit_gelu_bwd_colsum_unshuffle_bf16(const void* da, const void* z, void* dzun, float* db, int64_t D, int64_t H2, int64_t W2,
                                        int64_t C, void* stream);

/* Gradient of DiceLoss (models/losses.py:17-32) w.r.t. the raw logits, through sigmoid and clip(-5, 5)
 * (models/cryovit.py:39,49), masked to label > -1 (models/base_model.py:91-112). stats8 = the device-resident sums
 * of cvit_seg_stats for the same forward pass; scale multiplies the gradient (1 / world size for data parallel
 * averaging). Output: bf16 [n][8] with channel 0 = dL/dlogit and channels 1..7 zero (the operand of the narrow
 * convolution kernel that back-propagates through output_layer.2). */
int cvit_dice_bwd(const float* logits, const float* probs, const float* labels, const double* stats8, float scale,
                  void* dlogit8_bf16, int64_t n, void* stream);

/* out[c] += sum over rows of x[r, c] (bias gradients). x bf16 [R, C], out fp32 [C] (caller zeroes), C % 8 == 0. */
int cvit_colsum_bf16(const void* x, float* out, int64_t R, int64_t C, void* stream);

/* GroupNorm backward over a channels-last bf16 volume (models/cryovit.py:69): x = the forward INPUT, stats = the
 * forward statistics buffer of cvit_groupnorm_ndhwc_bf16; writes dx (bf16) and dgamma / dbeta (fp32 [C], zeroed
 * here). */
int cvit_groupnorm_bwd_ndhwc_bf16(const void* x, const void* dy, void* dx, const float* gamma, const float* stats,
                                  float* dgamma, float* dbeta, int64_t DHW, int64_t C, int64_t G, float eps, void* stream);
/* The same followed by the GELU backward of the layer below in ONE pass: z (bf16, x's shape) is the pre-activation with
 * x = gelu(z); dx receives d(z) = d(x) * gelu'(z), db (fp32 [C], zeroed by the caller) += its column sums (that layer's bias
 * gradient), and with W2 > 0 (x a [D, H2, W2, C] volume, H2 and W2 even) it is stored pixel-unshuffled, [D, H2/2, W2/2, 4C]
 * (the row layout of the transposed convolution's gradient GEMMs). z = null: exactly cvit_groupnorm_bwd_ndhwc_bf16. */
int cvit_groupnorm_bwd_gelu_ndhwc_bf16(const void* x, const void* dy, void* dx, const float* gamma, const float* stats, float* dgamma,
                                       float* dbeta, int64_t DHW, int64_t C, int64_t G, float eps, const void* z, float* db,
                                       int64_t W2, void* stream);

/* [D, 2H, 2W, C] -> [D, H, W, 4C], column (i*2+j)*C + c: the transposed convolution's output gradient laid out as the
 * rows of the GEMM that yields its input gradient. */
int cvit_pixel_unshuffle_1x2x2_bf16(const void* src, void* dst, int64_t D, int64_t H, int64_t W, int64_t C, void* stream);

/* channels-last bf16 [D,H,W,C] -> channels-first, zero-padded bf16 [C][pitch]: position p over the padded volume
 * (D + 2 pd, H + 2 ph, Wp) holds voxel (dp - pd, hp - ph, wp - pw + wshift) or zero; Wp >= W + 2 pw is the padded row
 * pitch, pitch >= the padded size, multiple of 8. Operand layout of cvit_wgrad_splitk (whose shifts must be multiples
 * of 8 elements: make Wp a multiple of 8 and take the +-1 column taps from copies made with wshift = -1 / +1). */
int cvit_ndhwc_to_cfirst_padded(const void* src, void* dst, int64_t D, int64_t H, int64_t W, int64_t C, int64_t pd,
                                int64_t ph, int64_t pw, int64_t Wp, int64_t wshift, int64_t pitch, void* stream);

/* The three column-shifted copies (wshift -1, 0, +1) of a narrow volume (C in {8, 16, 32}) in one pass. */
int cvit_ndhwc_to_cfirst_padded_x3(const void* src, void* dst_m1, void* dst_0, void* dst_p1, int64_t D, int64_t H,
                                   int64_t W, int64_t C, int64_t pd, int64_t ph, int64_t pw, int64_t Wp, int64_t pitch,
                                   void* stream);

/* out[t][m][n] += sum_k At[m][k] * Bt[n][k + koffs[t]]  for t < ntaps (fp32 out, caller zeroes; terms whose shifted
 * index falls outside [0, K) are zero). At bf16 [M][pitch_a], Bt bf16 [N][pitch_b]; koffs int32 [ntaps] on the
 * device, every shift a multiple of 8 (TMA start alignment). Split over the whole GPU along K; every partial tile is added with red.global.add.f32. */
int cvit_wgrad_splitk(const void* At, const void* Bt, float* out, const int* koffs, int64_t M, int64_t N, int64_t K,
                      int64_t pitch_a, int64_t pitch_b, int64_t ntaps, void* stream);

/* out[t][m][n] += sum over voxels v of  A[v + off_a(t)][m] * B[v + off_b(t)][n]   (fp32 out [ntaps][Ca][Cb], caller zeroes)
 * straight from two channels-last bf16 volumes a [D,H,W,Ca], b [D,H,W,Cb] (Ca, Cb >= 64, multiples of 8): the weight
 * gradient of a wide 3x3x3 depth-dilated "same" convolution (ntaps = 27, tap t = (kd*3+kh)*3+kw shifts the operand chosen
 * by shift_a by ((kd-1) dil, kh-1, kw-1), zero outside the volume; models/cryovit.py:58-66) or of a 1x1x1 / transposed
 * convolution over [rows][channels] matrices (ntaps = 1, W = rows, H = D = 1).  Both operands are read as MN-major
 * tensor-core operands through TMA boxes of the tensors as they lie: no channels-first, padded or column-shifted copies
 * (cvit_wgrad_splitk needs all three).  Split over the GPU along the voxels; partial tiles are added with red.global.add. */
int cvit_wgrad_mn_ndhwc(const void* a, const void* b, float* out, int64_t D, int64_t H, int64_t W, int64_t Ca, int64_t Cb,
                        int64_t dil, int64_t ntaps, int shift_a, void* stream);

/* The same weight gradient for the narrow convolutions (SynthesisBlocks 3-4, output_layer; (Cin, Cout) in {(8,8), (16,16),
 * (32,16), (32,32)}), straight from the channels-last volumes with warp-level MMAs (csrc/wgrad_narrow.cu; no operand
 * copies): dw (fp32 [27][Cout][Cin], tap = (kd*3+kh)*3+kw) += sum_v dz[v, co] * x[v + off(tap), ci]; x bf16 [D,H,W,Cin],
 * dz bf16 [D,H,W,Cout]. */
int cvit_wgrad_narrow_ndhwc(const void* x, const void* dz, float* dw, int64_t D, int64_t H, int64_t W, int64_t Cin,
                            int64_t Cout, int64_t dil, void* stream);

/* The 8 -> 8 channel case (output_layer.0 / output_layer.2 at full resolution) on tcgen05 (csrc/wgrad_tc.cu): the voxels
 * of a row are the K dimension of one MMA per 16 voxels for all 27 taps, both operands are the channels-last volumes as
 * they lie (MN-major, the column taps are 16-byte shifts of the same row). Same contract as cvit_wgrad_narrow_ndhwc with
 * Cin = Cout = 8; W must be a multiple of 8. */
int cvit_wgrad_tc8_ndhwc(const void* x, const void* dz, float* dw, int64_t D, int64_t H, int64_t W, int64_t dil,
                         void* stream);
/* The 16- / 32-channel layers, (Cin, Cout) in {(16,16), (32,16), (32,32)}, the same way: TMA boxes of (8 channels, one
 * chunk, 64 voxels) land as the [voxel][8] operand arrays, the column taps are separate (shifted) arrays of x, one MMA
 * (M 128, N 144) per 16 voxels and 144 accumulator columns. Same contract as cvit_wgrad_narrow_ndhwc, any W. */
int cvit_wgrad_tcn_ndhwc(const void* x, const void* dz, float* dw, int64_t D, int64_t H, int64_t W, int64_t Cin,
                         int64_t Cout, int64_t dil, void* stream);

/* AdamW step over a flat fp32 parameter vector, torch.optim.AdamW semantics (models/base_model.py:58-63):
 * decoupled weight decay, bias-corrected moments; g is multiplied by grad_scale first. step counts from 1. */
int cvit_adamw_f32(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                   float weight_decay, int64_t step, float grad_scale, void* stream);

/* Masked segmentation statistics, one pass: over voxels with label > -1 (BaseModel._masked_predict,
 * models/base_model.py:91-112) accumulates out8 (fp64, caller zeroes) = {sum p, sum y, sum p*y | sum y*[p>=thr],
 * sum [p>=thr] | sum y*[p>.5], sum (1-y)*[p>.5], sum y*(1-[p>.5])}: the reductions behind DiceLoss
 * (models/losses.py:17-32), DiceMetric (models/metrics.py:30-53, "pred < thr -> 0 else 1") and F1Metric
 * (models/metrics.py:69-93, strict "> 0.5"). probs, labels: fp32 [n]. */
int cvit_seg_stats(const float* probs, const float* labels, int64_t n, float threshold, double* out8, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CRYOVIT_B200_H */
