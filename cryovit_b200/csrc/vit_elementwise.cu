// HBM-bound ViT kernels: slice pre-processing + patchify, special-token assembly, LayerNorm,
// and the final-norm + fp16 (C, D, h, w) feature write-out.
#include "ptx.cuh"
#include "tmap.h"

namespace cvit {

// ------------------------------------------------------------------------------------------------
// Pre-processing. Restates VITDataset._load_tomogram + _dino_transform (reference
// src/cryovit/datasets/vit_dataset.py:71-123): uint8 -> /255 (float data passes through), edge-pad H,W up
// to multiples of 16, bicubic resample by 14/16 (ATen upsample_bicubic2d: A = -0.75, align_corners =
// False, scale passed explicitly so src = (dst + 0.5) * (1/0.875) - 0.5, border indices clamped), and the
// result cut into 14x14 patches laid out as GEMM rows [slice*Np + patch, i*14 + j] in bf16.
// The three input channels of the reference are identical copies, so one channel is produced and the
// patch-embed weight is pre-summed over its input channels on the host.
__device__ __forceinline__ float cubic1(float x, float A) { return ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f; }
__device__ __forceinline__ float cubic2(float x, float A) { return ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A; }

__device__ __forceinline__ float load_px(const uint8_t* p) { return static_cast<float>(*p) / 255.0f; }
__device__ __forceinline__ float load_px(const float* p) { return *p; }

// Patch rows are stored as bf16 (the 16-bit operand paths) or, for the TF32 GEMMs, as TF32-rounded fp32: bf16 keeps 8
// significant bits of the 10-bit-exact pixels the reference embeds, TF32 keeps 11.
__device__ __forceinline__ void store_patch(__nv_bfloat16* p, float v) { *p = __float2bfloat16(v); }
__device__ __forceinline__ void store_patch(float* p, float v) { *p = round_tf32(v); }

template <typename T, typename OutT>
__global__ void preproc_patchify_kernel(const T* __restrict__ src, OutT* __restrict__ dst, int D, int H,
                                        int W, int OH, int OW, int Kp, float inv_scale) {
  const int pw = OW / 14, ph = OH / 14;
  const int64_t total = (int64_t)D * ph * pw * Kp;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int col = (int)(idx % Kp);
    const int64_t row = idx / Kp;
    if (col >= 196) {
      store_patch(dst + idx, 0.f);
      continue;
    }
    const int p = (int)(row % (ph * pw));
    const int d = (int)(row / (ph * pw));
    const int oy = (p / pw) * 14 + col / 14;
    const int ox = (p % pw) * 14 + col % 14;
    const float A = -0.75f;
    const float sy = inv_scale * (oy + 0.5f) - 0.5f;
    const float sx = inv_scale * (ox + 0.5f) - 0.5f;
    const float fy = floorf(sy), fx = floorf(sx);
    const int iy = (int)fy, ix = (int)fx;
    const float ty = sy - fy, tx = sx - fx;
    float wy[4] = {cubic2(ty + 1.f, A), cubic1(ty, A), cubic1(1.f - ty, A), cubic2(2.f - ty, A)};
    float wx[4] = {cubic2(tx + 1.f, A), cubic1(tx, A), cubic1(1.f - tx, A), cubic2(2.f - tx, A)};
    const T* plane = src + (int64_t)d * H * W;
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      // the edge-pad to a multiple of 16 replicates the last row/column, which is what clamping to the
      // ORIGINAL extent gives as well
      const int y = min(max(iy - 1 + i, 0), H - 1);
      float r = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int x = min(max(ix - 1 + j, 0), W - 1);
        r += wx[j] * load_px(plane + (int64_t)y * W + x);
      }
      acc += wy[i] * r;
    }
    store_patch(dst + idx, acc);
  }
}

// Same resample, written in the reference's own layout f32 [D, 3, OH, OW] (three identical channels): what
// VITDataset.__getitem__ returns (vit_dataset.py:117-123), for callers that keep the reference's dataset seam.
template <typename T>
__global__ void preproc_resize3_kernel(const T* __restrict__ src, float* __restrict__ dst, int D, int H, int W, int OH,
                                       int OW, float inv_scale) {
  const int64_t plane_o = (int64_t)OH * OW, total = (int64_t)D * plane_o;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int ox = (int)(idx % OW), oy = (int)((idx / OW) % OH), d = (int)(idx / plane_o);
    const float A = -0.75f;
    const float sy = inv_scale * (oy + 0.5f) - 0.5f, sx = inv_scale * (ox + 0.5f) - 0.5f;
    const float fy = floorf(sy), fx = floorf(sx);
    const int iy = (int)fy, ix = (int)fx;
    const float ty = sy - fy, tx = sx - fx;
    const float wy[4] = {cubic2(ty + 1.f, A), cubic1(ty, A), cubic1(1.f - ty, A), cubic2(2.f - ty, A)};
    const float wx[4] = {cubic2(tx + 1.f, A), cubic1(tx, A), cubic1(1.f - tx, A), cubic2(2.f - tx, A)};
    const T* plane = src + (int64_t)d * H * W;
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int y = min(max(iy - 1 + i, 0), H - 1);
      float r = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) r += wx[j] * load_px(plane + (int64_t)y * W + min(max(ix - 1 + j, 0), W - 1));
      acc += wy[i] * r;
    }
    float* o = dst + (int64_t)d * 3 * plane_o + (int64_t)oy * OW + ox;
    o[0] = acc;
    o[plane_o] = acc;
    o[2 * plane_o] = acc;
  }
}

// General patchify for the reference-facing forward_features(x: f32[B,3,H',W']) entry (seam B2):
// rows [b*Np + patch], cols c*196 + i*14 + j, zero-padded to Kp.
template <typename OutT>
__global__ void patchify3_kernel(const float* __restrict__ src, OutT* __restrict__ dst, int B, int OH, int OW,
                                 int Kp) {
  const int pw = OW / 14, ph = OH / 14;
  const int64_t total = (int64_t)B * ph * pw * Kp;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int col = (int)(idx % Kp);
    const int64_t row = idx / Kp;
    if (col >= 588) {
      store_patch(dst + idx, 0.f);
      continue;
    }
    const int c = col / 196, ij = col % 196;
    const int p = (int)(row % (ph * pw));
    const int b = (int)(row / (ph * pw));
    const int oy = (p / pw) * 14 + ij / 14;
    const int ox = (p % pw) * 14 + ij % 14;
    store_patch(dst + idx, src[(((int64_t)b * 3 + c) * OH + oy) * OW + ox]);
  }
}

// ------------------------------------------------------------------------------------------------
// Special tokens: x[b, 0] = cls + pos[0]; x[b, 1 + r] = register r (upstream prepare_tokens_with_masks:
// pos-embed is added before the registers are spliced in, so they carry none).
__global__ void assemble_special_kernel(float* __restrict__ x, const float* __restrict__ special, int B, int T, int C,
                                        int S) {
  const int64_t total = (int64_t)B * S * C;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(idx % C);
    const int s = (int)((idx / C) % S);
    const int b = (int)(idx / ((int64_t)C * S));
    x[((int64_t)b * T + s) * C + c] = special[(int64_t)s * C + c];
  }
}

// ------------------------------------------------------------------------------------------------
// LayerNorm over C (fp32 in, bf16 out), one warp per row, two-pass statistics held in registers.
__device__ __forceinline__ void ln_store4(__nv_bfloat16* row, int i4, float o0, float o1, float o2, float o3) {
  reinterpret_cast<uint2*>(row)[i4] = make_uint2(pack_bf16x2(o0, o1), pack_bf16x2(o2, o3));
}
__device__ __forceinline__ void ln_store4(__half* row, int i4, float o0, float o1, float o2, float o3) {
  reinterpret_cast<uint2*>(row)[i4] = make_uint2(pack_f16x2(o0, o1), pack_f16x2(o2, o3));
}
__device__ __forceinline__ void ln_store4(float* row, int i4, float o0, float o1, float o2, float o3) {
  reinterpret_cast<float4*>(row)[i4] = make_float4(o0, o1, o2, o3);
}
// fp32 output rounded to TF32: the A operand of the TF32 linears (cvit_layernorm_f32_tf32)
struct Tf32Out {
  float v;
};
__device__ __forceinline__ void ln_store4(Tf32Out* row, int i4, float o0, float o1, float o2, float o3) {
  reinterpret_cast<float4*>(row)[i4] = make_float4(round_tf32(o0), round_tf32(o1), round_tf32(o2), round_tf32(o3));
}

template <int NV, typename OutT>  // float4 per lane: C == NV * 128
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, int64_t ldx,
                                                        const float* __restrict__ gamma, const float* __restrict__ beta,
                                                        OutT* __restrict__ out, int64_t ldo, int64_t M, float eps) {
  constexpr int C = NV * 128;
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const float4* xr = reinterpret_cast<const float4*>(x + row * ldx);
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i] = xr[lane + 32 * i];
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  const float mean = warp_sum(s) * (1.0f / C);
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    ss += (a * a + b * b) + (c * c + d * d);
  }
  const float rstd = rsqrtf(warp_sum(ss) * (1.0f / C) + eps);
  OutT* orow = out + row * ldo;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + lane + 32 * i);
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + lane + 32 * i);
    const float o0 = (v[i].x - mean) * rstd * g.x + b.x, o1 = (v[i].y - mean) * rstd * g.y + b.y;
    const float o2 = (v[i].z - mean) * rstd * g.z + b.z, o3 = (v[i].w - mean) * rstd * g.w + b.w;
    ln_store4(orow, lane + 32 * i, o0, o1, o2, o3);
  }
}

template <typename OutT>
static int launch_layernorm(const float* x, int64_t ldx, const float* gamma, const float* beta, OutT* o, int64_t ldo,
                            int64_t M, int64_t C, float eps, cudaStream_t st) {
  const int rows_per_block = 8;
  const int grid = (int)((M + rows_per_block - 1) / rows_per_block);
  switch (C) {
    case 128: layernorm_kernel<1, OutT><<<grid, 256, 0, st>>>(x, ldx, gamma, beta, o, ldo, M, eps); break;
    case 256: layernorm_kernel<2, OutT><<<grid, 256, 0, st>>>(x, ldx, gamma, beta, o, ldo, M, eps); break;
    case 384: layernorm_kernel<3, OutT><<<grid, 256, 0, st>>>(x, ldx, gamma, beta, o, ldo, M, eps); break;
    case 512: layernorm_kernel<4, OutT><<<grid, 256, 0, st>>>(x, ldx, gamma, beta, o, ldo, M, eps); break;
    case 768: layernorm_kernel<6, OutT><<<grid, 256, 0, st>>>(x, ldx, gamma, beta, o, ldo, M, eps); break;
    case 1024: layernorm_kernel<8, OutT><<<grid, 256, 0, st>>>(x, ldx, gamma, beta, o, ldo, M, eps); break;
    case 1536: layernorm_kernel<12, OutT><<<grid, 256, 0, st>>>(x, ldx, gamma, beta, o, ldo, M, eps); break;
    default:
      set_error("layernorm: C=%lld unsupported (128, 256, 384, 512, 768, 1024, 1536)", (long long)C);
      return CVIT_ERR_UNSUPPORTED;
  }
  return check_launch("layernorm_kernel");
}

// ------------------------------------------------------------------------------------------------
// Final LayerNorm + patch-token slice + (B, N, C) -> (C, D, h*w) transpose + fp16 cast. Restates
// x_norm_patchtokens followed by dino_features.py:58-61 (reshape, permute([3,0,1,2]).contiguous(), .half()).
// One CTA = 32 consecutive patch tokens of one slice: rows are normalised warp-per-row, parked in shared
// memory transposed as fp16, then stored as 64-byte runs along the patch axis of the (C, D, Np) volume.
constexpr int WO_TOK = 32;
constexpr int WO_PITCH = WO_TOK + 2;  // halves; 68-byte pitch -> conflict-free transposed writes

__global__ void __launch_bounds__(256) final_norm_writeout_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                                   const float* __restrict__ beta, __half* __restrict__ out,
                                                                   int T, int first_patch_token, int Np, int C, int Dtot,
                                                                   int d0, float eps) {
  extern __shared__ __half s_t[];  // [C][WO_PITCH]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tiles_per_slice = (Np + WO_TOK - 1) / WO_TOK;
  const int b = blockIdx.x / tiles_per_slice;
  const int p0 = (blockIdx.x - b * tiles_per_slice) * WO_TOK;
  const int nper = C / 32;  // channels per lane (<= 48)
  for (int tl = warp; tl < WO_TOK; tl += 8) {
    const int p = p0 + tl;
    if (p >= Np) continue;
    const float* xr = x + ((int64_t)b * T + first_patch_token + p) * C;
    float v[48];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 48; ++k) {
      v[k] = k < nper ? xr[lane + 32 * k] : 0.f;
      s += v[k];
    }
    const float mean = warp_sum(s) / C;
    float ss = 0.f;
#pragma unroll
    for (int k = 0; k < 48; ++k) {
      const float a = k < nper ? v[k] - mean : 0.f;
      ss += a * a;
    }
    const float rstd = rsqrtf(warp_sum(ss) / C + eps);
#pragma unroll
    for (int k = 0; k < 48; ++k) {
      if (k < nper) {
        const int c = lane + 32 * k;
        const float o = (v[k] - mean) * rstd * __ldg(gamma + c) + __ldg(beta + c);
        s_t[c * WO_PITCH + tl] = __float2half_rn(o);
      }
    }
  }
  __syncthreads();
  // half-warp per channel: 16 lanes x 4 bytes = 32 tokens
  const int hw = lane >> 4, l16 = lane & 15;
  const int ntok = min(WO_TOK, Np - p0);
  for (int c = warp * 2 + hw; c < C; c += 16) {
    const int t0 = 2 * l16;
    if (t0 >= ntok) continue;
    __half* orow = out + ((int64_t)c * Dtot + d0 + b) * Np + p0;
    if (t0 + 1 < ntok && ((Np & 1) == 0)) {
      *reinterpret_cast<__half2*>(orow + t0) = *reinterpret_cast<const __half2*>(&s_t[c * WO_PITCH + t0]);
    } else {
      orow[t0] = s_t[c * WO_PITCH + t0];
      if (t0 + 1 < ntok) orow[t0 + 1] = s_t[c * WO_PITCH + t0 + 1];
    }
  }
}

static int grid_for(int64_t total, int threads) {
  int64_t blocks = (total + threads - 1) / threads;
  int64_t cap = (int64_t)num_sms() * 16;
  return (int)(blocks < cap ? (blocks < 1 ? 1 : blocks) : cap);
}

}  // namespace cvit

using namespace cvit;

template <typename OutT>
static int preproc_patchify(const void* src, int src_is_u8, OutT* patches, int64_t D, int64_t H, int64_t W, int64_t Kp,
                            void* stream) {
  if (!src || !patches || D <= 0 || H <= 0 || W <= 0 || Kp < 196 || (Kp % 64) != 0) {
    set_error("preproc_patchify: bad arguments (D=%lld H=%lld W=%lld Kp=%lld)", (long long)D, (long long)H,
              (long long)W, (long long)Kp);
    return CVIT_ERR_INVALID;
  }
  const int H16 = (int)((H + 15) / 16 * 16), W16 = (int)((W + 15) / 16 * 16);
  const int OH = H16 / 16 * 14, OW = W16 / 16 * 14;  // floor(H16 * 0.875)
  const float inv_scale = static_cast<float>(1.0 / 0.875);
  const int64_t total = D * (OH / 14) * (OW / 14) * Kp;
  const int grid = grid_for(total, 256);
  if (src_is_u8)
    preproc_patchify_kernel<uint8_t, OutT><<<grid, 256, 0, (cudaStream_t)stream>>>(
        static_cast<const uint8_t*>(src), patches, (int)D, (int)H, (int)W, OH, OW, (int)Kp, inv_scale);
  else
    preproc_patchify_kernel<float, OutT><<<grid, 256, 0, (cudaStream_t)stream>>>(
        static_cast<const float*>(src), patches, (int)D, (int)H, (int)W, OH, OW, (int)Kp, inv_scale);
  return check_launch("preproc_patchify_kernel");
}

template <typename OutT>
static int patchify_f32_3ch(const float* src, OutT* patches, int64_t B, int64_t OH, int64_t OW, int64_t Kp, void* stream) {
  if (!src || !patches || B <= 0 || OH <= 0 || OW <= 0 || (OH % 14) || (OW % 14) || Kp < 588 || (Kp % 64)) {
    set_error("patchify_f32_3ch: bad arguments (B=%lld OH=%lld OW=%lld Kp=%lld)", (long long)B, (long long)OH,
              (long long)OW, (long long)Kp);
    return CVIT_ERR_INVALID;
  }
  const int64_t total = B * (OH / 14) * (OW / 14) * Kp;
  patchify3_kernel<OutT><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(src, patches, (int)B, (int)OH, (int)OW, (int)Kp);
  return check_launch("patchify3_kernel");
}

extern "C" {

int cvit_preproc_patchify(const void* src, int src_is_u8, void* patches_bf16, int64_t D, int64_t H, int64_t W,
                          int64_t Kp, void* stream) {
  return preproc_patchify(src, src_is_u8, static_cast<__nv_bfloat16*>(patches_bf16), D, H, W, Kp, stream);
}

int cvit_preproc_patchify_tf32(const void* src, int src_is_u8, float* patches, int64_t D, int64_t H, int64_t W,
                               int64_t Kp, void* stream) {
  return preproc_patchify(src, src_is_u8, patches, D, H, W, Kp, stream);
}

int cvit_preproc_resize_f32_3ch(const void* src, int src_is_u8, float* out, int64_t D, int64_t H, int64_t W,
                                void* stream) {
  if (!src || !out || D <= 0 || H <= 0 || W <= 0) {
    set_error("preproc_resize: bad arguments (D=%lld H=%lld W=%lld)", (long long)D, (long long)H, (long long)W);
    return CVIT_ERR_INVALID;
  }
  const int OH = (int)((H + 15) / 16 * 14), OW = (int)((W + 15) / 16 * 14);
  const float inv_scale = static_cast<float>(1.0 / 0.875);
  const int grid = grid_for(D * (int64_t)OH * OW, 256);
  if (src_is_u8)
    preproc_resize3_kernel<uint8_t><<<grid, 256, 0, (cudaStream_t)stream>>>(static_cast<const uint8_t*>(src), out, (int)D,
                                                                          (int)H, (int)W, OH, OW, inv_scale);
  else
    preproc_resize3_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(static_cast<const float*>(src), out, (int)D,
                                                                        (int)H, (int)W, OH, OW, inv_scale);
  return check_launch("preproc_resize3_kernel");
}

int cvit_patchify_f32_3ch(const float* src, void* patches_bf16, int64_t B, int64_t OH, int64_t OW, int64_t Kp,
                          void* stream) {
  return patchify_f32_3ch(src, static_cast<__nv_bfloat16*>(patches_bf16), B, OH, OW, Kp, stream);
}

int cvit_patchify_f32_3ch_tf32(const float* src, float* patches, int64_t B, int64_t OH, int64_t OW, int64_t Kp,
                               void* stream) {
  return patchify_f32_3ch(src, patches, B, OH, OW, Kp, stream);
}

int cvit_assemble_special_tokens(float* x, const float* special, int64_t B, int64_t T, int64_t C, int64_t S,
                                 void* stream) {
  if (!x || !special || B <= 0 || T <= 0 || C <= 0 || S <= 0 || S > T) {
    set_error("assemble_special_tokens: bad arguments");
    return CVIT_ERR_INVALID;
  }
  assemble_special_kernel<<<grid_for(B * S * C, 256), 256, 0, (cudaStream_t)stream>>>(x, special, (int)B, (int)T,
                                                                                      (int)C, (int)S);
  return check_launch("assemble_special_kernel");
}

int cvit_layernorm_f32_bf16(const float* x, int64_t ldx, const float* gamma, const float* beta, void* out,
                            int64_t ldo, int64_t M, int64_t C, float eps, void* stream) {
  if (!x || !gamma || !beta || !out || M <= 0 || (ldx % 4) || (ldo % 4)) {
    set_error("layernorm: bad arguments");
    return CVIT_ERR_INVALID;
  }
  return launch_layernorm(x, ldx, gamma, beta, static_cast<__nv_bfloat16*>(out), ldo, M, C, eps, (cudaStream_t)stream);
}

// Same with an IEEE fp16 result: the A operand of the fp16-operand linears (cvit_linear_*_fmt).
int cvit_layernorm_f32_f16(const float* x, int64_t ldx, const float* gamma, const float* beta, void* out,
                           int64_t ldo, int64_t M, int64_t C, float eps, void* stream) {
  if (!x || !gamma || !beta || !out || M <= 0 || (ldx % 4) || (ldo % 4)) {
    set_error("layernorm: bad arguments");
    return CVIT_ERR_INVALID;
  }
  return launch_layernorm(x, ldx, gamma, beta, static_cast<__half*>(out), ldo, M, C, eps, (cudaStream_t)stream);
}

int cvit_layernorm_f32_f32(const float* x, int64_t ldx, const float* gamma, const float* beta, float* out,
                           int64_t ldo, int64_t M, int64_t C, float eps, void* stream) {
  if (!x || !gamma || !beta || !out || M <= 0 || (ldx % 4) || (ldo % 4)) {
    set_error("layernorm_f32: bad arguments");
    return CVIT_ERR_INVALID;
  }
  return launch_layernorm(x, ldx, gamma, beta, out, ldo, M, C, eps, (cudaStream_t)stream);
}

int cvit_layernorm_f32_tf32(const float* x, int64_t ldx, const float* gamma, const float* beta, float* out,
                            int64_t ldo, int64_t M, int64_t C, float eps, void* stream) {
  if (!x || !gamma || !beta || !out || M <= 0 || (ldx % 4) || (ldo % 4)) {
    set_error("layernorm_tf32: bad arguments");
    return CVIT_ERR_INVALID;
  }
  return launch_layernorm(x, ldx, gamma, beta, reinterpret_cast<Tf32Out*>(out), ldo, M, C, eps, (cudaStream_t)stream);
}

int cvit_final_norm_writeout_f16(const float* x, const float* gamma, const float* beta, void* features_f16,
                                 int64_t n_slices, int64_t tokens_per_slice, int64_t first_patch_token,
                                 int64_t n_patches, int64_t C, int64_t D_total, int64_t d0, float eps, void* stream) {
  if (!x || !gamma || !beta || !features_f16 || n_slices <= 0 || C <= 0 || (C % 32) || C > 1536 ||
      d0 < 0 || d0 + n_slices > D_total || first_patch_token + n_patches > tokens_per_slice) {
    set_error("final_norm_writeout: bad arguments");
    return CVIT_ERR_INVALID;
  }
  const int smem = (int)C * WO_PITCH * (int)sizeof(__half);
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(final_norm_writeout_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         1536 * WO_PITCH * (int)sizeof(__half));
    if (e != cudaSuccess) {
      set_error("final_norm_writeout: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      return CVIT_ERR_CUDA;
    }
    configured = true;
  }
  const int tiles = (int)((n_patches + WO_TOK - 1) / WO_TOK);
  final_norm_writeout_kernel<<<(int)n_slices * tiles, 256, smem, (cudaStream_t)stream>>>(
      x, gamma, beta, static_cast<__half*>(features_f16), (int)tokens_per_slice, (int)first_patch_token,
      (int)n_patches, (int)C, (int)D_total, (int)d0, eps);
  return check_launch("final_norm_writeout_kernel");
}

}  // extern "C"
