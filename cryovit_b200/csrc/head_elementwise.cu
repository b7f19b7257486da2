// HBM-bound pieces of the CryoVIT 3-D head (reference src/cryovit/models/cryovit.py:10-83):
// feature-volume layout change, GroupNorm, and the narrow (8-channel) tail convolutions that are too thin
// for a tensor-core tile and run as direct convolutions on the CUDA cores from a shared-memory halo tile.
#include "det_reduce.cuh"
#include "ptx.cuh"
#include "tmap.h"

namespace cvit {

// ------------------------------------------------------------------------------------------------
// (C, DHW) fp16  ->  (DHW, C) bf16, 64x64 tiles through shared memory.
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f32(float v) { return v; }

template <typename T>
__global__ void __launch_bounds__(256) features_to_ndhwc_kernel(const T* __restrict__ src,
                                                                 __nv_bfloat16* __restrict__ dst, int C, int64_t DHW) {
  __shared__ float tile[64][65];
  const int64_t v0 = (int64_t)blockIdx.x * 64;
  const int c0 = blockIdx.y * 64;
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;  // 64 x 4
  for (int i = ty; i < 64; i += 4) {
    const int c = c0 + i;
    const int64_t v = v0 + tx;
    tile[i][tx] = (c < C && v < DHW) ? to_f32(src[(int64_t)c * DHW + v]) : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 64; i += 4) {
    const int64_t v = v0 + i;
    const int c = c0 + tx;
    if (c < C && v < DHW) dst[v * C + c] = __float2bfloat16(tile[tx][i]);
  }
}

// The fp16 case with 16-byte accesses on both sides (C % 64 == 0, DHW % 64 == 0, 16-byte aligned pointers): a CTA moves a
// 64-channel x 64-voxel tile; a thread loads 8 consecutive voxels of one channel (16 B, a warp covers four full 128 B
// lines), parks them as bf16 in shared memory, then gathers 8 consecutive channels of one voxel (eight 2-byte reads)
// and writes them as one 16-byte store (8 lanes = the voxel's 128 contiguous bytes of this channel tile).
constexpr int FT_PITCH = 72;  // halves per shared-memory row: 144 B keeps 16-byte alignment and skews the banks
__global__ void __launch_bounds__(256) features_f16_to_ndhwc_vec_kernel(const __half* __restrict__ src,
                                                                         __nv_bfloat16* __restrict__ dst, int C, int64_t DHW) {
  __shared__ __align__(16) __nv_bfloat16 tile[64 * FT_PITCH];
  const int64_t v0 = (int64_t)blockIdx.x * 64;
  const int c0 = blockIdx.y * 64;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int q = threadIdx.x + k * 256;  // 512 chunks: channel row q / 8, 8-voxel chunk q % 8
    const int cr = q >> 3, ch = q & 7;
    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(src + (int64_t)(c0 + cr) * DHW + v0 + ch * 8));
    const __half2* h = reinterpret_cast<const __half2*>(&raw);
    uint32_t o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = __half22float2(h[i]);
      o[i] = pack_bf16x2(f.x, f.y);
    }
    *reinterpret_cast<uint4*>(&tile[cr * FT_PITCH + ch * 8]) = make_uint4(o[0], o[1], o[2], o[3]);
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int q = threadIdx.x + k * 256;  // 512 stores: voxel q / 8, 8-channel group q % 8
    const int vl = q >> 3, cg = q & 7;
    const unsigned short* t16 = reinterpret_cast<const unsigned short*>(tile);
    uint32_t o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint32_t lo = t16[(cg * 8 + 2 * i) * FT_PITCH + vl], hi = t16[(cg * 8 + 2 * i + 1) * FT_PITCH + vl];
      o[i] = lo | (hi << 16);
    }
    *reinterpret_cast<uint4*>(dst + (v0 + vl) * C + c0 + cg * 8) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// ------------------------------------------------------------------------------------------------
// GroupNorm over channels-last bf16 [DHW, C]. Pass 1: per-group sum / sum of squares (fp32, block-reduced,
// one atomicAdd pair per (block, group)). Pass 2: normalise + affine.
// Thread t owns the 8-channel vector (t % (C/8)) and strides over rows.
// DET (deterministic mode): no atomics; stats is a [gridDim.x][2G] partial slab, each block's row summed over its threads in
// thread order.
template <bool DET>
__device__ __forceinline__ void groupnorm_stats_body(const __nv_bfloat16* __restrict__ x, float* __restrict__ stats, int64_t DHW, int C,
                                                     int G, int rows_per_block) {
  extern __shared__ float s_part[];  // [2][G] | DET: [256][4] = (s0, q0, s1, q1) per thread
  const int nvec = C / 8;
  const int cpg = C / G;  // channels per group: 8 or 4 (a vector spans 1 or 2 groups)
  if constexpr (!DET) {
    for (int i = threadIdx.x; i < 2 * G; i += blockDim.x) s_part[i] = 0.f;
    __syncthreads();
  }
  const int vec = threadIdx.x % nvec;
  const int rsub = threadIdx.x / nvec, rstep = blockDim.x / nvec;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r1 = min(r0 + rows_per_block, DHW);
  float s[2] = {0.f, 0.f}, q[2] = {0.f, 0.f};
  if (rsub < rstep) {
    for (int64_t r = r0 + rsub; r < r1; r += rstep) {
      const uint4 raw = *reinterpret_cast<const uint4*>(x + r * C + vec * 8);
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f = __bfloat1622float2(h[i]);
        const int half = (cpg == 4) ? (i >> 1) : 0;
        s[half] += f.x + f.y;
        q[half] += f.x * f.x + f.y * f.y;
      }
    }
    if constexpr (DET) {
      s_part[threadIdx.x * 4 + 0] = s[0];
      s_part[threadIdx.x * 4 + 1] = q[0];
      s_part[threadIdx.x * 4 + 2] = s[1];
      s_part[threadIdx.x * 4 + 3] = q[1];
    } else if (cpg >= 8) {
      const int g = (vec * 8) / cpg;
      atomicAdd(&s_part[g], s[0]);
      atomicAdd(&s_part[G + g], q[0]);
    } else {
      const int g = vec * 2;
      atomicAdd(&s_part[g], s[0]);
      atomicAdd(&s_part[G + g], q[0]);
      atomicAdd(&s_part[g + 1], s[1]);
      atomicAdd(&s_part[G + g + 1], q[1]);
    }
  }
  __syncthreads();
  if constexpr (DET) {
    // entry i of the row: group g = i % G, sum (i < G) or sum of squares; threads t < rstep * nvec in order
    const int tn = (blockDim.x / nvec) * nvec;
    for (int i = threadIdx.x; i < 2 * G; i += blockDim.x) {
      const int g = i % G, sq = i >= G ? 1 : 0;
      float a = 0.f;
      for (int t = 0; t < tn; ++t) {
        const int vec = t % nvec;
        if (cpg >= 8) {
          if ((vec * 8) / cpg == g) a += s_part[t * 4 + sq];
        } else if (vec * 2 == g) {
          a += s_part[t * 4 + sq];
        } else if (vec * 2 + 1 == g) {
          a += s_part[t * 4 + 2 + sq];
        }
      }
      stats[(size_t)blockIdx.x * 2 * G + i] = a;
    }
  } else {
    for (int i = threadIdx.x; i < 2 * G; i += blockDim.x) atomicAdd(&stats[i], s_part[i]);
  }
}

__global__ void __launch_bounds__(256) groupnorm_stats_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ stats,
                                                               int64_t DHW, int C, int G, int rows_per_block) {
  groupnorm_stats_body<false>(x, stats, DHW, C, G, rows_per_block);
}

__global__ void __launch_bounds__(256) groupnorm_stats_det_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ partials,
                                                                   int64_t DHW, int C, int G, int rows_per_block) {
  groupnorm_stats_body<true>(x, partials, DHW, C, G, rows_per_block);
}

__global__ void __launch_bounds__(256) groupnorm_apply_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ out,
                                                               const float* __restrict__ gamma, const float* __restrict__ beta,
                                                               const float* __restrict__ stats, int64_t DHW, int C, int G,
                                                               float eps) {
  // The grid stride (gridDim * 256 threads) is a multiple of C / 8 (a power-of-two <= 256 here, checked by the
  // launcher), so a thread meets the SAME 8 channels on every iteration: their scale / shift
  //   y = x * a + b,  a = gamma * rstd,  b = beta - mean * a
  // are computed once and live in registers; the loop is one 16-byte load, 8 FMAs and one 16-byte store, unrolled
  // four deep for memory-level parallelism.
  const int nvec = C / 8;
  const int cpg = C / G;
  const float inv_n = 1.0f / (static_cast<float>(DHW) * cpg);
  const int64_t total = DHW * nvec;
  const int64_t first = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
  const int vec = (int)(first % nvec);
  float a[8], b[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = vec * 8 + i;
    const int g = c / cpg;
    const float mean = stats[g] * inv_n;
    const float var = fmaxf(stats[G + g] * inv_n - mean * mean, 0.f);
    a[i] = rsqrtf(var + eps) * __ldg(gamma + c);
    b[i] = __ldg(beta + c) - mean * a[i];
  }
  auto apply = [&](const uint4& raw) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw);
    uint32_t o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = __bfloat1622float2(h[i]);
      o[i] = pack_bf16x2(fmaf(f.x, a[2 * i], b[2 * i]), fmaf(f.y, a[2 * i + 1], b[2 * i + 1]));
    }
    return make_uint4(o[0], o[1], o[2], o[3]);
  };
  int64_t idx = first;
  for (; idx + 3 * stride < total; idx += 4 * stride) {
    uint4 r[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) r[u] = *reinterpret_cast<const uint4*>(x + (idx + u * stride) * 8);
#pragma unroll
    for (int u = 0; u < 4; ++u) *reinterpret_cast<uint4*>(out + (idx + u * stride) * 8) = apply(r[u]);
  }
  for (; idx < total; idx += stride) *reinterpret_cast<uint4*>(out + idx * 8) = apply(*reinterpret_cast<const uint4*>(x + idx * 8));
}

// ------------------------------------------------------------------------------------------------
// Direct 3x3x3 (dilation 1, zero "same" padding) convolution, 8 input channels, COUT in {8, 1}.
// CTA tile: 1 depth plane x TH rows x 128 columns of outputs; the (3, TH+2, 130) x 8ch bf16 halo is staged in
// shared memory; each thread produces 4 voxels (w = lane + 32*i) so consecutive lanes read consecutive
// 16-byte voxels (conflict-free) and every weight fetched from shared memory feeds 4 FMAs.
constexpr int TAIL_TH = 8;
constexpr int TAIL_TW = 128;

template <int COUT, bool FINAL>
__global__ void __launch_bounds__(256) tail_conv_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w,
                                                         const float* __restrict__ bias, __nv_bfloat16* __restrict__ out_bf16,
                                                         float* __restrict__ logits, float* __restrict__ probs, int D, int H,
                                                         int W) {
  extern __shared__ __align__(16) uint8_t smem[];
  uint4* s_in = reinterpret_cast<uint4*>(smem);                                  // [3][TH+2][TW+2] voxels of 8 bf16
  float* s_w = reinterpret_cast<float*>(smem + 3 * (TAIL_TH + 2) * (TAIL_TW + 2) * 16);  // [27][COUT][8]
  const int tiles_w = (W + TAIL_TW - 1) / TAIL_TW, tiles_h = (H + TAIL_TH - 1) / TAIL_TH;
  int bid = blockIdx.x;
  const int tw = bid % tiles_w;
  bid /= tiles_w;
  const int th = bid % tiles_h;
  const int d = bid / tiles_h;
  const int h0 = th * TAIL_TH, w0 = tw * TAIL_TW;

  for (int i = threadIdx.x; i < 27 * COUT * 8; i += blockDim.x) s_w[i] = w[i];
  constexpr int PW = TAIL_TW + 2, PH = TAIL_TH + 2;
  for (int i = threadIdx.x; i < 3 * PH * PW; i += blockDim.x) {
    const int xw = i % PW, r = i / PW, yh = r % PH, zd = r / PH;
    const int gd = d + zd - 1, gh = h0 + yh - 1, gw = w0 + xw - 1;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (gd >= 0 && gd < D && gh >= 0 && gh < H && gw >= 0 && gw < W)
      v = *reinterpret_cast<const uint4*>(x + (((int64_t)gd * H + gh) * W + gw) * 8);
    s_in[i] = v;
  }
  __syncthreads();

  const int lane = threadIdx.x & 31, hrow = threadIdx.x >> 5;  // 8 warps -> 8 rows
  float acc[4][COUT];
#pragma unroll
  for (int v = 0; v < 4; ++v)
#pragma unroll
    for (int o = 0; o < COUT; ++o) acc[v][o] = __ldg(bias + o);

#pragma unroll 1
  for (int kd = 0; kd < 3; ++kd) {
#pragma unroll 1
    for (int kh = 0; kh < 3; ++kh) {
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const float* wt = s_w + ((kd * 3 + kh) * 3 + kw) * COUT * 8;
        float in[4][8];
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          const uint4 raw = s_in[(kd * PH + hrow + kh) * PW + lane + 32 * v + kw];
          const __nv_bfloat162* hp = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float2 f = __bfloat1622float2(hp[i]);
            in[v][2 * i] = f.x;
            in[v][2 * i + 1] = f.y;
          }
        }
#pragma unroll
        for (int o = 0; o < COUT; ++o) {
          const float4 wa = *reinterpret_cast<const float4*>(wt + o * 8);
          const float4 wb = *reinterpret_cast<const float4*>(wt + o * 8 + 4);
#pragma unroll
          for (int v = 0; v < 4; ++v) {
            acc[v][o] += in[v][0] * wa.x + in[v][1] * wa.y + in[v][2] * wa.z + in[v][3] * wa.w + in[v][4] * wb.x +
                         in[v][5] * wb.y + in[v][6] * wb.z + in[v][7] * wb.w;
          }
        }
      }
    }
  }
  const int gh = h0 + hrow;
  if (gh >= H) return;
#pragma unroll
  for (int v = 0; v < 4; ++v) {
    const int gw = w0 + lane + 32 * v;
    if (gw >= W) continue;
    const int64_t vox = ((int64_t)d * H + gh) * W + gw;
    if (!FINAL) {
      uint32_t o[COUT / 2 > 0 ? COUT / 2 : 1];
#pragma unroll
      for (int i = 0; i < COUT / 2; ++i) o[i] = pack_bf16x2(gelu_erf(acc[v][2 * i]), gelu_erf(acc[v][2 * i + 1]));
      if (COUT == 8) *reinterpret_cast<uint4*>(out_bf16 + vox * 8) = make_uint4(o[0], o[1], o[2], o[3]);
    } else {
      const float z = fminf(fmaxf(acc[v][0], -5.0f), 5.0f);
      if (logits) logits[vox] = z;
      if (probs) probs[vox] = 1.0f / (1.0f + expf(-z));
    }
  }
}

}  // namespace cvit

using namespace cvit;

extern "C" {

int cvit_features_to_ndhwc_bf16(const void* features_f16, void* out_bf16, int64_t C, int64_t DHW, void* stream) {
  if (!features_f16 || !out_bf16 || C <= 0 || DHW <= 0) {
    set_error("features_to_ndhwc: bad arguments");
    return CVIT_ERR_INVALID;
  }
  dim3 grid((unsigned)((DHW + 63) / 64), (unsigned)((C + 63) / 64));
  const bool vec = C % 64 == 0 && DHW % 64 == 0 &&
                   ((reinterpret_cast<uintptr_t>(features_f16) | reinterpret_cast<uintptr_t>(out_bf16)) & 15u) == 0;
  if (vec)
    features_f16_to_ndhwc_vec_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
        static_cast<const __half*>(features_f16), static_cast<__nv_bfloat16*>(out_bf16), (int)C, DHW);
  else
    features_to_ndhwc_kernel<__half><<<grid, 256, 0, (cudaStream_t)stream>>>(
        static_cast<const __half*>(features_f16), static_cast<__nv_bfloat16*>(out_bf16), (int)C, DHW);
  return check_launch("features_to_ndhwc_kernel");
}

int cvit_features_f32_to_ndhwc_bf16(const float* features_f32, void* out_bf16, int64_t C, int64_t DHW, void* stream) {
  if (!features_f32 || !out_bf16 || C <= 0 || DHW <= 0) {
    set_error("features_f32_to_ndhwc: bad arguments");
    return CVIT_ERR_INVALID;
  }
  dim3 grid((unsigned)((DHW + 63) / 64), (unsigned)((C + 63) / 64));
  features_to_ndhwc_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(
      features_f32, static_cast<__nv_bfloat16*>(out_bf16), (int)C, DHW);
  return check_launch("features_to_ndhwc_kernel<float>");
}

int cvit_groupnorm_ndhwc_bf16(const void* x, void* out, const float* gamma, const float* beta, float* stats,
                              int64_t DHW, int64_t C, int64_t G, float eps, void* stream) {
  if (!x || !out || !gamma || !beta || !stats || DHW <= 0 || C <= 0 || G <= 0 || (C % 8) || (C % G)) {
    set_error("groupnorm: bad arguments");
    return CVIT_ERR_INVALID;
  }
  const int cpg = (int)(C / G);
  const int nvec = (int)(C / 8);
  if (!(cpg == 4 || (cpg % 8) == 0) || nvec > 256 || (256 % nvec) != 0) {
    set_error("groupnorm: C=%lld G=%lld unsupported (channels per group must be 4 or a multiple of 8; C / 8 a divisor of 256)",
              (long long)C, (long long)G);
    return CVIT_ERR_UNSUPPORTED;
  }
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(stats, 0, 2 * G * sizeof(float), st);
  if (e != cudaSuccess) {
    set_error("groupnorm: memset: %s", cudaGetErrorString(e));
    return CVIT_ERR_CUDA;
  }
  int blocks = num_sms() * 8;
  int64_t rows_per_block = (DHW + blocks - 1) / blocks;
  if (rows_per_block < 1) rows_per_block = 1;
  blocks = (int)((DHW + rows_per_block - 1) / rows_per_block);
  groupnorm_stats_kernel<<<blocks, 256, 2 * G * sizeof(float), st>>>(static_cast<const __nv_bfloat16*>(x), stats, DHW,
                                                                     (int)C, (int)G, (int)rows_per_block);
  int rc = check_launch("groupnorm_stats_kernel");
  if (rc) return rc;
  const int64_t total = DHW * nvec;
  int64_t g2 = (total + 255) / 256;
  if (g2 > (int64_t)num_sms() * 16) g2 = (int64_t)num_sms() * 16;
  groupnorm_apply_kernel<<<(int)g2, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(x), static_cast<__nv_bfloat16*>(out),
                                                  gamma, beta, stats, DHW, (int)C, (int)G, eps);
  return check_launch("groupnorm_apply_kernel");
}

// Deterministic mode: the same two passes, the statistics as [blocks][2G] partial rows added in a fixed order.
static int groupnorm_stats_grid(int64_t DHW, int64_t* rpb_out) {
  int blocks = num_sms() * 8;
  int64_t rows_per_block = (DHW + blocks - 1) / blocks;
  if (rows_per_block < 1) rows_per_block = 1;
  *rpb_out = rows_per_block;
  return (int)((DHW + rows_per_block - 1) / rows_per_block);
}

int64_t cvit_groupnorm_ndhwc_bf16_det_partials(int64_t DHW, int64_t C, int64_t G) {
  int64_t rpb;
  return DHW > 0 && C > 0 && G > 0 ? (int64_t)groupnorm_stats_grid(DHW, &rpb) * 2 * G : 0;
}

int cvit_groupnorm_ndhwc_bf16_det(const void* x, void* out, const float* gamma, const float* beta, float* stats, int64_t DHW, int64_t C,
                                  int64_t G, float eps, float* scratch, int64_t scratch_elems, void* stream) {
  if (!x || !out || !gamma || !beta || !stats || DHW <= 0 || C <= 0 || G <= 0 || (C % 8) || (C % G)) {
    set_error("groupnorm_det: bad arguments");
    return CVIT_ERR_INVALID;
  }
  const int cpg = (int)(C / G);
  const int nvec = (int)(C / 8);
  if (!(cpg == 4 || (cpg % 8) == 0) || nvec > 256 || (256 % nvec) != 0) {
    set_error("groupnorm_det: C=%lld G=%lld unsupported (channels per group must be 4 or a multiple of 8; C / 8 a divisor of 256)",
              (long long)C, (long long)G);
    return CVIT_ERR_UNSUPPORTED;
  }
  if (int rc = det_check_scratch(scratch, scratch_elems, cvit_groupnorm_ndhwc_bf16_det_partials(DHW, C, G), "groupnorm_det")) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  int64_t rows_per_block;
  const int blocks = groupnorm_stats_grid(DHW, &rows_per_block);
  groupnorm_stats_det_kernel<<<blocks, 256, 256 * 4 * sizeof(float), st>>>(static_cast<const __nv_bfloat16*>(x), scratch, DHW, (int)C,
                                                                          (int)G, (int)rows_per_block);
  if (int rc = check_launch("groupnorm_stats_det_kernel")) return rc;
  if (int rc = det_finalize(scratch, blocks, 2 * G, 2 * G, stats, false, st)) return rc;
  const int64_t total = DHW * nvec;
  int64_t g2 = (total + 255) / 256;
  if (g2 > (int64_t)num_sms() * 16) g2 = (int64_t)num_sms() * 16;
  groupnorm_apply_kernel<<<(int)g2, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(x), static_cast<__nv_bfloat16*>(out), gamma, beta,
                                                  stats, DHW, (int)C, (int)G, eps);
  return check_launch("groupnorm_apply_kernel");
}

int cvit_head_tail_fused(const void* x, const float* w1, const float* b1, const float* w2, const float* b2,
                         float* logits, float* probs, void* scratch_bf16, int64_t D, int64_t H, int64_t W,
                         void* stream) {
  if (!x || !w1 || !b1 || !w2 || !b2 || !scratch_bf16 || D <= 0 || H <= 0 || W <= 0 || (!logits && !probs)) {
    set_error("head_tail: bad arguments");
    return CVIT_ERR_INVALID;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int halo = 3 * (TAIL_TH + 2) * (TAIL_TW + 2) * 16;
  const int smem1 = halo + 27 * 8 * 8 * 4, smem2 = halo + 27 * 8 * 4;
  static bool configured = false;
  if (!configured) {
    cudaError_t e1 = cudaFuncSetAttribute(tail_conv_kernel<8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem1);
    cudaError_t e2 = cudaFuncSetAttribute(tail_conv_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem2);
    if (e1 != cudaSuccess || e2 != cudaSuccess) {
      set_error("head_tail: cudaFuncSetAttribute failed");
      return CVIT_ERR_CUDA;
    }
    configured = true;
  }
  const int64_t blocks = D * ((H + TAIL_TH - 1) / TAIL_TH) * ((W + TAIL_TW - 1) / TAIL_TW);
  tail_conv_kernel<8, false><<<(unsigned)blocks, 256, smem1, st>>>(static_cast<const __nv_bfloat16*>(x), w1, b1,
                                                                    static_cast<__nv_bfloat16*>(scratch_bf16), nullptr,
                                                                    nullptr, (int)D, (int)H, (int)W);
  int rc = check_launch("tail_conv_kernel<8>");
  if (rc) return rc;
  tail_conv_kernel<1, true><<<(unsigned)blocks, 256, smem2, st>>>(static_cast<const __nv_bfloat16*>(scratch_bf16), w2, b2,
                                                                   nullptr, logits, probs, (int)D, (int)H, (int)W);
  return check_launch("tail_conv_kernel<1>");
}

// The last convolution alone: Conv3d(8 -> 1, k3) + clip(-5, 5) [+ sigmoid] in fp32 on the CUDA cores (the 8 -> 8
// convolution before it runs on tensor cores, cvit_conv3d_halo_ndhwc): models/cryovit.py:33,39,49.
int cvit_head_out_conv(const void* x, const float* w2, const float* b2, float* logits, float* probs, int64_t D, int64_t H,
                       int64_t W, void* stream) {
  if (!x || !w2 || !b2 || D <= 0 || H <= 0 || W <= 0 || (!logits && !probs)) {
    set_error("head_out_conv: bad arguments");
    return CVIT_ERR_INVALID;
  }
  const int smem2 = 3 * (TAIL_TH + 2) * (TAIL_TW + 2) * 16 + 27 * 8 * 4;
  static bool configured = false;
  if (!configured) {
    if (cudaFuncSetAttribute(tail_conv_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem2) != cudaSuccess) {
      set_error("head_out_conv: cudaFuncSetAttribute failed");
      return CVIT_ERR_CUDA;
    }
    configured = true;
  }
  const int64_t blocks = D * ((H + TAIL_TH - 1) / TAIL_TH) * ((W + TAIL_TW - 1) / TAIL_TW);
  tail_conv_kernel<1, true><<<(unsigned)blocks, 256, smem2, (cudaStream_t)stream>>>(
      static_cast<const __nv_bfloat16*>(x), w2, b2, nullptr, logits, probs, (int)D, (int)H, (int)W);
  return check_launch("tail_conv_kernel<1>");
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// Masked segmentation statistics in one pass over the volume: everything DiceLoss (losses.py:17-32),
// DiceMetric (metrics.py:30-53) and F1Metric (metrics.py:69-93) reduce over, restricted to voxels whose label is
// > -1 (BaseModel._masked_predict, base_model.py:91-112). out[8] (fp64, accumulated with atomics, caller zeroes):
//   0 sum p   1 sum y   2 sum p*y                          (DiceLoss)
//   3 sum y*[p >= thr]   4 sum [p >= thr]                  (DiceMetric: "pred < thr -> 0 else 1")
//   5 sum y*[p > .5]   6 sum (1-y)*[p > .5]   7 sum y*(1-[p > .5])     (F1Metric: strict ">")
namespace cvit {
// DET (deterministic mode): out is a [gridDim.x][8] partial slab, one row per block, added by rows8_score_finalize.
template <bool DET>
__device__ __forceinline__ void seg_stats_body(const float* __restrict__ probs, const float* __restrict__ labels, int64_t n, float thr,
                                               double* __restrict__ out) {
  float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float y = labels[i], p = probs[i];
    if (y > -1.0f) {
      const float hge = p >= thr ? 1.f : 0.f, hgt = p > 0.5f ? 1.f : 0.f;
      v[0] += p;
      v[1] += y;
      v[2] += p * y;
      v[3] += y * hge;
      v[4] += hge;
      v[5] += y * hgt;
      v[6] += (1.f - y) * hgt;
      v[7] += y * (1.f - hgt);
    }
  }
  __shared__ double red[8][8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    double t = v[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = t;
  }
  __syncthreads();
  if (threadIdx.x < 8) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += red[threadIdx.x][w];
    if constexpr (DET) {
      out[(size_t)blockIdx.x * 8 + threadIdx.x] = t;
    } else {
      atomicAdd(out + threadIdx.x, t);
    }
  }
}

__global__ void __launch_bounds__(256) seg_stats_kernel(const float* __restrict__ probs, const float* __restrict__ labels,
                                                        int64_t n, float thr, double* __restrict__ out) {
  seg_stats_body<false>(probs, labels, n, thr, out);
}

__global__ void __launch_bounds__(256) seg_stats_det_kernel(const float* __restrict__ probs, const float* __restrict__ labels,
                                                            int64_t n, float thr, double* __restrict__ partials) {
  seg_stats_body<true>(probs, labels, n, thr, partials);
}

static int64_t seg_stats_grid(int64_t n) {
  int64_t blocks = (n + 256 * 16 - 1) / (256 * 16);
  const int64_t cap = (int64_t)num_sms() * 8;
  return blocks > cap ? cap : blocks;
}
}  // namespace cvit

extern "C" int cvit_seg_stats(const float* probs, const float* labels, int64_t n, float threshold, double* out8,
                              void* stream) {
  if (!probs || !labels || !out8 || n <= 0) {
    cvit::set_error("seg_stats: bad arguments");
    return cvit::CVIT_ERR_INVALID;
  }
  int64_t blocks = (n + 256 * 16 - 1) / (256 * 16);
  const int64_t cap = (int64_t)cvit::num_sms() * 8;
  if (blocks > cap) blocks = cap;
  cvit::seg_stats_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(probs, labels, n, threshold, out8);
  return cvit::check_launch("seg_stats_kernel");
}

extern "C" int64_t cvit_seg_stats_det_partials(int64_t n) { return n > 0 ? cvit::seg_stats_grid(n) * 8 : 0; }

// Deterministic mode: out8 is OVERWRITTEN with the fixed-order sum of one fp64 row of 8 per block (scratch: doubles).
extern "C" int cvit_seg_stats_det(const float* probs, const float* labels, int64_t n, float threshold, double* out8, double* scratch,
                                  int64_t scratch_elems, void* stream) {
  if (!probs || !labels || !out8 || n <= 0) {
    cvit::set_error("seg_stats_det: bad arguments");
    return cvit::CVIT_ERR_INVALID;
  }
  if (int rc = cvit::det_check_scratch(scratch, scratch_elems, cvit_seg_stats_det_partials(n), "seg_stats_det")) return rc;
  const int64_t blocks = cvit::seg_stats_grid(n);
  cvit::seg_stats_det_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(probs, labels, n, threshold, scratch);
  if (int rc = cvit::check_launch("seg_stats_det_kernel")) return rc;
  return cvit::rows8_score_finalize(scratch, (int)blocks, out8, (cudaStream_t)stream);
}

