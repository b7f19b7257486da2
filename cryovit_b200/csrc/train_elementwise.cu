// HBM-bound kernels of CryoVIT head TRAINING (BASELINE config 5; reference models/base_model.py:58-63,91-164,
// models/losses.py:17-32, configs/trainer/fit.yaml): activation forward/backward, Dice-loss gradient through the
// sigmoid and the clip, GroupNorm backward, bias gradients, the pixel un-shuffle that turns the transposed
// convolution's input gradient into a GEMM, and AdamW. The tensor-core work (dgrad = the forward convolution
// kernels run on flipped / transposed weights, wgrad = csrc/wgrad.cu) lives elsewhere.
#include "det_reduce.cuh"
#include "ptx.cuh"
#include "tmap.h"

namespace cvit {

static int ew_grid(int64_t n, int per_thread = 8) {
  int64_t b = (n + 256 * per_thread - 1) / (256 * per_thread);
  const int64_t cap = (int64_t)num_sms() * 16;
  if (b > cap) b = cap;
  return (int)(b < 1 ? 1 : b);
}

// a = gelu(z), 8 bf16 per thread-iteration
__global__ void __launch_bounds__(256) gelu_fwd_kernel(const uint4* __restrict__ z, uint4* __restrict__ a, int64_t nvec) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    const uint4 raw = z[i];
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw);
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 f = __bfloat1622float2(h[k]);
      o[k] = pack_bf16x2(gelu_erf(f.x), gelu_erf(f.y));
    }
    a[i] = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// dz = da * gelu'(z)
__global__ void __launch_bounds__(256) gelu_bwd_kernel(const uint4* __restrict__ da, const uint4* __restrict__ z,
                                                        uint4* __restrict__ dz, int64_t nvec) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    const uint4 rg = da[i], rz = z[i];
    const __nv_bfloat162* g = reinterpret_cast<const __nv_bfloat162*>(&rg);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&rz);
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 fg = __bfloat1622float2(g[k]), fz = __bfloat1622float2(h[k]);
      o[k] = pack_bf16x2(fg.x * gelu_grad(fz.x), fg.y * gelu_grad(fz.y));
    }
    dz[i] = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// The same with the bias gradient db[c] += sum over rows of dz[r, c] accumulated on the way (the column sums of dz that
// every convolution's bias gradient is): thread t owns the 8-channel vector t % (C/8) and strides over the rows of its
// block's range, so the partial sums stay in registers; one shared-memory and one global atomic pass per block.
// W2 > 0: the rows are the voxels of a [D, H2, W2, C] volume (H2, W2 even) and dz is written PIXEL-UNSHUFFLED, as
// [D, H2/2, W2/2, (i, j, C)] with (i, j) the sub-pixel -- the row layout the transposed convolution's input-gradient and
// weight-gradient GEMMs read -- instead of through a separate permutation pass over the largest gradient volumes.
// DET (deterministic mode): no atomics; db is a [gridDim.x][C] partial slab, one fixed-order row per block.
template <bool DET>
__device__ __forceinline__ void gelu_bwd_colsum_body(const uint4* __restrict__ da, const uint4* __restrict__ z, uint4* __restrict__ dz,
                                                     float* __restrict__ db, int64_t R, int C, int64_t rows_per_block, int W2) {
  extern __shared__ float s_db[];  // [C] | DET: [256][8]
  if constexpr (!DET) {
    for (int i = threadIdx.x; i < C; i += blockDim.x) s_db[i] = 0.f;
    __syncthreads();
  }
  const int nvec = C / 8;
  const int vec = threadIdx.x % nvec, rsub = threadIdx.x / nvec, rstep = blockDim.x / nvec;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r1 = r0 + rows_per_block < R ? r0 + rows_per_block : R;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (rsub < rstep) {
    for (int64_t r = r0 + rsub; r < r1; r += rstep) {
      const int64_t i = r * nvec + vec;
      const uint4 rg = da[i], rz = z[i];
      const __nv_bfloat162* g = reinterpret_cast<const __nv_bfloat162*>(&rg);
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&rz);
      uint32_t o[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 fg = __bfloat1622float2(g[k]), fz = __bfloat1622float2(h[k]);
        const __nv_bfloat162 d2 = __floats2bfloat162_rn(fg.x * gelu_grad(fz.x), fg.y * gelu_grad(fz.y));
        o[k] = *reinterpret_cast<const uint32_t*>(&d2);
        const float2 dr = __bfloat1622float2(d2);  // the sums are over the STORED (bf16) gradient, as a separate pass would see it
        acc[2 * k] += dr.x;
        acc[2 * k + 1] += dr.y;
      }
      int64_t io = i;
      if (W2 > 0) {
        const int64_t dh2 = r / W2;
        const int wx = (int)(r - dh2 * W2);
        io = (((dh2 >> 1) * (W2 >> 1) + (wx >> 1)) * 4 + ((dh2 & 1) * 2 + (wx & 1))) * nvec + vec;
      }
      dz[io] = make_uint4(o[0], o[1], o[2], o[3]);
    }
    if constexpr (DET) {
#pragma unroll
      for (int k = 0; k < 8; ++k) s_db[threadIdx.x * 8 + k] = acc[k];
    } else {
#pragma unroll
      for (int k = 0; k < 8; ++k) atomicAdd(&s_db[vec * 8 + k], acc[k]);
    }
  }
  __syncthreads();
  if constexpr (DET) {
    det_block_colsum(s_db, C, nvec, rstep * nvec, 0, db + (size_t)blockIdx.x * C);
  } else {
    for (int i = threadIdx.x; i < C; i += blockDim.x) atomicAdd(db + i, s_db[i]);
  }
}

__global__ void __launch_bounds__(256) gelu_bwd_colsum_kernel(const uint4* __restrict__ da, const uint4* __restrict__ z,
                                                               uint4* __restrict__ dz, float* __restrict__ db, int64_t R, int C,
                                                               int64_t rows_per_block, int W2) {
  gelu_bwd_colsum_body<false>(da, z, dz, db, R, C, rows_per_block, W2);
}

__global__ void __launch_bounds__(256) gelu_bwd_colsum_det_kernel(const uint4* __restrict__ da, const uint4* __restrict__ z,
                                                                   uint4* __restrict__ dz, float* __restrict__ db_partials, int64_t R,
                                                                   int C, int64_t rows_per_block, int W2) {
  gelu_bwd_colsum_body<true>(da, z, dz, db_partials, R, C, rows_per_block, W2);
}

// Dice loss L = 1 - 2 I / (Sy + Sp + eps) over the voxels with label > -1, p = sigmoid(clip(x, -5, 5)):
//   dL/dp = -2 (y (Sy + Sp + eps) - I) / (Sy + Sp + eps)^2 ;  dp/dx = p (1 - p) inside the clip, 0 on it.
// stats = the fp64 sums of cvit_seg_stats ({Sp, Sy, I, ...}) of the SAME forward pass, read on the device.
// The gradient is written as an 8-channel bf16 voxel (channel 0 = dL/dx * scale, channels 1..7 = 0): the operand
// format of the narrow-layer convolution kernel that back-propagates it through output_layer.2.
__global__ void __launch_bounds__(256) dice_bwd_kernel(const float* __restrict__ logits, const float* __restrict__ probs,
                                                        const float* __restrict__ labels, const double* __restrict__ stats,
                                                        float scale, uint4* __restrict__ dlogit8, int64_t n) {
  const float S = (float)(stats[0] + stats[1] + 1e-3), I = (float)stats[2];
  const float inv = 1.0f / (S * S);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float y = labels[i], p = probs[i], x = logits[i];
    float g = 0.f;
    if (y > -1.0f && fabsf(x) < 5.0f) g = -2.0f * (y * S - I) * inv * p * (1.0f - p) * scale;
    dlogit8[i] = make_uint4(pack_bf16x2(g, 0.f), 0u, 0u, 0u);
  }
}

// column sums of a bf16 [R, C] matrix into fp32 [C] (bias gradients; caller zeroes `out`). C multiple of 8, <= 2048.
// DET: out is a [gridDim.x][C] partial slab, one fixed-order row per block.
template <bool DET>
__device__ __forceinline__ void colsum_body(const __nv_bfloat16* __restrict__ x, float* __restrict__ out, int64_t R, int C,
                                            int64_t rows_per_block) {
  extern __shared__ float s_acc[];  // [C] | DET: [256][8]
  if constexpr (!DET) {
    for (int i = threadIdx.x; i < C; i += blockDim.x) s_acc[i] = 0.f;
    __syncthreads();
  }
  const int nvec = C / 8;
  const int vec = threadIdx.x % nvec, rsub = threadIdx.x / nvec, rstep = blockDim.x / nvec;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block, r1 = min(r0 + rows_per_block, R);
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (rsub < rstep) {
    for (int64_t r = r0 + rsub; r < r1; r += rstep) {
      const uint4 raw = *reinterpret_cast<const uint4*>(x + r * C + vec * 8);
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 f = __bfloat1622float2(h[k]);
        acc[2 * k] += f.x;
        acc[2 * k + 1] += f.y;
      }
    }
    if constexpr (DET) {
#pragma unroll
      for (int k = 0; k < 8; ++k) s_acc[threadIdx.x * 8 + k] = acc[k];
    } else {
#pragma unroll
      for (int k = 0; k < 8; ++k) atomicAdd(&s_acc[vec * 8 + k], acc[k]);
    }
  }
  __syncthreads();
  if constexpr (DET) {
    det_block_colsum(s_acc, C, nvec, rstep * nvec, 0, out + (size_t)blockIdx.x * C);
  } else {
    for (int i = threadIdx.x; i < C; i += blockDim.x) atomicAdd(out + i, s_acc[i]);
  }
}

__global__ void __launch_bounds__(256) colsum_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ out,
                                                      int64_t R, int C, int64_t rows_per_block) {
  colsum_body<false>(x, out, R, C, rows_per_block);
}

__global__ void __launch_bounds__(256) colsum_det_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ partials,
                                                          int64_t R, int C, int64_t rows_per_block) {
  colsum_body<true>(x, partials, R, C, rows_per_block);
}

// GroupNorm backward, pass 1: per channel  A_c = sum dy * xhat,  B_c = sum dy  (these ARE dgamma and dbeta).
// xhat = (x - mean_g) * rstd_g from the forward statistics (sum, sum of squares per group).
// DET: dgamma is a [gridDim.x][2C] partial slab (row = A then B), dbeta unused; one fixed-order row per block.
template <bool DET>
__device__ __forceinline__ void groupnorm_bwd_reduce_body(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ dy,
                                                          const float* __restrict__ stats, float* __restrict__ dgamma,
                                                          float* __restrict__ dbeta, int64_t DHW, int C, int G, float eps,
                                                          int64_t rows_per_block) {
  extern __shared__ float s_ab[];  // [2][C] | DET: [2][256][8]
  if constexpr (!DET) {
    for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) s_ab[i] = 0.f;
    __syncthreads();
  }
  const int nvec = C / 8, cpg = C / G;
  const float inv_n = 1.0f / (static_cast<float>(DHW) * cpg);
  const int vec = threadIdx.x % nvec, rsub = threadIdx.x / nvec, rstep = blockDim.x / nvec;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block, r1 = min(r0 + rows_per_block, DHW);
  float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, b[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (rsub < rstep) {
    float mean[8], rstd[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int g = (vec * 8 + k) / cpg;
      mean[k] = stats[g] * inv_n;
      rstd[k] = rsqrtf(fmaxf(stats[G + g] * inv_n - mean[k] * mean[k], 0.f) + eps);
    }
    for (int64_t r = r0 + rsub; r < r1; r += rstep) {
      const uint4 rx = *reinterpret_cast<const uint4*>(x + r * C + vec * 8);
      const uint4 rd = *reinterpret_cast<const uint4*>(dy + r * C + vec * 8);
      const __nv_bfloat162* hx = reinterpret_cast<const __nv_bfloat162*>(&rx);
      const __nv_bfloat162* hd = reinterpret_cast<const __nv_bfloat162*>(&rd);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 fx = __bfloat1622float2(hx[k]), fd = __bfloat1622float2(hd[k]);
        a[2 * k] += fd.x * (fx.x - mean[2 * k]) * rstd[2 * k];
        a[2 * k + 1] += fd.y * (fx.y - mean[2 * k + 1]) * rstd[2 * k + 1];
        b[2 * k] += fd.x;
        b[2 * k + 1] += fd.y;
      }
    }
    if constexpr (DET) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        s_ab[threadIdx.x * 8 + k] = a[k];
        s_ab[256 * 8 + threadIdx.x * 8 + k] = b[k];
      }
    } else {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        atomicAdd(&s_ab[vec * 8 + k], a[k]);
        atomicAdd(&s_ab[C + vec * 8 + k], b[k]);
      }
    }
  }
  __syncthreads();
  if constexpr (DET) {
    float* row = dgamma + (size_t)blockIdx.x * 2 * C;
    det_block_colsum(s_ab, C, nvec, rstep * nvec, 0, row);
    det_block_colsum(s_ab + 256 * 8, C, nvec, rstep * nvec, 0, row + C);
  } else {
    for (int i = threadIdx.x; i < C; i += blockDim.x) {
      atomicAdd(dgamma + i, s_ab[i]);
      atomicAdd(dbeta + i, s_ab[C + i]);
    }
  }
}

__global__ void __launch_bounds__(256) groupnorm_bwd_reduce_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ dy,
                                                                    const float* __restrict__ stats, float* __restrict__ dgamma,
                                                                    float* __restrict__ dbeta, int64_t DHW, int C, int G, float eps,
                                                                    int64_t rows_per_block) {
  groupnorm_bwd_reduce_body<false>(x, dy, stats, dgamma, dbeta, DHW, C, G, eps, rows_per_block);
}

__global__ void __launch_bounds__(256) groupnorm_bwd_reduce_det_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ dy,
                                                                        const float* __restrict__ stats, float* __restrict__ partials,
                                                                        int64_t DHW, int C, int G, float eps, int64_t rows_per_block) {
  groupnorm_bwd_reduce_body<true>(x, dy, stats, partials, nullptr, DHW, C, G, eps, rows_per_block);
}

// pass 2: dx = rstd_g * ( gamma_c dy - ( s1_g + xhat s2_g ) / N_g ),  s1_g = sum_c gamma_c B_c, s2_g = sum_c gamma_c A_c
// DET (z != null only): db is a [gridDim.x][C] partial slab, one fixed-order row per block.
template <bool DET>
__device__ __forceinline__ void groupnorm_bwd_apply_body(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ dy,
                                                         __nv_bfloat16* __restrict__ dx, const float* __restrict__ gamma,
                                                         const float* __restrict__ stats, const float* __restrict__ dgamma,
                                                         const float* __restrict__ dbeta, int64_t DHW, int C, int G, float eps,
                                                         const __nv_bfloat16* __restrict__ z, float* __restrict__ db, int W2) {
  // z != null: the GroupNorm's input was gelu(z) (the block before ends in a transposed convolution + GELU, or the
  // projection + GELU): the result is multiplied by gelu'(z) right here -- dx is then the gradient of z -- its column sums
  // (that layer's bias gradient) go to db, and with W2 > 0 it is stored pixel-unshuffled ([D, H2/2, W2/2, 4C], see
  // gelu_bwd_colsum_kernel): one pass instead of two over the step's largest gradient volumes.
  extern __shared__ float s_g[];  // [4][G]: mean, rstd, s1/N, s2/N | z != null: + [C] column sums (DET: + [256][8])
  const int cpg = C / G;
  const float inv_n = 1.0f / (static_cast<float>(DHW) * cpg);
  for (int g = threadIdx.x; g < G; g += blockDim.x) {
    const float mean = stats[g] * inv_n;
    const float rstd = rsqrtf(fmaxf(stats[G + g] * inv_n - mean * mean, 0.f) + eps);
    float s1 = 0.f, s2 = 0.f;
    for (int c = g * cpg; c < (g + 1) * cpg; ++c) {
      s1 += gamma[c] * dbeta[c];
      s2 += gamma[c] * dgamma[c];
    }
    s_g[g] = mean;
    s_g[G + g] = rstd;
    s_g[2 * G + g] = s1 * inv_n;
    s_g[3 * G + g] = s2 * inv_n;
  }
  __syncthreads();
  const int nvec = C / 8;
  const int64_t total = DHW * nvec;
  float* s_db = s_g + 4 * G;
  if (!DET && z)
    for (int i = threadIdx.x; i < C; i += blockDim.x) s_db[i] = 0.f;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // this thread's 8 channels (the grid stride is a multiple of nvec)
  __syncthreads();
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int vec = (int)(idx % nvec);
    const uint4 rx = *reinterpret_cast<const uint4*>(x + idx * 8);
    const uint4 rd = *reinterpret_cast<const uint4*>(dy + idx * 8);
    uint4 rz = make_uint4(0u, 0u, 0u, 0u);
    if (z) rz = *reinterpret_cast<const uint4*>(z + idx * 8);
    const __nv_bfloat162* hz = reinterpret_cast<const __nv_bfloat162*>(&rz);
    const __nv_bfloat162* hx = reinterpret_cast<const __nv_bfloat162*>(&rx);
    const __nv_bfloat162* hd = reinterpret_cast<const __nv_bfloat162*>(&rd);
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int c = vec * 8 + 2 * k;
      const int g0 = c / cpg, g1 = (c + 1) / cpg;
      const float2 fx = __bfloat1622float2(hx[k]), fd = __bfloat1622float2(hd[k]);
      const float xh0 = (fx.x - s_g[g0]) * s_g[G + g0], xh1 = (fx.y - s_g[g1]) * s_g[G + g1];
      const float d0 = s_g[G + g0] * (__ldg(gamma + c) * fd.x - (s_g[2 * G + g0] + xh0 * s_g[3 * G + g0]));
      const float d1 = s_g[G + g1] * (__ldg(gamma + c + 1) * fd.y - (s_g[2 * G + g1] + xh1 * s_g[3 * G + g1]));
      if (z) {
        const float2 fz = __bfloat1622float2(hz[k]);
        const __nv_bfloat162 d2 = __floats2bfloat162_rn(d0 * gelu_grad(fz.x), d1 * gelu_grad(fz.y));
        o[k] = *reinterpret_cast<const uint32_t*>(&d2);
        const float2 dr = __bfloat1622float2(d2);  // sums over the STORED gradient, as the separate pass computes them
        acc[2 * k] += dr.x;
        acc[2 * k + 1] += dr.y;
      } else {
        o[k] = pack_bf16x2(d0, d1);
      }
    }
    int64_t io = idx;
    if (W2 > 0) {
      const int64_t r = idx / nvec, dh2 = r / W2;
      const int wx = (int)(r - dh2 * W2);
      io = (((dh2 >> 1) * (W2 >> 1) + (wx >> 1)) * 4 + ((dh2 & 1) * 2 + (wx & 1))) * nvec + vec;
    }
    *reinterpret_cast<uint4*>(dx + io * 8) = make_uint4(o[0], o[1], o[2], o[3]);
  }
  if constexpr (DET) {
    if (z) {
#pragma unroll
      for (int k = 0; k < 8; ++k) s_db[threadIdx.x * 8 + k] = acc[k];
      __syncthreads();
      det_block_colsum(s_db, C, nvec, blockDim.x, (int)(((int64_t)blockIdx.x * blockDim.x) % nvec), db + (size_t)blockIdx.x * C);
    }
  } else if (z) {
    const int vec = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) % nvec);
#pragma unroll
    for (int k = 0; k < 8; ++k) atomicAdd(&s_db[vec * 8 + k], acc[k]);
    __syncthreads();
    for (int i = threadIdx.x; i < C; i += blockDim.x) atomicAdd(db + i, s_db[i]);
  }
}

__global__ void __launch_bounds__(256) groupnorm_bwd_apply_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ dy,
                                                                   __nv_bfloat16* __restrict__ dx, const float* __restrict__ gamma,
                                                                   const float* __restrict__ stats, const float* __restrict__ dgamma,
                                                                   const float* __restrict__ dbeta, int64_t DHW, int C, int G, float eps,
                                                                   const __nv_bfloat16* __restrict__ z, float* __restrict__ db, int W2) {
  groupnorm_bwd_apply_body<false>(x, dy, dx, gamma, stats, dgamma, dbeta, DHW, C, G, eps, z, db, W2);
}

__global__ void __launch_bounds__(256) groupnorm_bwd_apply_det_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ dy,
                                                                       __nv_bfloat16* __restrict__ dx, const float* __restrict__ gamma,
                                                                       const float* __restrict__ stats, const float* __restrict__ dgamma,
                                                                       const float* __restrict__ dbeta, int64_t DHW, int C, int G, float eps,
                                                                       const __nv_bfloat16* __restrict__ z, float* __restrict__ db_partials,
                                                                       int W2) {
  groupnorm_bwd_apply_body<true>(x, dy, dx, gamma, stats, dgamma, dbeta, DHW, C, G, eps, z, db_partials, W2);
}

// [D, 2H, 2W, C] -> [D, H, W, 4C], column (i*2 + j) * C + c : the transposed convolution's output gradient as rows of
// the GEMM that gives its input gradient (and, channels-first, its weight gradient). C multiple of 8.
__global__ void __launch_bounds__(256) pixel_unshuffle_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, int D, int H,
                                                               int W, int C8) {
  const int64_t total = (int64_t)D * H * W * 4 * C8;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(idx % C8);
    int64_t r = idx / C8;
    const int ij = (int)(r % 4);
    r /= 4;
    const int w = (int)(r % W);
    r /= W;
    const int h = (int)(r % H), d = (int)(r / H);
    const int64_t s = (((int64_t)d * 2 * H + 2 * h + (ij >> 1)) * (2 * W) + 2 * w + (ij & 1)) * C8 + c;
    dst[idx] = src[s];
  }
}

// AdamW (torch.optim.AdamW semantics, base_model.py:58-63: lr 1e-4, weight decay 1e-3, betas (0.9, 0.999), eps 1e-8):
//   p <- p (1 - lr wd);  m <- b1 m + (1 - b1) g;  v <- b2 v + (1 - b2) g^2;  p <- p - lr/bc1 * m / (sqrt(v)/sqrt(bc2) + eps)
__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                     float* __restrict__ v, int64_t n, float lr, float b1, float b2, float eps,
                                                     float wd, float bc1, float rsqrt_bc2, float gscale) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = g[i] * gscale;
    const float mi = b1 * m[i] + (1.0f - b1) * gi;
    const float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) * rsqrt_bc2 + eps;
    p[i] = p[i] * (1.0f - lr * wd) - (lr / bc1) * (mi / denom);
  }
}

}  // namespace cvit

using namespace cvit;

extern "C" {

int cvit_gelu_fwd_bf16(const void* z, void* a, int64_t n, void* stream) {
  if (!z || !a || n <= 0 || (n % 8)) { set_error("gelu_fwd: bad arguments"); return CVIT_ERR_INVALID; }
  gelu_fwd_kernel<<<ew_grid(n / 8, 4), 256, 0, (cudaStream_t)stream>>>(static_cast<const uint4*>(z), static_cast<uint4*>(a), n / 8);
  return check_launch("gelu_fwd_kernel");
}

int cvit_gelu_bwd_bf16(const void* da, const void* z, void* dz, int64_t n, void* stream) {
  if (!da || !z || !dz || n <= 0 || (n % 8)) { set_error("gelu_bwd: bad arguments"); return CVIT_ERR_INVALID; }
  gelu_bwd_kernel<<<ew_grid(n / 8, 4), 256, 0, (cudaStream_t)stream>>>(static_cast<const uint4*>(da), static_cast<const uint4*>(z),
                                                                       static_cast<uint4*>(dz), n / 8);
  return check_launch("gelu_bwd_kernel");
}

// dz = da * gelu'(z) over a bf16 [R, C] matrix and db[c] += sum_r dz[r, c] (fp32 [C], caller zeroes); C % 8 == 0, C <= 2048.
static int gelu_bwd_colsum_launch(const void* da, const void* z, void* dz, float* db, int64_t R, int64_t C, int W2, void* stream) {
  if (!da || !z || !dz || !db || R <= 0 || C <= 0 || (C % 8) || C > 2048) { set_error("gelu_bwd_colsum: bad arguments"); return CVIT_ERR_INVALID; }
  int64_t blocks = (int64_t)num_sms() * 8;
  int64_t rpb = (R + blocks - 1) / blocks;
  if (rpb < 1) rpb = 1;
  blocks = (R + rpb - 1) / rpb;
  gelu_bwd_colsum_kernel<<<(unsigned)blocks, 256, C * sizeof(float), (cudaStream_t)stream>>>(
      static_cast<const uint4*>(da), static_cast<const uint4*>(z), static_cast<uint4*>(dz), db, R, (int)C, rpb, W2);
  return check_launch("gelu_bwd_colsum_kernel");
}

int cvit_gelu_bwd_colsum_bf16(const void* da, const void* z, void* dz, float* db, int64_t R, int64_t C, void* stream) {
  return gelu_bwd_colsum_launch(da, z, dz, db, R, C, 0, stream);
}

// The same over a [D, H2, W2, C] volume with dz stored pixel-unshuffled, [D, H2/2, W2/2, 4 C] (sub-pixel (i, j) major): the
// gradient of a transposed convolution's pre-activation in the row layout its GEMMs read (replaces the pass of
// cvit_pixel_unshuffle_1x2x2_bf16 over the step's largest gradient volumes).
int cvit_gelu_bwd_colsum_unshuffle_bf16(const void* da, const void* z, void* dzun, float* db, int64_t D, int64_t H2, int64_t W2,
                                        int64_t C, void* stream) {
  if (D <= 0 || H2 <= 0 || W2 <= 0 || (H2 & 1) || (W2 & 1)) { set_error("gelu_bwd_colsum_unshuffle: H2 and W2 must be even"); return CVIT_ERR_INVALID; }
  return gelu_bwd_colsum_launch(da, z, dzun, db, D * H2 * W2, C, (int)W2, stream);
}

// ---------------------------------------------------------------------------------------------- deterministic mode
// The column-sum kernels below have the grid of their default twins (num_sms() * 8 blocks of rows_per_block rows); each
// block writes one [C] row of the scratch slab and det_finalize adds the rows in order (csrc/det_reduce.cuh).
static int64_t colsum_grid(int64_t R, int64_t* rpb_out) {
  int64_t blocks = (int64_t)num_sms() * 8;
  int64_t rpb = (R + blocks - 1) / blocks;
  if (rpb < 1) rpb = 1;
  *rpb_out = rpb;
  return (R + rpb - 1) / rpb;
}

int64_t cvit_colsum_bf16_det_partials(int64_t R, int64_t C) {
  int64_t rpb;
  return R > 0 && C > 0 ? colsum_grid(R, &rpb) * C : 0;
}

int cvit_colsum_bf16_det(const void* x, float* out, int64_t R, int64_t C, float* scratch, int64_t scratch_elems, void* stream) {
  if (!x || !out || R <= 0 || C <= 0 || (C % 8) || C > 2048) { set_error("colsum_det: bad arguments"); return CVIT_ERR_INVALID; }
  if (int rc = det_check_scratch(scratch, scratch_elems, cvit_colsum_bf16_det_partials(R, C), "colsum_det")) return rc;
  int64_t rpb;
  const int64_t blocks = colsum_grid(R, &rpb);
  colsum_det_kernel<<<(unsigned)blocks, 256, 256 * 8 * sizeof(float), (cudaStream_t)stream>>>(static_cast<const __nv_bfloat16*>(x), scratch,
                                                                                             R, (int)C, rpb);
  if (int rc = check_launch("colsum_det_kernel")) return rc;
  return det_finalize(scratch, blocks, C, C, out, true, (cudaStream_t)stream);
}

static int gelu_bwd_colsum_det_launch(const void* da, const void* z, void* dz, float* db, int64_t R, int64_t C, int W2, float* scratch,
                                      int64_t scratch_elems, void* stream) {
  if (!da || !z || !dz || !db || R <= 0 || C <= 0 || (C % 8) || C > 2048) { set_error("gelu_bwd_colsum_det: bad arguments"); return CVIT_ERR_INVALID; }
  if (int rc = det_check_scratch(scratch, scratch_elems, cvit_colsum_bf16_det_partials(R, C), "gelu_bwd_colsum_det")) return rc;
  int64_t rpb;
  const int64_t blocks = colsum_grid(R, &rpb);
  gelu_bwd_colsum_det_kernel<<<(unsigned)blocks, 256, 256 * 8 * sizeof(float), (cudaStream_t)stream>>>(
      static_cast<const uint4*>(da), static_cast<const uint4*>(z), static_cast<uint4*>(dz), scratch, R, (int)C, rpb, W2);
  if (int rc = check_launch("gelu_bwd_colsum_det_kernel")) return rc;
  return det_finalize(scratch, blocks, C, C, db, true, (cudaStream_t)stream);
}

int64_t cvit_gelu_bwd_colsum_bf16_det_partials(int64_t R, int64_t C) { return cvit_colsum_bf16_det_partials(R, C); }

int cvit_gelu_bwd_colsum_bf16_det(const void* da, const void* z, void* dz, float* db, int64_t R, int64_t C, float* scratch,
                                  int64_t scratch_elems, void* stream) {
  return gelu_bwd_colsum_det_launch(da, z, dz, db, R, C, 0, scratch, scratch_elems, stream);
}

int64_t cvit_gelu_bwd_colsum_unshuffle_bf16_det_partials(int64_t D, int64_t H2, int64_t W2, int64_t C) {
  return cvit_colsum_bf16_det_partials(D * H2 * W2, C);
}

int cvit_gelu_bwd_colsum_unshuffle_bf16_det(const void* da, const void* z, void* dzun, float* db, int64_t D, int64_t H2, int64_t W2,
                                            int64_t C, float* scratch, int64_t scratch_elems, void* stream) {
  if (D <= 0 || H2 <= 0 || W2 <= 0 || (H2 & 1) || (W2 & 1)) { set_error("gelu_bwd_colsum_unshuffle_det: H2 and W2 must be even"); return CVIT_ERR_INVALID; }
  return gelu_bwd_colsum_det_launch(da, z, dzun, db, D * H2 * W2, C, (int)W2, scratch, scratch_elems, stream);
}

int cvit_dice_bwd(const float* logits, const float* probs, const float* labels, const double* stats8, float scale,
                  void* dlogit8_bf16, int64_t n, void* stream) {
  if (!logits || !probs || !labels || !stats8 || !dlogit8_bf16 || n <= 0) { set_error("dice_bwd: bad arguments"); return CVIT_ERR_INVALID; }
  dice_bwd_kernel<<<ew_grid(n, 4), 256, 0, (cudaStream_t)stream>>>(logits, probs, labels, stats8, scale,
                                                                   static_cast<uint4*>(dlogit8_bf16), n);
  return check_launch("dice_bwd_kernel");
}

int cvit_colsum_bf16(const void* x, float* out, int64_t R, int64_t C, void* stream) {
  if (!x || !out || R <= 0 || C <= 0 || (C % 8) || C > 2048) { set_error("colsum: bad arguments"); return CVIT_ERR_INVALID; }
  int blocks = num_sms() * 8;
  int64_t rpb = (R + blocks - 1) / blocks;
  if (rpb < 1) rpb = 1;
  blocks = (int)((R + rpb - 1) / rpb);
  colsum_kernel<<<blocks, 256, C * sizeof(float), (cudaStream_t)stream>>>(static_cast<const __nv_bfloat16*>(x), out, R, (int)C, rpb);
  return check_launch("colsum_kernel");
}

int cvit_groupnorm_bwd_gelu_ndhwc_bf16(const void* x, const void* dy, void* dx, const float* gamma, const float* stats, float* dgamma,
                                       float* dbeta, int64_t DHW, int64_t C, int64_t G, float eps, const void* z, float* db,
                                       int64_t W2, void* stream);

int cvit_groupnorm_bwd_ndhwc_bf16(const void* x, const void* dy, void* dx, const float* gamma, const float* stats,
                                  float* dgamma, float* dbeta, int64_t DHW, int64_t C, int64_t G, float eps, void* stream) {
  return cvit_groupnorm_bwd_gelu_ndhwc_bf16(x, dy, dx, gamma, stats, dgamma, dbeta, DHW, C, G, eps, nullptr, nullptr, 0, stream);
}

// GroupNorm backward; with z (bf16, x's shape: x = gelu(z)) the result is d(z) = d(x) * gelu'(z), db (fp32 [C], zeroed by the
// caller) += its column sums, and W2 > 0 (x is a [D, H2, W2, C] volume, H2 and W2 even) stores it pixel-unshuffled.
int cvit_groupnorm_bwd_gelu_ndhwc_bf16(const void* x, const void* dy, void* dx, const float* gamma, const float* stats, float* dgamma,
                                       float* dbeta, int64_t DHW, int64_t C, int64_t G, float eps, const void* z, float* db,
                                       int64_t W2, void* stream) {
  if (!x || !dy || !dx || !gamma || !stats || !dgamma || !dbeta || DHW <= 0 || C <= 0 || G <= 0 || (C % 8) || (C % G) || C > 2048 ||
      (z && !db) || (!z && W2 != 0) || W2 < 0 || (W2 & 1) || (W2 > 0 && (DHW % (2 * W2)) != 0)) {
    set_error("groupnorm_bwd: bad arguments");
    return CVIT_ERR_INVALID;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (cudaMemsetAsync(dgamma, 0, C * sizeof(float), st) != cudaSuccess || cudaMemsetAsync(dbeta, 0, C * sizeof(float), st) != cudaSuccess) {
    set_error("groupnorm_bwd: memset failed");
    return CVIT_ERR_CUDA;
  }
  int blocks = num_sms() * 8;
  int64_t rpb = (DHW + blocks - 1) / blocks;
  if (rpb < 1) rpb = 1;
  blocks = (int)((DHW + rpb - 1) / rpb);
  groupnorm_bwd_reduce_kernel<<<blocks, 256, 2 * C * sizeof(float), st>>>(static_cast<const __nv_bfloat16*>(x),
                                                                          static_cast<const __nv_bfloat16*>(dy), stats, dgamma, dbeta,
                                                                          DHW, (int)C, (int)G, eps, rpb);
  int rc = check_launch("groupnorm_bwd_reduce_kernel");
  if (rc) return rc;
  groupnorm_bwd_apply_kernel<<<ew_grid(DHW * (C / 8), 4), 256, (4 * G + (z ? C : 0)) * sizeof(float), st>>>(
      static_cast<const __nv_bfloat16*>(x), static_cast<const __nv_bfloat16*>(dy), static_cast<__nv_bfloat16*>(dx), gamma, stats,
      dgamma, dbeta, DHW, (int)C, (int)G, eps, static_cast<const __nv_bfloat16*>(z), db, (int)W2);
  return check_launch("groupnorm_bwd_apply_kernel");
}

// Deterministic mode: the reduce pass writes [blocks][2C] rows (dgamma | dbeta), two finalizes write dgamma and dbeta; with z
// the apply pass writes [blocks][C] rows of db (the same scratch, reused after the first finalizes) and a third adds them.
static int64_t gn_bwd_reduce_grid(int64_t DHW, int64_t* rpb_out) { return colsum_grid(DHW, rpb_out); }

int64_t cvit_groupnorm_bwd_gelu_ndhwc_bf16_det_partials(int64_t DHW, int64_t C, int64_t G) {
  if (DHW <= 0 || C <= 0 || G <= 0) return 0;
  int64_t rpb;
  const int64_t a = gn_bwd_reduce_grid(DHW, &rpb) * 2 * C, b = (int64_t)ew_grid(DHW * (C / 8), 4) * C;
  return a > b ? a : b;
}

int cvit_groupnorm_bwd_gelu_ndhwc_bf16_det(const void* x, const void* dy, void* dx, const float* gamma, const float* stats, float* dgamma,
                                           float* dbeta, int64_t DHW, int64_t C, int64_t G, float eps, const void* z, float* db,
                                           int64_t W2, float* scratch, int64_t scratch_elems, void* stream) {
  if (!x || !dy || !dx || !gamma || !stats || !dgamma || !dbeta || DHW <= 0 || C <= 0 || G <= 0 || (C % 8) || (C % G) || C > 2048 ||
      (z && !db) || (!z && W2 != 0) || W2 < 0 || (W2 & 1) || (W2 > 0 && (DHW % (2 * W2)) != 0)) {
    set_error("groupnorm_bwd_det: bad arguments");
    return CVIT_ERR_INVALID;
  }
  if (int rc = det_check_scratch(scratch, scratch_elems, cvit_groupnorm_bwd_gelu_ndhwc_bf16_det_partials(DHW, C, G), "groupnorm_bwd_det"))
    return rc;
  cudaStream_t st = (cudaStream_t)stream;
  int64_t rpb;
  const int64_t blocks = gn_bwd_reduce_grid(DHW, &rpb);
  groupnorm_bwd_reduce_det_kernel<<<(unsigned)blocks, 256, 2 * 256 * 8 * sizeof(float), st>>>(
      static_cast<const __nv_bfloat16*>(x), static_cast<const __nv_bfloat16*>(dy), stats, scratch, DHW, (int)C, (int)G, eps, rpb);
  if (int rc = check_launch("groupnorm_bwd_reduce_det_kernel")) return rc;
  if (int rc = det_finalize(scratch, blocks, C, 2 * C, dgamma, false, st)) return rc;
  if (int rc = det_finalize(scratch + C, blocks, C, 2 * C, dbeta, false, st)) return rc;
  const int g2 = ew_grid(DHW * (C / 8), 4);
  if (!z) {
    groupnorm_bwd_apply_kernel<<<g2, 256, 4 * G * sizeof(float), st>>>(
        static_cast<const __nv_bfloat16*>(x), static_cast<const __nv_bfloat16*>(dy), static_cast<__nv_bfloat16*>(dx), gamma, stats, dgamma,
        dbeta, DHW, (int)C, (int)G, eps, nullptr, nullptr, 0);
    return check_launch("groupnorm_bwd_apply_kernel");
  }
  groupnorm_bwd_apply_det_kernel<<<g2, 256, (4 * G + 256 * 8) * sizeof(float), st>>>(
      static_cast<const __nv_bfloat16*>(x), static_cast<const __nv_bfloat16*>(dy), static_cast<__nv_bfloat16*>(dx), gamma, stats, dgamma,
      dbeta, DHW, (int)C, (int)G, eps, static_cast<const __nv_bfloat16*>(z), scratch, (int)W2);
  if (int rc = check_launch("groupnorm_bwd_apply_det_kernel")) return rc;
  return det_finalize(scratch, g2, C, C, db, true, st);
}

int cvit_pixel_unshuffle_1x2x2_bf16(const void* src, void* dst, int64_t D, int64_t H, int64_t W, int64_t C, void* stream) {
  if (!src || !dst || D <= 0 || H <= 0 || W <= 0 || C <= 0 || (C % 8)) { set_error("pixel_unshuffle: bad arguments"); return CVIT_ERR_INVALID; }
  pixel_unshuffle_kernel<<<ew_grid(D * H * W * 4 * (C / 8), 4), 256, 0, (cudaStream_t)stream>>>(
      static_cast<const uint4*>(src), static_cast<uint4*>(dst), (int)D, (int)H, (int)W, (int)(C / 8));
  return check_launch("pixel_unshuffle_kernel");
}

int cvit_adamw_f32(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                   float weight_decay, int64_t step, float grad_scale, void* stream) {
  if (!p || !g || !m || !v || n <= 0 || step <= 0) { set_error("adamw: bad arguments"); return CVIT_ERR_INVALID; }
  const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
  adamw_kernel<<<ew_grid(n, 4), 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, (float)bc1,
                                                                (float)(1.0 / sqrt(bc2)), grad_scale);
  return check_launch("adamw_kernel");
}

int cvit_accumulate_f32(float* dst, const float* src, int64_t n, void* stream) {
  if (!dst || !src || n <= 0) { set_error("accumulate_f32: bad arguments"); return CVIT_ERR_INVALID; }
  return det_finalize(src, 1, n, n, dst, true, (cudaStream_t)stream);
}

}  // extern "C"
