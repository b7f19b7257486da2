// Weight gradients of the CryoVIT head (training, BASELINE config 5) as split-K tcgen05 GEMMs.
//
//   dW[tap][co][ci] = sum over voxels v of  dZ[v, co] * X[v + off(tap), ci]
//
// Both operands are used CHANNELS-FIRST and zero-padded (cvit_ndhwc_to_cfirst_padded makes the copies):
//   At[co][p], Bt[ci][p]   with p the linear index over the padded volume (D + 2*pd, H + 2, Wp),
// so a convolution tap is a constant shift koff of p, and the reduction over voxels is the K dimension of a plain
// K-major GEMM  D[co, ci] = At[co, :] . Bt[ci, : + koff]  -- the same TMA / UMMA layouts as the forward GEMMs. The
// borders of At are zero, so positions where the shifted index would wrap to the next row / plane contribute nothing.
// TMA needs the innermost start coordinate 16-byte aligned, so koff must be a multiple of 8 elements: the padded row
// pitch Wp is a multiple of 8 (depth / row taps are then aligned shifts) and the three column taps use three copies
// of X made with a built-in column shift of -1, 0, +1. 1x1x1 and transposed convolutions are the one-tap case.
//
// Narrow layers (co <= 64) would waste most of the 128 MMA rows, so several taps are PACKED into one A tile: since
//   sum_p At[co][p] Bt[ci][p + koff] = sum_q At[co][q - koff] Bt[ci][q],
// tap t's rows are just At loaded with a start coordinate shifted by -koff[t] (one small TMA box per tap, stacked at
// row t * Mp of the stage), B is loaded once, unshifted, and ONE MMA chain produces 128 / Mp taps at a time.
//
// The reduction is split over the grid: a work item is (tap, 128-row tile of co, BN-column tile of ci, K range); every
// item accumulates in TMEM and adds its partial tile into the fp32 result with red.global.add (the result buffer is
// zeroed by the caller). One CTA per SM, 192 threads: TMA producer, MMA issuer (warp-uniform, elect.sync), four
// epilogue warps (thread = output row).
#include "det_reduce.cuh"
#include "ptx.cuh"
#include "tmap.h"

namespace cvit {

constexpr int WG_BM = 128, WG_KC = 64, WG_THREADS = 192;

template <int BN>
struct WgCfg {
  static constexpr int A_BYTES = WG_BM * 128, B_BYTES = BN * 128, STAGE = A_BYTES + B_BYTES;
  static constexpr int STAGES_RAW = (200 * 1024) / STAGE;
  static constexpr int STAGES = STAGES_RAW > 8 ? 8 : STAGES_RAW;
  static constexpr int ACC = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;
  static constexpr int TMEM_COLS = 2 * ACC;
  static constexpr int SMEM = STAGES * STAGE + 256 + 1024;
};

struct WgArgs {
  float* out;           // [ntaps][M][N] fp32, accumulated into (deterministic mode: [ksplit][ntaps][M][N], stored)
  const int* koffs;     // [ntaps] shift of the B operand along K (elements), device memory
  int M, N, ntaps;      // valid rows of A (co), valid rows of B (ci)
  int k_chunks;         // ceil(K / 64)
  int ksplit;           // K ranges per (tap, tile)
  int pack;             // taps per A tile (1 = one tap per item, A tile = 128 rows of co; > 1: Mp rows per tap)
  int Mp;               // rows per packed tap (co rounded up to 8), pack * Mp <= 128
};

// DET (deterministic mode): an item's tile is STORED into K slice ks of the [ksplit][ntaps][M][N] slab (zeros for an empty
// K range), and det_finalize adds the slices in ks order.
template <int BN, bool DET>
__device__ __forceinline__ void wgrad_tcgen05_body(const CUtensorMap& tmA, const CUtensorMap& tmB, const WgArgs& args) {
  using Cfg = WgCfg<BN>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sA = smem_base, sB = smem_base + STAGES * Cfg::A_BYTES;
  const uint32_t sBar = smem_base + STAGES * Cfg::STAGE;
  const uint32_t bar_full = sBar, bar_empty = sBar + 8 * STAGES;
  const uint32_t bar_tfull = sBar + 16 * STAGES, bar_tempty = bar_tfull + 16, tmem_slot = bar_tempty + 16;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const int pack = args.pack;
  const int m_tiles = pack > 1 ? 1 : (args.M + WG_BM - 1) / WG_BM, n_tiles = (args.N + BN - 1) / BN;
  const int per_tap = m_tiles * n_tiles * args.ksplit;
  const int tap_groups = (args.ntaps + pack - 1) / pack;  // "tap" below is a group of `pack` taps
  const int num_items = tap_groups * per_tap;
  const int kc_per = (args.k_chunks + args.ksplit - 1) / args.ksplit;
  auto item_of = [&](int item, int& tap, int& m0, int& n0, int& kc0, int& kc1) {
    tap = item / per_tap;
    int r = item - tap * per_tap;
    const int ks = r % args.ksplit;
    r /= args.ksplit;
    n0 = (r % n_tiles) * BN;
    m0 = (r / n_tiles) * WG_BM;
    kc0 = ks * kc_per;
    kc1 = min(args.k_chunks, kc0 + kc_per);
  };

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_tfull + 8 * i, 1);
      mbar_init(bar_tempty + 8 * i, 4);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  if (warp == 0) {
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
        int tap, m0, n0, kc0, kc1;
        item_of(item, tap, m0, n0, kc0, kc1);
        if (pack > 1) {
          const int t0 = tap * pack, nt = min(pack, args.ntaps - t0);
          for (int kc = kc0; kc < kc1; ++kc) {
            mbar_wait(bar_empty + 8 * s, ph ^ 1u);
            mbar_arrive_expect_tx(bar_full + 8 * s, nt * args.Mp * 128 + Cfg::B_BYTES);
            for (int t = 0; t < nt; ++t)  // tap t's rows: the same co rows, shifted the other way
              tma_load_2d(sA + s * Cfg::A_BYTES + t * args.Mp * 128, &tmA, bar_full + 8 * s,
                          kc * WG_KC - __ldg(args.koffs + t0 + t), 0);
            tma_load_2d(sB + s * Cfg::B_BYTES, &tmB, bar_full + 8 * s, kc * WG_KC, n0);
            if (++s == STAGES) { s = 0; ph ^= 1u; }
          }
          continue;
        }
        const int koff = __ldg(args.koffs + tap);
        for (int kc = kc0; kc < kc1; ++kc) {
          mbar_wait(bar_empty + 8 * s, ph ^ 1u);
          mbar_arrive_expect_tx(bar_full + 8 * s, Cfg::STAGE);
          tma_load_2d(sA + s * Cfg::A_BYTES, &tmA, bar_full + 8 * s, kc * WG_KC, m0);
          tma_load_2d(sB + s * Cfg::B_BYTES, &tmB, bar_full + 8 * s, kc * WG_KC + koff, n0);  // OOB (also negative) = 0
          if (++s == STAGES) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = umma_idesc_bf16_f32(WG_BM, BN);
    int s = 0, acc = 0;
    uint32_t ph = 0, acc_ph = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
      int tap, m0, n0, kc0, kc1;
      item_of(item, tap, m0, n0, kc0, kc1);
      mbar_wait(bar_tempty + 8 * acc, acc_ph ^ 1u);
      tcgen05_fence_after();
      const uint32_t d_tmem = tmem_base + acc * Cfg::ACC;
      for (int kc = kc0; kc < kc1; ++kc) {
        mbar_wait(bar_full + 8 * s, ph);
        tcgen05_fence_after();
        if (elect_one_sync()) {
          const uint64_t ad = umma_smem_desc_kmajor<128>(sA + s * Cfg::A_BYTES);
          const uint64_t bd = umma_smem_desc_kmajor<128>(sB + s * Cfg::B_BYTES);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16(d_tmem, ad + 2 * k, bd + 2 * k, idesc, (kc > kc0) | (k > 0));
          umma_commit(bar_empty + 8 * s);
        }
        __syncwarp();
        if (++s == STAGES) { s = 0; ph ^= 1u; }
      }
      if (elect_one_sync()) umma_commit(bar_tfull + 8 * acc);
      __syncwarp();
      acc ^= 1;
      if (acc == 0) acc_ph ^= 1u;
    }
  } else {
    const int q = warp & 3;
    const int r = q * 32 + lane;
    int acc = 0;
    uint32_t acc_ph = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
      int tap, m0, n0, kc0, kc1;
      item_of(item, tap, m0, n0, kc0, kc1);
      mbar_wait(bar_tfull + 8 * acc, acc_ph);
      tcgen05_fence_after();
      const uint32_t t_acc = tmem_base + acc * Cfg::ACC + (static_cast<uint32_t>(q * 32) << 16);
      int row = m0 + r, otap = tap;
      bool live = row < args.M;
      if (pack > 1) {  // row r of the tile = tap (tap * pack + r / Mp), output channel r % Mp
        otap = tap * pack + r / args.Mp;
        row = r % args.Mp;
        live = r < pack * args.Mp && otap < args.ntaps && row < args.M;
      }
      float* orow = args.out + ((size_t)otap * args.M + row) * args.N + n0;
      if constexpr (DET) orow += (size_t)((item % per_tap) % args.ksplit) * args.ntaps * args.M * args.N;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32(t_acc + c0, v);
        tmem_ld_wait();
        if constexpr (DET) {
          if (live) {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (n0 + c0 + i < args.N) orow[c0 + i] = kc1 > kc0 ? __uint_as_float(v[i]) : 0.f;
          }
        } else if (live && kc1 > kc0) {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (n0 + c0 + i < args.N) atomicAdd(orow + c0 + i, __uint_as_float(v[i]));
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
      acc ^= 1;
      if (acc == 0) acc_ph ^= 1u;
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tcgen05_fence_after();
    tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

template <int BN>
__global__ void __launch_bounds__(WG_THREADS, 1)
wgrad_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const WgArgs args) {
  wgrad_tcgen05_body<BN, false>(tmA, tmB, args);
}

template <int BN>
__global__ void __launch_bounds__(WG_THREADS, 1)
wgrad_tcgen05_det_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const WgArgs args) {
  wgrad_tcgen05_body<BN, true>(tmA, tmB, args);
}

template <int BN, bool DET = false>
static int launch_wgrad(const CUtensorMap& tmA, const CUtensorMap& tmB, const WgArgs& a, cudaStream_t st) {
  using Cfg = WgCfg<BN>;
  auto kern = DET ? wgrad_tcgen05_det_kernel<BN> : wgrad_tcgen05_kernel<BN>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM);
    if (e != cudaSuccess) {
      set_error("wgrad: cudaFuncSetAttribute(smem=%d): %s", Cfg::SMEM, cudaGetErrorString(e));
      return CVIT_ERR_CUDA;
    }
    configured = true;
  }
  const int m_tiles = a.pack > 1 ? 1 : (a.M + WG_BM - 1) / WG_BM, n_tiles = (a.N + BN - 1) / BN;
  const int items = ((a.ntaps + a.pack - 1) / a.pack) * m_tiles * n_tiles * a.ksplit;
  int grid = num_sms();
  if (grid > items) grid = items;
  kern<<<grid, WG_THREADS, Cfg::SMEM, st>>>(tmA, tmB, a);
  return check_launch(DET ? "wgrad_tcgen05_det_kernel" : "wgrad_tcgen05_kernel");
}

// ------------------------------------------------------------------------------------------------
// channels-last bf16 [D, H, W, C] -> channels-first, zero-padded bf16 [C][(D + 2 pd) (H + 2 ph) (W + 2 pw)] (row pitch
// `pitch` elements, a multiple of 8 for TMA): the operand layout of the split-K weight-gradient GEMM. The padding
// is written here too (whole destination is covered), 32x32 transposes through shared memory.
__global__ void __launch_bounds__(256) ndhwc_to_cfirst_padded_kernel(const __nv_bfloat16* __restrict__ src,
                                                                      __nv_bfloat16* __restrict__ dst, int D, int H, int W,
                                                                      int C, int pd, int ph, int pw, int Wp, int wshift,
                                                                      int64_t pitch) {
  __shared__ __nv_bfloat16 tile[32][33];
  const int Hp = H + 2 * ph, Dp = D + 2 * pd;
  const int64_t P = (int64_t)Dp * Hp * Wp;
  const int64_t p0 = (int64_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int i = ty; i < 32; i += 8) {  // rows = padded positions, cols = channels (contiguous in src)
    const int64_t p = p0 + i;
    const int c = c0 + tx;
    __nv_bfloat16 v = __float2bfloat16(0.f);
    if (p < P && c < C) {
      const int w = (int)(p % Wp) - pw + wshift, h = (int)((p / Wp) % Hp) - ph, d = (int)(p / ((int64_t)Wp * Hp)) - pd;
      if (w >= 0 && w < W && h >= 0 && h < H && d >= 0 && d < D) v = src[(((int64_t)d * H + h) * W + w) * C + c];
    }
    tile[i][tx] = v;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i;
    const int64_t p = p0 + tx;
    if (c < C && p < pitch) dst[(int64_t)c * pitch + p] = p < P ? tile[tx][i] : __float2bfloat16(0.f);
  }
}

// The same for C % 64 == 0 with 16-byte accesses on both sides: a CTA moves 64 padded positions x 64 channels; a thread
// loads 8 consecutive channels of one position (16 B; a warp reads four 128-byte runs), parks them in shared memory,
// then gathers 8 consecutive positions of one channel (eight conflict-free 2-byte reads: the 32 lanes of a warp take 32
// consecutive channels) and writes them as one 16-byte store. The scalar kernel above did three 64-bit divisions and
// two 2-byte memory operations per element: 12.5 ms of a 52 ms training step for 10 GB of traffic.
constexpr int CF_PITCH = 72;  // halves per shared-memory row (144 B: 16-byte aligned rows, skewed banks)
__global__ void __launch_bounds__(256) ndhwc_to_cfirst_padded_vec_kernel(const __nv_bfloat16* __restrict__ src,
                                                                          __nv_bfloat16* __restrict__ dst, int D, int H, int W,
                                                                          int C, int pd, int ph, int pw, int Wp, int wshift,
                                                                          int64_t pitch) {
  __shared__ __align__(16) __nv_bfloat16 tile[64 * CF_PITCH];
  const int Hp = H + 2 * ph, Dp = D + 2 * pd;
  const int64_t P = (int64_t)Dp * Hp * Wp;
  const int64_t p0 = (int64_t)blockIdx.x * 64;
  const int c0 = blockIdx.y * 64;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int q = threadIdx.x + k * 256;  // 512 loads: position q / 8, 8-channel chunk q % 8
    const int pl = q >> 3, ch = q & 7;
    const int64_t p = p0 + pl;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (p < P) {
      const int64_t row = p / Wp;
      const int w = (int)(p - row * Wp) - pw + wshift;
      const int dpl = (int)(row / Hp);
      const int h = (int)(row - (int64_t)dpl * Hp) - ph, d = dpl - pd;
      if (w >= 0 && w < W && h >= 0 && h < H && d >= 0 && d < D)
        v = __ldg(reinterpret_cast<const uint4*>(src + (((int64_t)d * H + h) * W + w) * C + c0 + ch * 8));
    }
    *reinterpret_cast<uint4*>(&tile[pl * CF_PITCH + ch * 8]) = v;
  }
  __syncthreads();
  const unsigned short* t16 = reinterpret_cast<const unsigned short*>(tile);
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int q = threadIdx.x + k * 256;  // 512 stores: channel q % 64 (fastest: conflict-free reads), position group q / 64
    const int c = q & 63, pg = q >> 6;
    const int64_t p = p0 + pg * 8;
    if (p >= pitch) continue;  // pitch is a multiple of 8: a group is inside or outside as a whole
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t lo = t16[(pg * 8 + 2 * j) * CF_PITCH + c], hi = t16[(pg * 8 + 2 * j + 1) * CF_PITCH + c];
      o[j] = lo | (hi << 16);
    }
    *reinterpret_cast<uint4*>(dst + (int64_t)(c0 + c) * pitch + p) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// Narrow volumes (C <= 32, the layers with tens of millions of voxels): one thread turns 8 consecutive padded positions
// of one 8-channel chunk into 8 x 16-byte stores (one per channel row, 8 positions each), so a warp writes 512
// contiguous bytes per row; with NSHIFT = 3 the column-shifted copies -1, 0, +1 come out of the same loads.
template <int NSHIFT>
__global__ void __launch_bounds__(256) ndhwc_to_cfirst_padded_narrow_kernel(const __nv_bfloat16* __restrict__ src,
                                                                             __nv_bfloat16* __restrict__ dst0,
                                                                             __nv_bfloat16* __restrict__ dst1,
                                                                             __nv_bfloat16* __restrict__ dst2, int D, int H, int W,
                                                                             int C, int pd, int ph, int pw, int Wp, int wshift,
                                                                             int64_t pitch) {
  const int Hp = H + 2 * ph;
  const int nchunk = C / 8;
  const int64_t groups = pitch / 8, total = groups * nchunk;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t gp = idx % groups;  // position group fastest: coalesced stores along each channel row
    const int chunk = (int)(idx / groups);
    const int64_t p0 = gp * 8;
    const int wp0 = (int)(p0 % Wp), hp = (int)((p0 / Wp) % Hp);
    const int d = (int)(p0 / ((int64_t)Wp * Hp)) - pd, h = hp - ph;
    const bool row_ok = d >= 0 && d < D && h >= 0 && h < H;
    const __nv_bfloat16* row = src + (((int64_t)(row_ok ? d : 0) * H + (row_ok ? h : 0)) * W) * C + chunk * 8;
    constexpr int NV = NSHIFT == 3 ? 10 : 8;
    uint4 v[NV];
    const int wbase = wp0 - pw + (NSHIFT == 3 ? -1 : wshift);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int w = wbase + i;
      v[i] = (row_ok && w >= 0 && w < W) ? *reinterpret_cast<const uint4*>(row + (int64_t)w * C) : make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int sft = 0; sft < NSHIFT; ++sft) {
      __nv_bfloat16* dst = sft == 0 ? dst0 : sft == 1 ? dst1 : dst2;
#pragma unroll
      for (int k = 0; k < 8; ++k) {  // channel k of the chunk: gather its value from the 8 voxels
        uint32_t o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint32_t lo = reinterpret_cast<const uint32_t*>(&v[2 * j + sft])[k >> 1];
          const uint32_t hi = reinterpret_cast<const uint32_t*>(&v[2 * j + 1 + sft])[k >> 1];
          o[j] = (k & 1) ? __byte_perm(lo, hi, 0x7632) : __byte_perm(lo, hi, 0x5410);
        }
        *reinterpret_cast<uint4*>(dst + (int64_t)(chunk * 8 + k) * pitch + p0) = make_uint4(o[0], o[1], o[2], o[3]);
      }
    }
  }
}

}  // namespace cvit

using namespace cvit;

// Three column-shifted copies (-1, 0, +1) in one pass (narrow volumes; C in {8, 16, 32}).
extern "C" int cvit_ndhwc_to_cfirst_padded_x3(const void* src, void* dst_m1, void* dst_0, void* dst_p1, int64_t D, int64_t H,
                                              int64_t W, int64_t C, int64_t pd, int64_t ph, int64_t pw, int64_t Wp, int64_t pitch,
                                              void* stream) {
  const int64_t P = (D + 2 * pd) * (H + 2 * ph) * Wp;
  if (!src || !dst_m1 || !dst_0 || !dst_p1 || D <= 0 || H <= 0 || W <= 0 || (C != 8 && C != 16 && C != 32) || pd < 0 || ph < 0 ||
      pw < 1 || Wp < W + 2 * pw || (Wp % 8) != 0 || pitch != P) {
    set_error("ndhwc_to_cfirst_padded_x3: bad arguments");
    return CVIT_ERR_INVALID;
  }
  const int64_t total = pitch / 8 * (C / 8);
  int64_t blocks = (total + 255) / 256;
  if (blocks > (int64_t)num_sms() * 32) blocks = (int64_t)num_sms() * 32;
  ndhwc_to_cfirst_padded_narrow_kernel<3><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
      static_cast<const __nv_bfloat16*>(src), static_cast<__nv_bfloat16*>(dst_m1), static_cast<__nv_bfloat16*>(dst_0),
      static_cast<__nv_bfloat16*>(dst_p1), (int)D, (int)H, (int)W, (int)C, (int)pd, (int)ph, (int)pw, (int)Wp, 0, pitch);
  return check_launch("ndhwc_to_cfirst_padded_narrow_kernel<3>");
}

extern "C" int cvit_ndhwc_to_cfirst_padded(const void* src, void* dst, int64_t D, int64_t H, int64_t W, int64_t C,
                                           int64_t pd, int64_t ph, int64_t pw, int64_t Wp, int64_t wshift, int64_t pitch,
                                           void* stream) {
  const int64_t P = (D + 2 * pd) * (H + 2 * ph) * Wp;
  if (!src || !dst || D <= 0 || H <= 0 || W <= 0 || C <= 0 || pd < 0 || ph < 0 || pw < 0 || Wp < W + 2 * pw || pitch < P ||
      (pitch % 8) != 0) {
    set_error("ndhwc_to_cfirst_padded: bad arguments");
    return CVIT_ERR_INVALID;
  }
  if ((C == 8 || C == 16 || C == 32) && (Wp % 8) == 0 && pitch == P) {  // narrow volume: register transpose
    const int64_t total = pitch / 8 * (C / 8);
    int64_t blocks = (total + 255) / 256;
    if (blocks > (int64_t)num_sms() * 32) blocks = (int64_t)num_sms() * 32;
    ndhwc_to_cfirst_padded_narrow_kernel<1><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        static_cast<const __nv_bfloat16*>(src), static_cast<__nv_bfloat16*>(dst), nullptr, nullptr, (int)D, (int)H, (int)W, (int)C,
        (int)pd, (int)ph, (int)pw, (int)Wp, (int)wshift, pitch);
    return check_launch("ndhwc_to_cfirst_padded_narrow_kernel<1>");
  }
  if (C % 64 == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15u) == 0) {
    dim3 gridv((unsigned)((pitch + 63) / 64), (unsigned)(C / 64));
    ndhwc_to_cfirst_padded_vec_kernel<<<gridv, 256, 0, (cudaStream_t)stream>>>(
        static_cast<const __nv_bfloat16*>(src), static_cast<__nv_bfloat16*>(dst), (int)D, (int)H, (int)W, (int)C, (int)pd,
        (int)ph, (int)pw, (int)Wp, (int)wshift, pitch);
    return check_launch("ndhwc_to_cfirst_padded_vec_kernel");
  }
  dim3 grid((unsigned)((pitch + 31) / 32), (unsigned)((C + 31) / 32));
  ndhwc_to_cfirst_padded_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
      static_cast<const __nv_bfloat16*>(src), static_cast<__nv_bfloat16*>(dst), (int)D, (int)H, (int)W, (int)C, (int)pd,
      (int)ph, (int)pw, (int)Wp, (int)wshift, pitch);
  return check_launch("ndhwc_to_cfirst_padded_kernel");
}

// Launch geometry of cvit_wgrad_splitk: N tile, taps per A tile and K split.
static void splitk_geometry(int64_t M, int64_t N, int64_t K, int64_t ntaps, int* bn, int* pack, int* Mp, int* k_chunks, int* ksplit) {
  *bn = N > 192 ? 256 : N > 128 ? 192 : N > 64 ? 128 : N > 32 ? 64 : 32;  // 192: one exact tile for the 192-channel layers
  // narrow outputs: pack several taps into the 128 MMA rows (see the header comment)
  *Mp = (int)((M + 7) / 8 * 8);
  *pack = (M <= 64 && ntaps > 1) ? WG_BM / *Mp : 1;
  if (*pack > ntaps) *pack = (int)ntaps;
  *k_chunks = (int)((K + WG_KC - 1) / WG_KC);
  const int m_tiles = *pack > 1 ? 1 : (int)((M + WG_BM - 1) / WG_BM), n_tiles = (int)((N + *bn - 1) / *bn);
  const int64_t tiles = ((ntaps + *pack - 1) / *pack) * m_tiles * n_tiles;
  // enough K ranges for ~4 items per SM, but never K ranges shorter than 32 chunks (2048 reduction steps)
  int ks = (int)((4 * (int64_t)num_sms() + tiles - 1) / tiles);
  const int max_split = *k_chunks / 32 > 0 ? *k_chunks / 32 : 1;
  if (ks > max_split) ks = max_split;
  if (ks < 1) ks = 1;
  *ksplit = ks;
}

extern "C" int64_t cvit_wgrad_splitk_det_partials(int64_t M, int64_t N, int64_t K, int64_t ntaps) {
  if (M <= 0 || N <= 0 || K <= 0 || ntaps <= 0) return 0;
  int bn, pack, Mp, k_chunks, ksplit;
  splitk_geometry(M, N, K, ntaps, &bn, &pack, &Mp, &k_chunks, &ksplit);
  return (int64_t)ksplit * ntaps * M * N;
}

// Deterministic mode: out += the same product, every item's tile stored into its K slice of scratch
// (cvit_wgrad_splitk_det_partials floats) and the slices added in K order.
extern "C" int cvit_wgrad_splitk_det(const void* At, const void* Bt, float* out, const int* koffs, int64_t M, int64_t N, int64_t K,
                                     int64_t pitch_a, int64_t pitch_b, int64_t ntaps, float* scratch, int64_t scratch_elems, void* stream) {
  if (!At || !Bt || !out || !koffs || M <= 0 || N <= 0 || K <= 0 || ntaps <= 0 || pitch_a < K || pitch_b < K ||
      (pitch_a % 8) != 0 || (pitch_b % 8) != 0) {
    set_error("wgrad_splitk_det: bad arguments (M=%lld N=%lld K=%lld pitches %lld %lld taps %lld)", (long long)M, (long long)N,
              (long long)K, (long long)pitch_a, (long long)pitch_b, (long long)ntaps);
    return CVIT_ERR_INVALID;
  }
  if (int rc = det_check_scratch(scratch, scratch_elems, cvit_wgrad_splitk_det_partials(M, N, K, ntaps), "wgrad_splitk_det")) return rc;
  if (((reinterpret_cast<uintptr_t>(At) | reinterpret_cast<uintptr_t>(Bt)) & 15u) != 0) {
    set_error("wgrad_splitk_det: operands must be 16-byte aligned");
    return CVIT_ERR_INVALID;
  }
  int bn, pack, Mp, k_chunks, ksplit;
  splitk_geometry(M, N, K, ntaps, &bn, &pack, &Mp, &k_chunks, &ksplit);
  CUtensorMap tmA, tmB;
  {
    uint64_t dims[2] = {(uint64_t)K, (uint64_t)M};
    uint64_t strides[2] = {0, (uint64_t)pitch_a * 2};
    uint32_t box[2] = {WG_KC, pack > 1 ? (uint32_t)Mp : (uint32_t)WG_BM};
    int rc = encode_tmap(&tmA, TmapDtype::BF16, 2, At, dims, strides, box, 128);
    if (rc) return rc;
  }
  {
    uint64_t dims[2] = {(uint64_t)K, (uint64_t)N};
    uint64_t strides[2] = {0, (uint64_t)pitch_b * 2};
    uint32_t box[2] = {WG_KC, (uint32_t)bn};
    int rc = encode_tmap(&tmB, TmapDtype::BF16, 2, Bt, dims, strides, box, 128);
    if (rc) return rc;
  }
  WgArgs a;
  a.out = scratch;
  a.koffs = koffs;
  a.M = (int)M;
  a.N = (int)N;
  a.ntaps = (int)ntaps;
  a.k_chunks = k_chunks;
  a.pack = pack;
  a.Mp = Mp;
  a.ksplit = ksplit;
  cudaStream_t st = (cudaStream_t)stream;
  int rc;
  switch (bn) {
    case 256: rc = launch_wgrad<256, true>(tmA, tmB, a, st); break;
    case 192: rc = launch_wgrad<192, true>(tmA, tmB, a, st); break;
    case 128: rc = launch_wgrad<128, true>(tmA, tmB, a, st); break;
    case 64: rc = launch_wgrad<64, true>(tmA, tmB, a, st); break;
    default: rc = launch_wgrad<32, true>(tmA, tmB, a, st); break;
  }
  if (rc) return rc;
  const int64_t n = ntaps * M * N;
  return det_finalize(scratch, ksplit, n, n, out, true, st);
}

extern "C" int cvit_wgrad_splitk(const void* At, const void* Bt, float* out, const int* koffs, int64_t M, int64_t N,
                                 int64_t K, int64_t pitch_a, int64_t pitch_b, int64_t ntaps, void* stream) {
  if (!At || !Bt || !out || !koffs || M <= 0 || N <= 0 || K <= 0 || ntaps <= 0 || pitch_a < K || pitch_b < K ||
      (pitch_a % 8) != 0 || (pitch_b % 8) != 0) {
    set_error("wgrad_splitk: bad arguments (M=%lld N=%lld K=%lld pitches %lld %lld taps %lld)", (long long)M, (long long)N,
              (long long)K, (long long)pitch_a, (long long)pitch_b, (long long)ntaps);
    return CVIT_ERR_INVALID;
  }
  if (((reinterpret_cast<uintptr_t>(At) | reinterpret_cast<uintptr_t>(Bt)) & 15u) != 0) {
    set_error("wgrad_splitk: operands must be 16-byte aligned");
    return CVIT_ERR_INVALID;
  }
  const int bn = N > 192 ? 256 : N > 128 ? 192 : N > 64 ? 128 : N > 32 ? 64 : 32;  // 192: one exact tile for the 192-channel layers
  // narrow outputs: pack several taps into the 128 MMA rows (see the header comment)
  const int Mp = (int)((M + 7) / 8 * 8);
  int pack = (M <= 64 && ntaps > 1) ? WG_BM / Mp : 1;
  if (pack > ntaps) pack = (int)ntaps;
  CUtensorMap tmA, tmB;
  {
    uint64_t dims[2] = {(uint64_t)K, (uint64_t)M};
    uint64_t strides[2] = {0, (uint64_t)pitch_a * 2};
    uint32_t box[2] = {WG_KC, pack > 1 ? (uint32_t)Mp : (uint32_t)WG_BM};
    int rc = encode_tmap(&tmA, TmapDtype::BF16, 2, At, dims, strides, box, 128);
    if (rc) return rc;
  }
  {
    uint64_t dims[2] = {(uint64_t)K, (uint64_t)N};
    uint64_t strides[2] = {0, (uint64_t)pitch_b * 2};
    uint32_t box[2] = {WG_KC, (uint32_t)bn};
    int rc = encode_tmap(&tmB, TmapDtype::BF16, 2, Bt, dims, strides, box, 128);
    if (rc) return rc;
  }
  WgArgs a;
  a.out = out;
  a.koffs = koffs;
  a.M = (int)M;
  a.N = (int)N;
  a.ntaps = (int)ntaps;
  a.k_chunks = (int)((K + WG_KC - 1) / WG_KC);
  a.pack = pack;
  a.Mp = Mp;
  const int m_tiles = pack > 1 ? 1 : (int)((M + WG_BM - 1) / WG_BM), n_tiles = (int)((N + bn - 1) / bn);
  const int64_t tiles = ((ntaps + pack - 1) / pack) * m_tiles * n_tiles;
  // enough K ranges for ~4 items per SM, but never K ranges shorter than 32 chunks (2048 reduction steps)
  int ksplit = (int)((4 * (int64_t)num_sms() + tiles - 1) / tiles);
  const int max_split = a.k_chunks / 32 > 0 ? a.k_chunks / 32 : 1;
  if (ksplit > max_split) ksplit = max_split;
  if (ksplit < 1) ksplit = 1;
  a.ksplit = ksplit;
  cudaStream_t st = (cudaStream_t)stream;
  switch (bn) {
    case 256: return launch_wgrad<256>(tmA, tmB, a, st);
    case 192: return launch_wgrad<192>(tmA, tmB, a, st);
    case 128: return launch_wgrad<128>(tmA, tmB, a, st);
    case 64: return launch_wgrad<64>(tmA, tmB, a, st);
    default: return launch_wgrad<32>(tmA, tmB, a, st);
  }
}
