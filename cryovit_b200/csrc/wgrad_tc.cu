// Weight gradient of the 8 -> 8 channel 3x3x3 convolutions of the CryoVIT head (output_layer.0 / output_layer.2 at full
// resolution, models/cryovit.py:30-34; head training, BASELINE config 5) on tcgen05, straight from the channels-last
// volumes:
//
//   dW[kd][kh][kw][co][ci] = sum over output voxels (z, y, x) of  dZ[z, y, x][co] * X[z + (kd-1) dil, y + kh - 1, x + kw - 1][ci]
//
// 116 GFLOP whose result is 1728 numbers: a reduction over 33.5 M voxels. The warp-level kernel (csrc/wgrad_narrow.cu) is
// bound by the mma.sync rate of this chip (1.07 ms per launch, two launches per step). Here the VOXELS ARE THE K DIMENSION
// OF ONE tcgen05 MMA and nothing is re-laid-out:
//
//   * 8 channels of a channels-last voxel are 16 bytes, so a row segment [voxels][8] in shared memory is, as it lies, an
//     MN-major SWIZZLE_NONE operand: a core matrix is 8 consecutive voxels (K) x 8 channels (M or N) = 128 contiguous
//     bytes, the next 8 voxels follow 128 bytes on (LBO).
//   * A = X. The three column taps kw are the SAME row read one voxel further on, and one voxel is 16 bytes = the stride
//     between core matrices along M (SBO = 16): accumulator row m = kw * 8 + ci reads X[.., x0 + k - 1 + kw][ci]. No
//     shifted copies. (The MMA's other rows read further "taps"; those accumulator rows are never looked at.)
//   * B = dZ. For the X row (z0, y0) the nine (kd, kh) taps pair it with the dZ rows (z0 - (kd-1) dil, y0 - (kh-1)). A stage
//     holds the dZ rows y0 - 1 .. y0 + R of the three planes as equal-sized arrays ordered [row][plane], so the nine arrays
//     of one X row are consecutive: accumulator column n = ((yr * 3 + kd) * 8 + co), SBO = array size. R consecutive X
//     rows share the stage's dZ rows: (R + 2) * 3 row loads per R rows instead of 9 R.
//   * Every TMA box is whole 128-byte lines ([8 voxels][8 channels]); out-of-bounds zero fill is the convolution's
//     padding (x = -1, x = W, rows and planes outside the volume) and the ragged ends of the tiling.
//
// One MMA (M 64, N 80, K 16 voxels) per 16 voxels of a row for all 27 taps: 2.1 M MMAs per launch over 148 SMs. The
// accumulator (80 TMEM columns) lives for the whole kernel; one red.global.add pass per CTA at the end.
// One CTA per SM, 192 threads: warp 0 TMA producer, warp 1 MMA issuer + TMEM owner, warp 4 the final read-out.
#include <cstdlib>

#include "det_reduce.cuh"
#include "ptx.cuh"
#include "tmap.h"

namespace cvit {

constexpr int WT_THREADS = 192;
constexpr int WT_R = 8;        // X rows per stage
constexpr int WT_KSEG = 128;   // voxels of a row per stage
constexpr int WT_XARR = (WT_KSEG + 16) * 16;  // X row array: voxels x0 - 8 .. x0 + KSEG + 7 (whole 128-byte lines)
constexpr int WT_ZARR = WT_KSEG * 16;         // dZ row array: voxels x0 .. x0 + KSEG - 1
constexpr int WT_X_BYTES = WT_R * WT_XARR;
constexpr int WT_Z_BYTES = ((WT_R + 2) * 3 + 1) * WT_ZARR;  // + one array: N = 80 reads a tenth (ignored) column block
constexpr int WT_STAGE = (WT_X_BYTES + WT_Z_BYTES + 1023) / 1024 * 1024;
constexpr int WT_STAGES = 2;
constexpr int WT_SMEM = WT_STAGES * WT_STAGE + 256 + 1024;
constexpr int WT_N = 80, WT_TMEM_COLS = 128;
// M = 64 halves the A tile the tensor core streams per MMA (24 of the rows are used either way): 0.475 -> 0.382 ms per
// launch. -DWT_M=128 builds the full-height variant (A/B).
#ifndef WT_M
#define WT_M 64
#endif
constexpr uint32_t WT_TX_BYTES = WT_R * WT_XARR + (WT_R + 2) * 3 * WT_ZARR;

struct WtArgs {
  float* dw;  // [27][Cout][Cin] fp32, accumulated into (tap = (kd*3+kh)*3+kw, then co, then ci); deterministic mode:
              // [gridDim.x][27][Cout][Cin], one row per CTA, stored
  const __nv_bfloat16* x;   // [D, H, W, Cin]  (read directly by the cp.async loaders of the 16 / 32-channel kernel)
  const __nv_bfloat16* dz;  // [D, H, W, Cout]
  int D, H, W, dil;
};

// MN-major SWIZZLE_NONE operand: core matrix = 8 K-rows of 16 bytes; LBO = next 8 K, SBO = next 8 M/N elements
// (cute::UMMA canonical layout ((1,n),(8,k)):((X,SBO),(1,LBO)) in 16-byte units)
__device__ __forceinline__ uint64_t wt_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) {
#ifdef WT_SWAP_LBO_SBO
  const uint32_t t = lbo; lbo = sbo; sbo = t;
#endif
  return static_cast<uint64_t>((addr & 0x3ffffu) >> 4) | (static_cast<uint64_t>(lbo >> 4) << 16) |
         (static_cast<uint64_t>(sbo >> 4) << 32) | (1ull << 46);
}

// DET (deterministic mode): the CTA's accumulator is STORED into its own row of the dw slab (every one of the 27 x 8 x 8 entries
// is written once); det_finalize adds the rows in CTA order. A CTA's blocks are blockIdx.x + k gridDim.x, so a row's content
// depends on the grid size only.
template <bool DET>
__device__ __forceinline__ void wgrad_tc8_body(const CUtensorMap& tmX, const CUtensorMap& tmZ, const WtArgs& args) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sBar = smem_base + WT_STAGES * WT_STAGE;
  const uint32_t bar_full = sBar, bar_empty = sBar + 8 * WT_STAGES, bar_done = sBar + 16 * WT_STAGES, tmem_slot = bar_done + 8;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const int segs = (args.W + WT_KSEG - 1) / WT_KSEG, hblocks = (args.H + WT_R - 1) / WT_R;
  const int num_blocks = args.D * hblocks * segs;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmZ);
    for (int s = 0; s < WT_STAGES; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    mbar_init(bar_done, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<WT_TMEM_COLS>(tmem_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      uint32_t it = 0;
      for (int blk = blockIdx.x; blk < num_blocks; blk += gridDim.x, ++it) {
        const int seg = blk % segs, hb = (blk / segs) % hblocks, z0 = blk / (segs * hblocks);
        const int x0 = seg * WT_KSEG, yb = hb * WT_R;
        const uint32_t s = it % WT_STAGES;
        mbar_wait(bar_empty + 8 * s, ((it / WT_STAGES) & 1) ^ 1u);
        const uint32_t sX = smem_base + s * WT_STAGE, sZ = sX + WT_X_BYTES, bar = bar_full + 8 * s;
        mbar_arrive_expect_tx(bar, WT_TX_BYTES);
        for (int r = 0; r < WT_R; ++r)  // voxels x0 - 8 .. x0 + KSEG + 7 of row yb + r
          tma_load_4d(sX + r * WT_XARR, &tmX, bar, 0, x0 / 8 - 1, yb + r, z0);
        for (int rr = 0; rr < WT_R + 2; ++rr)
          for (int kd = 0; kd < 3; ++kd)
            tma_load_4d(sZ + (rr * 3 + kd) * WT_ZARR, &tmZ, bar, 0, x0 / 8, yb - 1 + rr, z0 - (kd - 1) * args.dil);
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (warp-uniform, one elected lane)
    constexpr uint32_t idesc = umma_idesc_bf16_f32(WT_M, WT_N) | (1u << 15) | (1u << 16);  // A and B MN-major
    uint32_t it = 0;
    for (int blk = blockIdx.x; blk < num_blocks; blk += gridDim.x, ++it) {
      const uint32_t s = it % WT_STAGES;
      mbar_wait(bar_full + 8 * s, (it / WT_STAGES) & 1);
      tcgen05_fence_after();
      if (elect_one_sync()) {
        const uint32_t sX = smem_base + s * WT_STAGE, sZ = sX + WT_X_BYTES;
#pragma unroll 1
        for (int r = 0; r < WT_R; ++r) {
          // A: row r from voxel x0 - 1 (array voxel 7); B: the nine dZ arrays (rows r .. r + 2 of the stage, three planes)
          const uint64_t ad = wt_desc(sX + r * WT_XARR + 7 * 16, 128, 16);
          const uint64_t bd = wt_desc(sZ + r * 3 * WT_ZARR, 128, WT_ZARR);
#pragma unroll
          for (int ks = 0; ks < WT_KSEG / 16; ++ks)  // 16 voxels = 256 bytes further on in both operands
            umma_bf16(tmem_base, ad + 16 * ks, bd + 16 * ks, idesc, (it | r | ks) != 0);
        }
        umma_commit(bar_empty + 8 * s);
      }
      __syncwarp();
    }
    if (elect_one_sync()) umma_commit(bar_done);
    __syncwarp();
  } else if (warp == 4 || (WT_M == 64 && warp == 5)) {
    // ------------------------------------------------------------------ read-out: accumulator row m = (kw, ci) < 24.
    // M = 128: TMEM lane = row. M = 64: rows 16 q .. 16 q + 15 sit in lanes 32 q .. 32 q + 15 (one 16-lane slice per warp quarter).
    mbar_wait(bar_done, 0);
    tcgen05_fence_after();
    {
      const int q = warp & 3;
      const int m = WT_M == 64 ? (lane < 16 ? q * 16 + lane : 99) : lane;
      const int kw = m >> 3, ci = m & 7;
#pragma unroll 1
      for (int c = 0; c < 5; ++c) {
        uint32_t v[16];
        tmem_ld_32x16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + c * 16, v);
        tmem_ld_wait();
        if (m < 24) {
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const int n = c * 16 + i;
            if (n < 72) {
              const int co = n & 7, blkn = n >> 3, yr = blkn / 3, kd = blkn - 3 * yr, kh = 2 - yr;
              if constexpr (DET)
                args.dw[(size_t)blockIdx.x * 27 * 64 + (((kd * 3 + kh) * 3 + kw) * 8 + co) * 8 + ci] = __uint_as_float(v[i]);
              else
                atomicAdd(args.dw + ((((kd * 3 + kh) * 3 + kw) * 8 + co) * 8 + ci), __uint_as_float(v[i]));
            }
          }
        }
      }
    }
    tcgen05_fence_before();
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tcgen05_fence_after();
    tmem_dealloc<WT_TMEM_COLS>(tmem_base);
  }
}

__global__ void __launch_bounds__(WT_THREADS, 1)
wgrad_tc8_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmZ, const WtArgs args) {
  wgrad_tc8_body<false>(tmX, tmZ, args);
}

__global__ void __launch_bounds__(WT_THREADS, 1)
wgrad_tc8_det_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmZ, const WtArgs args) {
  wgrad_tc8_body<true>(tmX, tmZ, args);
}

// ------------------------------------------------------------------------------------------------------------------
// 16 / 32 channels: the same formulation with the volumes split into 8-channel chunks. TMA boxes of (8 channels, one
// chunk, KSEG voxels) land as [voxel][8] arrays, i.e. the operand layout above; the accumulator rows are
// m = (kw * NCX + j) * 8 + t (array (kw, j) = chunk j of the row shifted by kw - 1 voxels: with more than one chunk per
// voxel the column taps are separate arrays, equally spaced), the columns n = ((yr * 3 + kd) * NCZ + jz) * 8 + t'.
// One MMA (M 128, N 144) per 16 voxels and 144 columns: 96 x 144 useful of 128 x 144 for 32 -> 16.
// Loader of the chunk arrays: TMA boxes (default) or, with -DWTN_CPASYNC=1, four warps of 16-byte cp.async (A/B arm, measured
// SLOWER: 32 -> 16 1.16 ms against 0.70 ms, 16 -> 16 0.95 against 0.52 -- an LDGSTS warp instruction with 32 scattered 16-byte
// destinations costs ~58 cycles on this chip, 9 B/clk/SM against TMA's 14; profiles/r02_train_notes.md).
#ifndef WTN_CPASYNC
#define WTN_CPASYNC 0
#endif
__device__ __forceinline__ void wt_cp_async16_ca(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void wt_cp_async16_cg(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}

template <int CIN, int COUT, int R, int KSEG>
struct WtnCfg {
  static constexpr int NCX = CIN / 8, NCZ = COUT / 8;
  static constexpr int S = KSEG * 16;                              // one [KSEG][8] array
  static constexpr int XA = R * 3 * NCX, ZA = (R + 2) * 3 * NCZ;   // arrays per stage
  static constexpr int STAGE = ((XA + ZA) * S + 1023) / 1024 * 1024;
  static constexpr int STAGES_RAW = (227 * 1024 - 2048) / STAGE;
  static constexpr int STAGES = STAGES_RAW > 4 ? 4 : STAGES_RAW;
  static constexpr int SMEM = STAGES * STAGE + 256 + 1024;
  static constexpr int MROWS = 24 * NCX;
  static constexpr int MM = MROWS <= 64 ? 64 : 128;                // MMA height
  static constexpr int N = 72 * NCZ, NSPLIT = N > 256 ? 2 : 1, NH = N / NSPLIT;
  static constexpr int TMEM_COLS = N <= 128 ? 128 : N <= 256 ? 256 : 512;
  static constexpr uint32_t TX_BYTES = (XA + ZA) * S;
  static_assert(NCX >= 2 && NCZ >= 2 && NH % 16 == 0 && NH <= 256 && STAGES >= 2, "unsupported layer");
  static_assert(16 <= XA - 3 * NCX * (R - 1) + ZA, "M = 128 over-reads 16 arrays from the last row's first");
};

template <int CIN, int COUT, int R, int KSEG>
__global__ void __launch_bounds__(WT_THREADS, 1)
wgrad_tcn_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmZ, const WtArgs args) {
  using Cfg = WtnCfg<CIN, COUT, R, KSEG>;
  constexpr int STAGES = Cfg::STAGES, S = Cfg::S, NCX = Cfg::NCX, NCZ = Cfg::NCZ;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sBar = smem_base + STAGES * Cfg::STAGE;
  const uint32_t bar_full = sBar, bar_empty = sBar + 8 * STAGES, bar_done = sBar + 16 * STAGES, tmem_slot = bar_done + 8;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const int segs = (args.W + KSEG - 1) / KSEG, hblocks = (args.H + R - 1) / R;
  const int num_blocks = args.D * hblocks * segs;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmZ);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(bar_full + 8 * s, WTN_CPASYNC ? 4 : 1);  // one arrival per loader warp / the TMA transaction count
      mbar_init(bar_empty + 8 * s, 1);
    }
    mbar_init(bar_done, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  if (warp == 0) {
#if !WTN_CPASYNC
    // ------------------------------------------------------------------ TMA producer: the whole warp issues boxes
    // (A/B arm: boxes with a 16-byte inner extent move ~14 B/clk/SM, which bounds the kernel: 0.70 ms for 32 -> 16)
    uint32_t it = 0;
    for (int blk = blockIdx.x; blk < num_blocks; blk += gridDim.x, ++it) {
      const int seg = blk % segs, hb = (blk / segs) % hblocks, z0 = blk / (segs * hblocks);
      const int x0 = seg * KSEG, yb = hb * R;
      const uint32_t s = it % STAGES;
      const uint32_t sX = smem_base + s * Cfg::STAGE, sZ = sX + Cfg::XA * S, bar = bar_full + 8 * s;
      if (lane == 0) {
        mbar_wait(bar_empty + 8 * s, ((it / STAGES) & 1) ^ 1u);
        mbar_arrive_expect_tx(bar, Cfg::TX_BYTES);
      }
      __syncwarp();
      for (int i = lane; i < Cfg::XA; i += 32) {  // array i = (r * 3 + kw) * NCX + j
        const int j = i % NCX, kw = (i / NCX) % 3, r = i / (3 * NCX);
        tma_load_5d(sX + i * S, &tmX, bar, 0, j, x0 - 1 + kw, yb + r, z0);
      }
      for (int i = lane; i < Cfg::ZA; i += 32) {  // array i = (rr * 3 + kd) * NCZ + jz
        const int jz = i % NCZ, kd = (i / NCZ) % 3, rr = i / (3 * NCZ);
        tma_load_5d(sZ + i * S, &tmZ, bar, 0, jz, x0, yb - 1 + rr, z0 - (kd - 1) * args.dil);
      }
    }
#endif
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc = umma_idesc_bf16_f32(Cfg::MM, Cfg::NH) | (1u << 15) | (1u << 16);  // A and B MN-major
    uint32_t it = 0;
    for (int blk = blockIdx.x; blk < num_blocks; blk += gridDim.x, ++it) {
      const uint32_t s = it % STAGES;
      mbar_wait(bar_full + 8 * s, (it / STAGES) & 1);
      tcgen05_fence_after();
      if (elect_one_sync()) {
        const uint32_t sX = smem_base + s * Cfg::STAGE, sZ = sX + Cfg::XA * S;
#pragma unroll 1
        for (int r = 0; r < R; ++r) {
          const uint64_t ad = wt_desc(sX + r * 3 * NCX * S, 128, S);
#pragma unroll
          for (int h = 0; h < Cfg::NSPLIT; ++h) {
            const uint64_t bd = wt_desc(sZ + (r * 3 * NCZ + h * (Cfg::NH / 8)) * S, 128, S);
#pragma unroll
            for (int ks = 0; ks < KSEG / 16; ++ks)
              umma_bf16(tmem_base + h * Cfg::NH, ad + 16 * ks, bd + 16 * ks, idesc, (it | r | ks) != 0);
          }
        }
        umma_commit(bar_empty + 8 * s);
      }
      __syncwarp();
    }
    if (elect_one_sync()) umma_commit(bar_done);
    __syncwarp();
  } else {
#if WTN_CPASYNC
    // ------------------------------------------------------------------ loaders (warps 2-5): global -> chunk arrays, cp.async
    // A row segment is contiguous in global memory: consecutive threads copy consecutive 16-byte chunks (chunk c = voxel
    // c / NC, channel block c % NC) to array (c % NC) -- and, for x, to the three column-tap arrays, shifted by one voxel
    // each (the second and third read of a chunk hit L1). Zero fill is the padding. A thread signals stage n - 1 after
    // issuing stage n (cp.async.wait_group 1, proxy fence, one arrival per warp): two stages of loads in flight.
    {
      const int t = threadIdx.x - 64;
      uint32_t it = 0;
      for (int blk = blockIdx.x; blk < num_blocks; blk += gridDim.x, ++it) {
        const int seg = blk % segs, hb = (blk / segs) % hblocks, z0 = blk / (segs * hblocks);
        const int x0 = seg * KSEG, yb = hb * R;
        const uint32_t s = it % STAGES;
        const uint32_t sX = smem_base + s * Cfg::STAGE, sZ = sX + Cfg::XA * S;
        mbar_wait(bar_empty + 8 * s, ((it / STAGES) & 1) ^ 1u);
#pragma unroll 1
        for (int r = 0; r < R; ++r) {
          const int y = yb + r;
          const bool row_ok = y < args.H;
          const __nv_bfloat16* src_row = args.x + (((int64_t)z0 * args.H + (row_ok ? y : 0)) * args.W) * CIN;
          for (int c = t; c < (KSEG + 2) * NCX; c += 128) {
            const int v = c / NCX, j = c % NCX, xg = x0 - 1 + v;
            const bool ok = row_ok && xg >= 0 && xg < args.W;
            const __nv_bfloat16* src = ok ? src_row + (int64_t)xg * CIN + j * 8 : args.x;
            const uint32_t dst = sX + (r * 3 * NCX + j) * S + v * 16;  // array (r, kw = 0, j), voxel v
#pragma unroll
            for (int kw = 0; kw < 3; ++kw) {
              const int k = v - kw;
              if (k >= 0 && k < KSEG) wt_cp_async16_ca(dst + kw * (NCX * S - 16), src, ok ? 16u : 0u);
            }
          }
        }
#pragma unroll 1
        for (int a = 0; a < (R + 2) * 3; ++a) {
          const int rr = a / 3, kd = a - 3 * rr;
          const int y = yb - 1 + rr, z = z0 - (kd - 1) * args.dil;
          const bool row_ok = y >= 0 && y < args.H && z >= 0 && z < args.D;
          const __nv_bfloat16* src_row = args.dz + (((int64_t)(row_ok ? z : 0) * args.H + (row_ok ? y : 0)) * args.W) * COUT;
          for (int c = t; c < KSEG * NCZ; c += 128) {
            const int v = c / NCZ, jz = c % NCZ, xg = x0 + v;
            const bool ok = row_ok && xg < args.W;
            wt_cp_async16_cg(sZ + (a * NCZ + jz) * S + v * 16, ok ? src_row + (int64_t)xg * COUT + jz * 8 : args.dz, ok ? 16u : 0u);
          }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        if (it > 0) {
          asm volatile("cp.async.wait_group 1;" ::: "memory");
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_full + 8 * ((it - 1) % STAGES));
        }
      }
      if (it > 0) {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_full + 8 * ((it - 1) % STAGES));
      }
    }
#endif
    // ------------------------------------------------------------------ read-out: TMEM lane = (kw, j, t)
    const int q = warp & 3;
    mbar_wait(bar_done, 0);
    tcgen05_fence_after();
    // M = 128: TMEM lane = accumulator row; M = 64: rows 16 q .. 16 q + 15 sit in lanes 32 q .. 32 q + 15
    const int m = Cfg::MM == 64 ? (lane < 16 ? q * 16 + lane : Cfg::MROWS) : q * 32 + lane;
    if ((Cfg::MM == 64 ? q * 16 : q * 32) < Cfg::MROWS) {
      const int t = m & 7, j = (m >> 3) % NCX, kw = m / (8 * NCX), ci = j * 8 + t;
#pragma unroll 1
      for (int c2 = 0; c2 < Cfg::N / 16; ++c2) {  // two column blocks c = (yr * 3 + kd) * NCZ + jz at a time
        uint32_t v[16];
        tmem_ld_32x16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + c2 * 16, v);
        tmem_ld_wait();
        if (m < Cfg::MROWS) {
#pragma unroll
          for (int hb = 0; hb < 2; ++hb) {
            const int c = 2 * c2 + hb;
            const int jz = c % NCZ, rest = c / NCZ, yr = rest / 3, kd = rest - 3 * yr, kh = 2 - yr;
            float* dst = args.dw + ((size_t)(((kd * 3 + kh) * 3 + kw) * COUT + jz * 8) * CIN + ci);
#pragma unroll
            for (int i = 0; i < 8; ++i) atomicAdd(dst + (size_t)i * CIN, __uint_as_float(v[hb * 8 + i]));
          }
        }
      }
    }
    tcgen05_fence_before();
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tcgen05_fence_after();
    tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

template <int CIN, int COUT, int R, int KSEG>
static int launch_wgrad_tcn(const void* x, const void* dz, float* dw, int64_t D, int64_t H, int64_t W, int64_t dil, cudaStream_t stream) {
  using Cfg = WtnCfg<CIN, COUT, R, KSEG>;
  CUtensorMap tmX, tmZ;
  // (8 channels, chunk, x, y, z)
  uint64_t dimsX[5] = {8, (uint64_t)Cfg::NCX, (uint64_t)W, (uint64_t)H, (uint64_t)D};
  uint64_t strX[5] = {0, 16, (uint64_t)CIN * 2, (uint64_t)W * CIN * 2, (uint64_t)H * W * CIN * 2};
  uint64_t dimsZ[5] = {8, (uint64_t)Cfg::NCZ, (uint64_t)W, (uint64_t)H, (uint64_t)D};
  uint64_t strZ[5] = {0, 16, (uint64_t)COUT * 2, (uint64_t)W * COUT * 2, (uint64_t)H * W * COUT * 2};
  uint32_t box[5] = {8, 1, KSEG, 1, 1};
  int rc = encode_tmap(&tmX, TmapDtype::BF16, 5, x, dimsX, strX, box, 0);
  if (rc) return rc;
  rc = encode_tmap(&tmZ, TmapDtype::BF16, 5, dz, dimsZ, strZ, box, 0);
  if (rc) return rc;
  auto kern = wgrad_tcn_kernel<CIN, COUT, R, KSEG>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM);
    if (e != cudaSuccess) {
      set_error("wgrad_tcn: cudaFuncSetAttribute(smem=%d): %s", Cfg::SMEM, cudaGetErrorString(e));
      return CVIT_ERR_CUDA;
    }
    configured = true;
  }
  const int64_t blocks = D * ((H + R - 1) / R) * ((W + KSEG - 1) / KSEG);
  int grid = num_sms();
  if (grid > blocks) grid = (int)blocks;
  WtArgs a;
  a.dw = dw;
  a.x = static_cast<const __nv_bfloat16*>(x);
  a.dz = static_cast<const __nv_bfloat16*>(dz);
  a.D = (int)D;
  a.H = (int)H;
  a.W = (int)W;
  a.dil = (int)dil;
  kern<<<grid, WT_THREADS, Cfg::SMEM, stream>>>(tmX, tmZ, a);
  return check_launch("wgrad_tcn_kernel");
}

// ------------------------------------------------------------------------------------------------------------------
// The same kernel fed differently (default): TMA moves WHOLE ROWS of both volumes (boxes {all channels, voxels, rows}: 32- / 64-byte
// inner extents, four boxes per stage) into a raw staging buffer, and the four otherwise idle warps de-interleave them into the
// 8-channel chunk arrays with LDS.128 / STS.128 -- writing each x chunk to its three column-tap arrays, so x is fetched once
// instead of three times. The chunk boxes of wgrad_tcn_kernel (16-byte inner extent) arrive at ~14 B/clk/SM and bound it.
template <int CIN, int COUT, int R, int KSEG, int RS>
struct WtsCfg {
  static constexpr int NCX = CIN / 8, NCZ = COUT / 8;
  static constexpr int S = KSEG * 16;
  static constexpr int XA = R * 3 * NCX, ZA = (R + 2) * 3 * NCZ;
  static constexpr int ARR_STAGE = (XA + ZA) * S;
  static constexpr int RAW_X = (R * (KSEG + 2) * CIN * 2 + 127) / 128 * 128;
  static constexpr int RAW_ZP = (R + 2) * KSEG * COUT * 2;  // one plane's rows
  static constexpr int RAW_STAGE = RAW_X + 3 * RAW_ZP;
  // RS raw stages: the kernel is bound by bytes in flight x L2 latency (~2 us under load: 2 x 33 KB per SM gave 3.9 TB/s
  // aggregate, exactly what the chunk-box version reached), so the raw ring is as deep as shared memory allows
  static constexpr int SMEM = 2 * ARR_STAGE + RS * RAW_STAGE + 256 + 1024;
  static constexpr int MROWS = 24 * NCX;
  static constexpr int MM = MROWS <= 64 ? 64 : 128;
  static constexpr int N = 72 * NCZ, NSPLIT = N > 256 ? 2 : 1, NH = N / NSPLIT;
  static constexpr int TMEM_COLS = N <= 128 ? 128 : N <= 256 ? 256 : 512;
  static constexpr uint32_t TX_BYTES = R * (KSEG + 2) * CIN * 2 + 3 * RAW_ZP;
  static_assert(NCX >= 2 && NCZ >= 2 && NH % 16 == 0 && NH <= 256 && SMEM <= 232448 && RAW_ZP % 128 == 0, "unsupported layer");
  static_assert(16 <= XA - 3 * NCX * (R - 1) + ZA, "M = 128 over-reads 16 arrays from the last row's first");
};

// DET: as wgrad_tc8_body, one [27][COUT][CIN] row per CTA.
template <int CIN, int COUT, int R, int KSEG, int RS, bool DET>
__device__ __forceinline__ void wgrad_tcs_body(const CUtensorMap& tmX, const CUtensorMap& tmZ, const WtArgs& args) {
  using Cfg = WtsCfg<CIN, COUT, R, KSEG, RS>;
  constexpr int S = Cfg::S, NCX = Cfg::NCX, NCZ = Cfg::NCZ;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sArr = smem_base, sRaw = smem_base + 2 * Cfg::ARR_STAGE, sBar = sRaw + RS * Cfg::RAW_STAGE;
  const uint32_t raw_full = sBar, raw_empty = sBar + 8 * RS, arr_full = sBar + 16 * RS, arr_empty = arr_full + 16, bar_done = arr_full + 32,
                 tmem_slot = arr_full + 40;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const int segs = (args.W + KSEG - 1) / KSEG, hblocks = (args.H + R - 1) / R;
  const int num_blocks = args.D * hblocks * segs;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmZ);
    for (int s = 0; s < RS; ++s) {
      mbar_init(raw_full + 8 * s, 1);
      mbar_init(raw_empty + 8 * s, 4);   // one arrival per copy warp
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(arr_full + 8 * s, 4);
      mbar_init(arr_empty + 8 * s, 1);   // the MMAs that read the arrays have retired
    }
    mbar_init(bar_done, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer: four boxes of whole rows per stage
    if (lane == 0) {
      uint32_t it = 0;
      for (int blk = blockIdx.x; blk < num_blocks; blk += gridDim.x, ++it) {
        const int seg = blk % segs, hb = (blk / segs) % hblocks, z0 = blk / (segs * hblocks);
        const int x0 = seg * KSEG, yb = hb * R;
        const uint32_t s = it % RS, dst = sRaw + s * Cfg::RAW_STAGE, bar = raw_full + 8 * s;
        mbar_wait(raw_empty + 8 * s, ((it / RS) & 1) ^ 1u);
        mbar_arrive_expect_tx(bar, Cfg::TX_BYTES);
        tma_load_4d(dst, &tmX, bar, 0, x0 - 1, yb, z0);  // [R][KSEG + 2][CIN]
#pragma unroll
        for (int kd = 0; kd < 3; ++kd)                   // [R + 2][KSEG][COUT] of plane z0 - (kd - 1) dil
          tma_load_4d(dst + Cfg::RAW_X + kd * Cfg::RAW_ZP, &tmZ, bar, 0, x0, yb - 1, z0 - (kd - 1) * args.dil);
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc = umma_idesc_bf16_f32(Cfg::MM, Cfg::NH) | (1u << 15) | (1u << 16);  // A and B MN-major
    uint32_t it = 0;
    for (int blk = blockIdx.x; blk < num_blocks; blk += gridDim.x, ++it) {
      const uint32_t s = it & 1;
      mbar_wait(arr_full + 8 * s, (it >> 1) & 1);
      tcgen05_fence_after();
      if (elect_one_sync()) {
        const uint32_t sX = sArr + s * Cfg::ARR_STAGE, sZ = sX + Cfg::XA * S;
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const uint64_t ad = wt_desc(sX + r * 3 * NCX * S, 128, S);
#pragma unroll
          for (int h = 0; h < Cfg::NSPLIT; ++h) {
            const uint64_t bd = wt_desc(sZ + (r * 3 * NCZ + h * (Cfg::NH / 8)) * S, 128, S);
#pragma unroll
            for (int ks = 0; ks < KSEG / 16; ++ks)
              umma_bf16(tmem_base + h * Cfg::NH, ad + 16 * ks, bd + 16 * ks, idesc, (it | r | ks) != 0);
          }
        }
        umma_commit(arr_empty + 8 * s);
      }
      __syncwarp();
    }
    if (elect_one_sync()) umma_commit(bar_done);
    __syncwarp();
  } else {
    // ------------------------------------------------------------------ warps 2-5: raw rows -> chunk arrays, then the read-out
    {
      const int t = threadIdx.x - 64;
      uint32_t it = 0;
      for (int blk = blockIdx.x; blk < num_blocks; blk += gridDim.x, ++it) {
        const uint32_t s = it & 1, rs = it % RS;
        const uint32_t rX = sRaw + rs * Cfg::RAW_STAGE, rZ = rX + Cfg::RAW_X;
        const uint32_t aX = sArr + s * Cfg::ARR_STAGE, aZ = aX + Cfg::XA * S;
        mbar_wait(raw_full + 8 * rs, (it / RS) & 1);
        mbar_wait(arr_empty + 8 * s, ((it >> 1) & 1) ^ 1u);
        // x: chunk (voxel v = x0 - 1 + .., channel block j) of row r -> arrays (r, kw, j) at voxel v - kw. A thread keeps its
        // channel block and strides over the voxels (no division per chunk: the copy is instruction-bound otherwise).
        {
          const int j = t % NCX;
#pragma unroll
          for (int r = 0; r < R; ++r) {
#pragma unroll 2
            for (int v = t / NCX; v < KSEG + 2; v += 128 / NCX) {
              uint32_t a, b, cc, d;
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(cc), "=r"(d)
                           : "r"(rX + ((r * (KSEG + 2) + v) * NCX + j) * 16));
              const uint32_t dst = aX + (r * 3 * NCX + j) * S + v * 16;  // array (r, kw = 0, j), voxel v
#pragma unroll
              for (int kw = 0; kw < 3; ++kw) {
                const int k = v - kw;
                if (k >= 0 && k < KSEG)
                  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst + kw * (NCX * S - 16)), "r"(a), "r"(b), "r"(cc), "r"(d) : "memory");
              }
            }
          }
        }
        // dz: raw [kd][rr][v][jz] -> array ((rr * 3 + kd) * NCZ + jz), voxel v: a row is KSEG * NCZ = 128 chunks, one per thread
        {
          static_assert(KSEG * NCZ == 128, "one dz chunk per copy thread and row");
          const int v = t / NCZ, jz = t % NCZ;
#pragma unroll
          for (int kd = 0; kd < 3; ++kd)
#pragma unroll
            for (int rr = 0; rr < R + 2; ++rr) {
              uint32_t a, b, cc, d;
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(cc), "=r"(d)
                           : "r"(rZ + ((kd * (R + 2) + rr) * 128 + t) * 16));
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(aZ + ((rr * 3 + kd) * NCZ + jz) * S + v * 16), "r"(a), "r"(b),
                           "r"(cc), "r"(d)
                           : "memory");
            }
        }
        fence_proxy_async_smem();  // generic-proxy stores -> visible to the tensor core (async proxy)
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(arr_full + 8 * s);
          mbar_arrive(raw_empty + 8 * rs);
        }
      }
    }
    const int q = warp & 3;
    mbar_wait(bar_done, 0);
    tcgen05_fence_after();
    const int m = Cfg::MM == 64 ? (lane < 16 ? q * 16 + lane : Cfg::MROWS) : q * 32 + lane;
    if ((Cfg::MM == 64 ? q * 16 : q * 32) < Cfg::MROWS) {
      const int tt = m & 7, j = (m >> 3) % NCX, kw = m / (8 * NCX), ci = j * 8 + tt;
#pragma unroll 1
      for (int c2 = 0; c2 < Cfg::N / 16; ++c2) {
        uint32_t v[16];
        tmem_ld_32x16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + c2 * 16, v);
        tmem_ld_wait();
        if (m < Cfg::MROWS) {
#pragma unroll
          for (int hb = 0; hb < 2; ++hb) {
            const int c = 2 * c2 + hb;
            const int jz = c % NCZ, rest = c / NCZ, yr = rest / 3, kd = rest - 3 * yr, kh = 2 - yr;
            float* dst = args.dw + ((size_t)(((kd * 3 + kh) * 3 + kw) * COUT + jz * 8) * CIN + ci);
            if constexpr (DET) {
              dst += (size_t)blockIdx.x * 27 * COUT * CIN;
#pragma unroll
              for (int i = 0; i < 8; ++i) dst[(size_t)i * CIN] = __uint_as_float(v[hb * 8 + i]);
            } else {
#pragma unroll
              for (int i = 0; i < 8; ++i) atomicAdd(dst + (size_t)i * CIN, __uint_as_float(v[hb * 8 + i]));
            }
          }
        }
      }
    }
    tcgen05_fence_before();
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tcgen05_fence_after();
    tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

template <int CIN, int COUT, int R, int KSEG, int RS>
__global__ void __launch_bounds__(WT_THREADS, 1)
wgrad_tcs_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmZ, const WtArgs args) {
  wgrad_tcs_body<CIN, COUT, R, KSEG, RS, false>(tmX, tmZ, args);
}

template <int CIN, int COUT, int R, int KSEG, int RS>
__global__ void __launch_bounds__(WT_THREADS, 1)
wgrad_tcs_det_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmZ, const WtArgs args) {
  wgrad_tcs_body<CIN, COUT, R, KSEG, RS, true>(tmX, tmZ, args);
}

// Grid of the 16 / 32-channel kernels and of wgrad_tc8: one CTA per SM, at most one per block of rows.
static int wgrad_tc_grid(int64_t D, int64_t H, int64_t W, int R, int KSEG) {
  const int64_t blocks = D * ((H + R - 1) / R) * ((W + KSEG - 1) / KSEG);
  int grid = num_sms();
  if (grid > blocks) grid = (int)blocks;
  return grid;
}

// det_slab != null: deterministic mode, dw += the rows of det_slab ([grid][27][COUT][CIN]) added in CTA order.
template <int CIN, int COUT, int R, int KSEG, int RS>
static int launch_wgrad_tcs(const void* x, const void* dz, float* dw, int64_t D, int64_t H, int64_t W, int64_t dil, cudaStream_t stream,
                            float* det_slab = nullptr) {
  using Cfg = WtsCfg<CIN, COUT, R, KSEG, RS>;
  CUtensorMap tmX, tmZ;
  uint64_t dimsX[4] = {(uint64_t)CIN, (uint64_t)W, (uint64_t)H, (uint64_t)D};
  uint64_t strX[4] = {0, (uint64_t)CIN * 2, (uint64_t)W * CIN * 2, (uint64_t)H * W * CIN * 2};
  uint64_t dimsZ[4] = {(uint64_t)COUT, (uint64_t)W, (uint64_t)H, (uint64_t)D};
  uint64_t strZ[4] = {0, (uint64_t)COUT * 2, (uint64_t)W * COUT * 2, (uint64_t)H * W * COUT * 2};
  uint32_t boxX[4] = {(uint32_t)CIN, KSEG + 2, R, 1}, boxZ[4] = {(uint32_t)COUT, KSEG, R + 2, 1};
  int rc = encode_tmap(&tmX, TmapDtype::BF16, 4, x, dimsX, strX, boxX, 0);
  if (rc) return rc;
  rc = encode_tmap(&tmZ, TmapDtype::BF16, 4, dz, dimsZ, strZ, boxZ, 0);
  if (rc) return rc;
  auto kern = det_slab ? wgrad_tcs_det_kernel<CIN, COUT, R, KSEG, RS> : wgrad_tcs_kernel<CIN, COUT, R, KSEG, RS>;
  static bool configured[2] = {false, false};
  if (!configured[det_slab != nullptr]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM);
    if (e != cudaSuccess) {
      set_error("wgrad_tcs: cudaFuncSetAttribute(smem=%d): %s", Cfg::SMEM, cudaGetErrorString(e));
      return CVIT_ERR_CUDA;
    }
    configured[det_slab != nullptr] = true;
  }
  const int64_t blocks = D * ((H + R - 1) / R) * ((W + KSEG - 1) / KSEG);
  int grid = num_sms();
  if (grid > blocks) grid = (int)blocks;
  WtArgs a;
  a.dw = det_slab ? det_slab : dw;
  a.x = static_cast<const __nv_bfloat16*>(x);
  a.dz = static_cast<const __nv_bfloat16*>(dz);
  a.D = (int)D;
  a.H = (int)H;
  a.W = (int)W;
  a.dil = (int)dil;
  kern<<<grid, WT_THREADS, Cfg::SMEM, stream>>>(tmX, tmZ, a);
  if (!det_slab) return check_launch("wgrad_tcs_kernel");
  if (int rc = check_launch("wgrad_tcs_det_kernel")) return rc;
  return det_finalize(det_slab, grid, 27 * COUT * CIN, 27 * COUT * CIN, dw, true, stream);
}

}  // namespace cvit

using namespace cvit;

// dw (fp32 [27][8][8], tap = (kd*3+kh)*3+kw, then co, then ci) += weight gradient of an 8 -> 8 channel 3x3x3 depth-dilated
// "same" convolution: x the forward input, dz the output gradient, both bf16 [D,H,W,8], W a multiple of 8.
static int wgrad_tc8_run(const void* x, const void* dz, float* dw, int64_t D, int64_t H, int64_t W, int64_t dil, void* stream,
                         float* det_slab);

extern "C" int cvit_wgrad_tc8_ndhwc(const void* x, const void* dz, float* dw, int64_t D, int64_t H, int64_t W, int64_t dil,
                                    void* stream) {
  return wgrad_tc8_run(x, dz, dw, D, H, W, dil, stream, nullptr);
}

// Deterministic mode (see wgrad_tc8_body): scratch holds cvit_wgrad_tc8_ndhwc_det_partials(D, H, W) floats, one [27][8][8] row per
// CTA; dw += the rows added in CTA order.
extern "C" int64_t cvit_wgrad_tc8_ndhwc_det_partials(int64_t D, int64_t H, int64_t W) {
  return D > 0 && H > 0 && W > 0 ? (int64_t)wgrad_tc_grid(D, H, W, WT_R, WT_KSEG) * 27 * 64 : 0;
}

extern "C" int cvit_wgrad_tc8_ndhwc_det(const void* x, const void* dz, float* dw, int64_t D, int64_t H, int64_t W, int64_t dil,
                                        float* scratch, int64_t scratch_elems, void* stream) {
  if (D > 0 && H > 0 && W > 0) {
    if (int rc = det_check_scratch(scratch, scratch_elems, cvit_wgrad_tc8_ndhwc_det_partials(D, H, W), "wgrad_tc8_det")) return rc;
  }
  return wgrad_tc8_run(x, dz, dw, D, H, W, dil, stream, scratch);
}

static int wgrad_tc8_run(const void* x, const void* dz, float* dw, int64_t D, int64_t H, int64_t W, int64_t dil, void* stream,
                         float* det_slab) {
  if (!x || !dz || !dw || D <= 0 || H <= 0 || W <= 0 || dil <= 0) {
    set_error("wgrad_tc8: bad arguments (D=%lld H=%lld W=%lld dil=%lld)", (long long)D, (long long)H, (long long)W, (long long)dil);
    return CVIT_ERR_INVALID;
  }
  if (W % 8) {
    set_error("wgrad_tc8: W=%lld must be a multiple of 8 (use cvit_wgrad_narrow_ndhwc otherwise)", (long long)W);
    return CVIT_ERR_UNSUPPORTED;
  }
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dz)) & 15u) {
    set_error("wgrad_tc8: x and dz must be 16-byte aligned");
    return CVIT_ERR_INVALID;
  }
  // both volumes as (128-byte line = 8 voxels x 8 channels, lines per row, rows, planes)
  CUtensorMap tmX, tmZ;
  uint64_t dims[4] = {64, (uint64_t)(W / 8), (uint64_t)H, (uint64_t)D};
  uint64_t strides[4] = {0, 128, (uint64_t)W * 16, (uint64_t)H * W * 16};
  uint32_t boxX[4] = {64, WT_KSEG / 8 + 2, 1, 1}, boxZ[4] = {64, WT_KSEG / 8, 1, 1};
  int rc = encode_tmap(&tmX, TmapDtype::BF16, 4, x, dims, strides, boxX, 0);
  if (rc) return rc;
  rc = encode_tmap(&tmZ, TmapDtype::BF16, 4, dz, dims, strides, boxZ, 0);
  if (rc) return rc;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(wgrad_tc8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WT_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(wgrad_tc8_det_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WT_SMEM);
    if (e != cudaSuccess) {
      set_error("wgrad_tc8: cudaFuncSetAttribute(smem=%d): %s", WT_SMEM, cudaGetErrorString(e));
      return CVIT_ERR_CUDA;
    }
    configured = true;
  }
  const int grid = wgrad_tc_grid(D, H, W, WT_R, WT_KSEG);
  WtArgs a;
  a.dw = det_slab ? det_slab : dw;
  a.x = static_cast<const __nv_bfloat16*>(x);
  a.dz = static_cast<const __nv_bfloat16*>(dz);
  a.D = (int)D;
  a.H = (int)H;
  a.W = (int)W;
  a.dil = (int)dil;
  if (!det_slab) {
    wgrad_tc8_kernel<<<grid, WT_THREADS, WT_SMEM, (cudaStream_t)stream>>>(tmX, tmZ, a);
    return check_launch("wgrad_tc8_kernel");
  }
  wgrad_tc8_det_kernel<<<grid, WT_THREADS, WT_SMEM, (cudaStream_t)stream>>>(tmX, tmZ, a);
  if (int rc = check_launch("wgrad_tc8_det_kernel")) return rc;
  return det_finalize(det_slab, grid, 27 * 64, 27 * 64, dw, true, (cudaStream_t)stream);
}

// The 16- / 32-channel layers (SynthesisBlocks 3-4): (Cin, Cout) in {(16,16), (32,16), (32,32)}, any W. Same contract as
// cvit_wgrad_narrow_ndhwc: dw fp32 [27][Cout][Cin] accumulated into.
extern "C" int cvit_wgrad_tcn_ndhwc(const void* x, const void* dz, float* dw, int64_t D, int64_t H, int64_t W, int64_t Cin,
                                    int64_t Cout, int64_t dil, void* stream) {
  if (!x || !dz || !dw || D <= 0 || H <= 0 || W <= 0 || dil <= 0) {
    set_error("wgrad_tcn: bad arguments (D=%lld H=%lld W=%lld dil=%lld)", (long long)D, (long long)H, (long long)W, (long long)dil);
    return CVIT_ERR_INVALID;
  }
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dz)) & 15u) {
    set_error("wgrad_tcn: x and dz must be 16-byte aligned");
    return CVIT_ERR_INVALID;
  }
  cudaStream_t st = (cudaStream_t)stream;
  // default: whole rows by TMA + shared-memory de-interleave (wgrad_tcs_kernel); CVIT_WGRAD_CHUNK_TMA=1: 16-byte chunk boxes (A/B arm)
  static const bool chunk_tma = getenv("CVIT_WGRAD_CHUNK_TMA") && atoi(getenv("CVIT_WGRAD_CHUNK_TMA")) != 0;
  if (!chunk_tma) {
    if (Cin == 16 && Cout == 16) return launch_wgrad_tcs<16, 16, 4, 64, 2>(x, dz, dw, D, H, W, dil, st);
    if (Cin == 32 && Cout == 16) return launch_wgrad_tcs<32, 16, 2, 64, 3>(x, dz, dw, D, H, W, dil, st);
    if (Cin == 32 && Cout == 32) return launch_wgrad_tcs<32, 32, 2, 32, 5>(x, dz, dw, D, H, W, dil, st);
  }
  if (Cin == 16 && Cout == 16) return launch_wgrad_tcn<16, 16, 4, 64>(x, dz, dw, D, H, W, dil, st);
  if (Cin == 32 && Cout == 16) return launch_wgrad_tcn<32, 16, 4, 64>(x, dz, dw, D, H, W, dil, st);
  if (Cin == 32 && Cout == 32) return launch_wgrad_tcn<32, 32, 2, 64>(x, dz, dw, D, H, W, dil, st);
  set_error("wgrad_tcn: (Cin, Cout) = (%lld, %lld) unsupported: (16,16), (32,16), (32,32)", (long long)Cin, (long long)Cout);
  return CVIT_ERR_UNSUPPORTED;
}

// Deterministic mode of cvit_wgrad_tcn_ndhwc: always the whole-row kernel (wgrad_tcs_body), one [27][Cout][Cin] row per CTA in
// scratch (cvit_wgrad_tcn_ndhwc_det_partials floats), dw += the rows added in CTA order.
extern "C" int64_t cvit_wgrad_tcn_ndhwc_det_partials(int64_t D, int64_t H, int64_t W, int64_t Cin, int64_t Cout) {
  if (D <= 0 || H <= 0 || W <= 0) return 0;
  int grid = 0;
  if (Cin == 16 && Cout == 16) grid = wgrad_tc_grid(D, H, W, 4, 64);
  else if (Cin == 32 && Cout == 16) grid = wgrad_tc_grid(D, H, W, 2, 64);
  else if (Cin == 32 && Cout == 32) grid = wgrad_tc_grid(D, H, W, 2, 32);
  return (int64_t)grid * 27 * Cin * Cout;
}

extern "C" int cvit_wgrad_tcn_ndhwc_det(const void* x, const void* dz, float* dw, int64_t D, int64_t H, int64_t W, int64_t Cin,
                                        int64_t Cout, int64_t dil, float* scratch, int64_t scratch_elems, void* stream) {
  if (!x || !dz || !dw || D <= 0 || H <= 0 || W <= 0 || dil <= 0) {
    set_error("wgrad_tcn_det: bad arguments (D=%lld H=%lld W=%lld dil=%lld)", (long long)D, (long long)H, (long long)W, (long long)dil);
    return CVIT_ERR_INVALID;
  }
  if (int rc = det_check_scratch(scratch, scratch_elems, cvit_wgrad_tcn_ndhwc_det_partials(D, H, W, Cin, Cout), "wgrad_tcn_det")) return rc;
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dz)) & 15u) {
    set_error("wgrad_tcn_det: x and dz must be 16-byte aligned");
    return CVIT_ERR_INVALID;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (Cin == 16 && Cout == 16) return launch_wgrad_tcs<16, 16, 4, 64, 2>(x, dz, dw, D, H, W, dil, st, scratch);
  if (Cin == 32 && Cout == 16) return launch_wgrad_tcs<32, 16, 2, 64, 3>(x, dz, dw, D, H, W, dil, st, scratch);
  if (Cin == 32 && Cout == 32) return launch_wgrad_tcs<32, 32, 2, 32, 5>(x, dz, dw, D, H, W, dil, st, scratch);
  set_error("wgrad_tcn_det: (Cin, Cout) = (%lld, %lld) unsupported: (16,16), (32,16), (32,32)", (long long)Cin, (long long)Cout);
  return CVIT_ERR_UNSUPPORTED;
}
