// Weight gradients of the WIDE layers of the CryoVIT head (>= 64 channels: the 3x3x3 convolutions of SynthesisBlocks 1-2,
// the transposed convolutions, the 1x1x1 projection; head training, BASELINE config 5) as split-K tcgen05 GEMMs STRAIGHT
// FROM THE CHANNELS-LAST VOLUMES:
//
//   dW[tap][m][n] = sum over voxels v of  P[v + off(tap)][m] * Q[v][n]        (P, Q = x and dZ in either order)
//
// The reduction runs over voxels, and a channels-last tile [64 voxels][64 channels] staged by TMA with the 128-byte
// swizzle IS a tensor-core operand whose contiguous dimension is M (resp. N): an MN-major SWIZZLE_128B atom stack (the
// layout attention feeds V with and the head's projection reads the on-disk features with). So both operands are TMA
// boxes of the tensors as they lie -- no channels-first copies, no zero-padded copies, no three column-shifted copies
// (csrc/wgrad.cu needed all of them: 25 launches and 2.9 ms of a 28 ms training step) -- and the tap is nothing but the
// box origin of the shifted operand: (w0 + kw - 1, h0 + kh - 1, d + (kd - 1) dil), with TMA's out-of-bounds zero fill as
// the convolution's padding; K chunks whose depth tap leaves the volume are skipped. 1x1x1 and transposed convolutions
// are the one-tap case over a [rows][channels] matrix (W = rows, H = D = 1).
//
// A K chunk is a 64-voxel patch (BW x BH) of one depth plane; a work item is (tap, 128-row M tile, BN-column N tile, range
// of K chunks); items accumulate in TMEM (two buffers) and add their partial tile into the fp32 result with
// red.global.add (the caller zeroes it). One CTA per SM, 192 threads: TMA producer, MMA issuer (warp-uniform,
// elect.sync), four epilogue warps (thread = output row).
#include "det_reduce.cuh"
#include "ptx.cuh"
#include "tmap.h"

namespace cvit {

constexpr int WM_BM = 128, WM_KC = 64, WM_THREADS = 192;
constexpr int WM_BLOCK = WM_KC * 128;  // one [64 voxels][64 channels] box: 8 KB

template <int BN>
struct WmCfg {
  static constexpr int A_BYTES = (WM_BM / 64) * WM_BLOCK, B_BYTES = (BN / 64) * WM_BLOCK, STAGE = A_BYTES + B_BYTES;
  static constexpr int STAGES_RAW = (200 * 1024) / STAGE;
  static constexpr int STAGES = STAGES_RAW > 8 ? 8 : STAGES_RAW;
  static constexpr int ACC = BN <= 64 ? 64 : BN <= 128 ? 128 : 256;
  static constexpr int TMEM_COLS = 2 * ACC;
  static constexpr int SMEM = STAGES * STAGE + 256 + 1024;
  static_assert(BN % 64 == 0 && BN <= 256, "N tile = whole 64-channel boxes");
};

struct WmArgs {
  float* out;          // [ntaps][M][N] fp32, accumulated into (deterministic mode: [ksplit][ntaps][M][N], stored)
  int M, N;            // channels of the A operand / of the B operand
  int D, H, W, dil;    // voxel grid both operands live on (rows mode: W = rows, H = D = 1)
  int BW, BH;          // K chunk = BW x BH voxels of one plane (BW * BH == 64)
  int ntaps;           // 27 (3x3x3, tap = (kd*3+kh)*3+kw) or 1
  int shift_a;         // 1: the tap shifts the A operand's box, 0: the B operand's
  int ksplit;
};

// DET (deterministic mode): an item's tile is STORED into K slice ks of the [ksplit][ntaps][M][N] slab (zeros when every
// chunk was skipped), and det_finalize adds the slices in ks order.
template <int BN, bool DET>
__device__ __forceinline__ void wgrad_mn_body(const CUtensorMap& tmA, const CUtensorMap& tmB, const WmArgs& args) {
  using Cfg = WmCfg<BN>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sA = smem_base, sB = smem_base + STAGES * Cfg::A_BYTES;
  const uint32_t sBar = smem_base + STAGES * Cfg::STAGE;
  const uint32_t bar_full = sBar, bar_empty = sBar + 8 * STAGES;
  const uint32_t bar_tfull = sBar + 16 * STAGES, bar_tempty = bar_tfull + 16, tmem_slot = bar_tempty + 16;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const int m_tiles = (args.M + WM_BM - 1) / WM_BM, n_tiles = (args.N + BN - 1) / BN;
  const int tiles_w = (args.W + args.BW - 1) / args.BW, tiles_h = (args.H + args.BH - 1) / args.BH;
  const int per_plane = tiles_w * tiles_h;
  const int k_chunks = args.D * per_plane;
  const int per_tap = m_tiles * n_tiles * args.ksplit;
  const int num_items = args.ntaps * per_tap;
  const int kc_per = (k_chunks + args.ksplit - 1) / args.ksplit;
  auto item_of = [&](int item, int& tap, int& m0, int& n0, int& kc0, int& kc1) {
    tap = item / per_tap;
    int r = item - tap * per_tap;
    const int ks = r % args.ksplit;
    r /= args.ksplit;
    n0 = (r % n_tiles) * BN;
    m0 = (r / n_tiles) * WM_BM;
    kc0 = ks * kc_per;
    kc1 = min(k_chunks, kc0 + kc_per);
  };
  // K chunk -> (d, h0, w0); the tap's offset; whether the shifted plane exists
  auto chunk_of = [&](int kc, int& d, int& h0, int& w0) {
    d = kc / per_plane;
    const int r = kc - d * per_plane;
    const int th = r / tiles_w;
    h0 = th * args.BH;
    w0 = (r - th * tiles_w) * args.BW;
  };
  auto tap_off = [&](int tap, int& dz, int& dy, int& dx) {
    if (args.ntaps == 1) {
      dz = dy = dx = 0;
      return;
    }
    const int kd = tap / 9, kr = tap - kd * 9, kh = kr / 3;
    dz = (kd - 1) * args.dil;
    dy = kh - 1;
    dx = kr - kh * 3 - 1;
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
        int tap, m0, n0, kc0, kc1, dz, dy, dx;
        item_of(item, tap, m0, n0, kc0, kc1);
        tap_off(tap, dz, dy, dx);
        for (int kc = kc0; kc < kc1; ++kc) {
          int d, h0, w0;
          chunk_of(kc, d, h0, w0);
          if (d + dz < 0 || d + dz >= args.D) continue;  // the shifted plane is zero padding: the chunk contributes nothing
          mbar_wait(bar_empty + 8 * s, ph ^ 1u);
          mbar_arrive_expect_tx(bar_full + 8 * s, Cfg::STAGE);
          const int ad = args.shift_a ? dz : 0, ah = args.shift_a ? dy : 0, aw = args.shift_a ? dx : 0;
          const int bd = args.shift_a ? 0 : dz, bh = args.shift_a ? 0 : dy, bw = args.shift_a ? 0 : dx;
#pragma unroll
          for (int b = 0; b < WM_BM / 64; ++b)
            tma_load_4d(sA + s * Cfg::A_BYTES + b * WM_BLOCK, &tmA, bar_full + 8 * s, m0 + 64 * b, w0 + aw, h0 + ah, d + ad);
#pragma unroll
          for (int b = 0; b < BN / 64; ++b)
            tma_load_4d(sB + s * Cfg::B_BYTES + b * WM_BLOCK, &tmB, bar_full + 8 * s, n0 + 64 * b, w0 + bw, h0 + bh, d + bd);
          if (++s == STAGES) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // both operands MN-major (bits 15 / 16 of the instruction descriptor)
    constexpr uint32_t idesc = umma_idesc_bf16_f32(WM_BM, BN) | (1u << 15) | (1u << 16);
    int s = 0, acc = 0;
    uint32_t ph = 0, acc_ph = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
      int tap, m0, n0, kc0, kc1, dz, dy, dx;
      item_of(item, tap, m0, n0, kc0, kc1);
      tap_off(tap, dz, dy, dx);
      mbar_wait(bar_tempty + 8 * acc, acc_ph ^ 1u);
      tcgen05_fence_after();
      const uint32_t d_tmem = tmem_base + acc * Cfg::ACC;
      uint32_t accumulate = 0;
      for (int kc = kc0; kc < kc1; ++kc) {
        const int d = kc / per_plane;
        if (d + dz < 0 || d + dz >= args.D) continue;
        mbar_wait(bar_full + 8 * s, ph);
        tcgen05_fence_after();
        if (elect_one_sync()) {
          const uint64_t ad = umma_smem_desc_mnmajor_sw128(sA + s * Cfg::A_BYTES, WM_BLOCK);
          const uint64_t bd = umma_smem_desc_mnmajor_sw128(sB + s * Cfg::B_BYTES, WM_BLOCK);
#pragma unroll
          for (int k = 0; k < WM_KC / 16; ++k)  // 16 voxels per step: 16 rows of 128 B = +128 in 16-byte units
            umma_bf16(d_tmem, ad + 128 * k, bd + 128 * k, idesc, accumulate | (k > 0));
          umma_commit(bar_empty + 8 * s);
        }
        __syncwarp();
        accumulate = 1;
        if (++s == STAGES) { s = 0; ph ^= 1u; }
      }
      // an item whose every chunk was skipped never touched its accumulator: the epilogue must not add it
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
      int tap, m0, n0, kc0, kc1, dz, dy, dx;
      item_of(item, tap, m0, n0, kc0, kc1);
      tap_off(tap, dz, dy, dx);
      // did any chunk of this item run? (same test as the producer / issuer: planes d with d + dz inside the volume)
      bool any = false;
      if (kc1 > kc0) {
        const int d_lo = kc0 / per_plane, d_hi = (kc1 - 1) / per_plane;
        const int lo = max(d_lo, -dz), hi = min(d_hi, args.D - 1 - dz);
        any = lo <= hi;
      }
      mbar_wait(bar_tfull + 8 * acc, acc_ph);
      tcgen05_fence_after();
      const uint32_t t_acc = tmem_base + acc * Cfg::ACC + (static_cast<uint32_t>(q * 32) << 16);
      const int row = m0 + r;
      const bool live = any && row < args.M;
      float* orow = args.out + ((size_t)tap * args.M + row) * args.N + n0;
      if constexpr (DET) orow += (size_t)((item % per_tap) % args.ksplit) * args.ntaps * args.M * args.N;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32(t_acc + c0, v);
        tmem_ld_wait();
        if constexpr (DET) {
          if (row < args.M) {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (n0 + c0 + i < args.N) orow[c0 + i] = any ? __uint_as_float(v[i]) : 0.f;
          }
        } else if (live) {
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
__global__ void __launch_bounds__(WM_THREADS, 1)
wgrad_mn_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const WmArgs args) {
  wgrad_mn_body<BN, false>(tmA, tmB, args);
}

template <int BN>
__global__ void __launch_bounds__(WM_THREADS, 1)
wgrad_mn_det_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const WmArgs args) {
  wgrad_mn_body<BN, true>(tmA, tmB, args);
}

template <int BN, bool DET>
static int launch_wgrad_mn(const CUtensorMap& tmA, const CUtensorMap& tmB, const WmArgs& a, cudaStream_t st) {
  using Cfg = WmCfg<BN>;
  auto kern = DET ? wgrad_mn_det_kernel<BN> : wgrad_mn_kernel<BN>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM);
    if (e != cudaSuccess) {
      set_error("wgrad_mn: cudaFuncSetAttribute(smem=%d): %s", Cfg::SMEM, cudaGetErrorString(e));
      return CVIT_ERR_CUDA;
    }
    configured = true;
  }
  const int m_tiles = (a.M + WM_BM - 1) / WM_BM, n_tiles = (a.N + BN - 1) / BN;
  const int items = a.ntaps * m_tiles * n_tiles * a.ksplit;
  int grid = num_sms();
  if (grid > items) grid = items;
  kern<<<grid, WM_THREADS, Cfg::SMEM, st>>>(tmA, tmB, a);
  return check_launch(DET ? "wgrad_mn_det_kernel" : "wgrad_mn_kernel");
}

}  // namespace cvit

using namespace cvit;

// The K split of a launch: enough K ranges for ~4 items per SM, but never K ranges shorter than 32 chunks (2048 reduction steps)
static int64_t wgrad_mn_ksplit(int64_t D, int64_t H, int64_t W, int64_t Ca, int64_t Cb, int64_t ntaps, int* BW_out, int* bn_out) {
  int BW = 8;
  while (BW < W && BW < 64) BW <<= 1;
  const int BH = 64 / BW;
  const int bn = Cb > 192 ? 256 : Cb > 128 ? 192 : Cb > 64 ? 128 : 64;
  const int64_t k_chunks = D * ((H + BH - 1) / BH) * ((W + BW - 1) / BW);
  const int64_t tiles = ntaps * ((Ca + WM_BM - 1) / WM_BM) * ((Cb + bn - 1) / bn);
  int64_t ksplit = (4 * (int64_t)num_sms() + tiles - 1) / tiles;
  const int64_t max_split = k_chunks / 32 > 0 ? k_chunks / 32 : 1;
  if (ksplit > max_split) ksplit = max_split;
  if (ksplit < 1) ksplit = 1;
  if (BW_out) *BW_out = BW;
  if (bn_out) *bn_out = bn;
  return ksplit;
}

// See include/cryovit_b200.h.
extern "C" int cvit_wgrad_mn_ndhwc(const void* a, const void* b, float* out, int64_t D, int64_t H, int64_t W, int64_t Ca, int64_t Cb,
                                   int64_t dil, int64_t ntaps, int shift_a, void* stream) {
  if (!a || !b || !out || D <= 0 || H <= 0 || W <= 0 || Ca <= 0 || Cb <= 0 || dil <= 0 || (ntaps != 1 && ntaps != 27) ||
      (Ca % 8) != 0 || (Cb % 8) != 0 || Ca < 64 || Cb < 64) {
    set_error("wgrad_mn: bad arguments (D=%lld H=%lld W=%lld Ca=%lld Cb=%lld dil=%lld taps=%lld): channels >= 64, multiples of 8",
              (long long)D, (long long)H, (long long)W, (long long)Ca, (long long)Cb, (long long)dil, (long long)ntaps);
    return CVIT_ERR_INVALID;
  }
  if (((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15u) != 0) {
    set_error("wgrad_mn: operands must be 16-byte aligned");
    return CVIT_ERR_INVALID;
  }
  WmArgs args;
  args.out = out;
  args.M = (int)Ca;
  args.N = (int)Cb;
  args.D = (int)D;
  args.H = (int)H;
  args.W = (int)W;
  args.dil = (int)dil;
  args.ntaps = (int)ntaps;
  args.shift_a = shift_a ? 1 : 0;
  int BW = 8;
  while (BW < W && BW < 64) BW <<= 1;
  args.BW = BW;
  args.BH = 64 / BW;
  const int bn = Cb > 192 ? 256 : Cb > 128 ? 192 : Cb > 64 ? 128 : 64;
  CUtensorMap tmA, tmB;
  {
    uint64_t dims[4] = {(uint64_t)Ca, (uint64_t)W, (uint64_t)H, (uint64_t)D};
    uint64_t strides[4] = {0, (uint64_t)Ca * 2, (uint64_t)W * Ca * 2, (uint64_t)H * W * Ca * 2};
    uint32_t box[4] = {64, (uint32_t)args.BW, (uint32_t)args.BH, 1};
    int rc = encode_tmap(&tmA, TmapDtype::BF16, 4, a, dims, strides, box, 128);
    if (rc) return rc;
  }
  {
    uint64_t dims[4] = {(uint64_t)Cb, (uint64_t)W, (uint64_t)H, (uint64_t)D};
    uint64_t strides[4] = {0, (uint64_t)Cb * 2, (uint64_t)W * Cb * 2, (uint64_t)H * W * Cb * 2};
    uint32_t box[4] = {64, (uint32_t)args.BW, (uint32_t)args.BH, 1};
    int rc = encode_tmap(&tmB, TmapDtype::BF16, 4, b, dims, strides, box, 128);
    if (rc) return rc;
  }
  const int64_t k_chunks = D * ((H + args.BH - 1) / args.BH) * ((W + args.BW - 1) / args.BW);
  const int64_t tiles = ntaps * ((Ca + WM_BM - 1) / WM_BM) * ((Cb + bn - 1) / bn);
  // enough K ranges for ~4 items per SM, but never K ranges shorter than 32 chunks (2048 reduction steps)
  int64_t ksplit = (4 * (int64_t)num_sms() + tiles - 1) / tiles;
  const int64_t max_split = k_chunks / 32 > 0 ? k_chunks / 32 : 1;
  if (ksplit > max_split) ksplit = max_split;
  if (ksplit < 1) ksplit = 1;
  args.ksplit = (int)ksplit;
  cudaStream_t st = (cudaStream_t)stream;
  switch (bn) {
    case 256: return launch_wgrad_mn<256, false>(tmA, tmB, args, st);
    case 192: return launch_wgrad_mn<192, false>(tmA, tmB, args, st);
    case 128: return launch_wgrad_mn<128, false>(tmA, tmB, args, st);
    default: return launch_wgrad_mn<64, false>(tmA, tmB, args, st);
  }
}

// Deterministic mode: the same GEMM with every item's tile stored into its K slice of scratch ([ksplit][ntaps][Ca][Cb] fp32,
// cvit_wgrad_mn_ndhwc_det_partials floats), then out += the slices added in K order.
extern "C" int64_t cvit_wgrad_mn_ndhwc_det_partials(int64_t D, int64_t H, int64_t W, int64_t Ca, int64_t Cb, int64_t ntaps) {
  if (D <= 0 || H <= 0 || W <= 0 || Ca <= 0 || Cb <= 0 || ntaps <= 0) return 0;
  return wgrad_mn_ksplit(D, H, W, Ca, Cb, ntaps, nullptr, nullptr) * ntaps * Ca * Cb;
}

extern "C" int cvit_wgrad_mn_ndhwc_det(const void* a, const void* b, float* out, int64_t D, int64_t H, int64_t W, int64_t Ca, int64_t Cb,
                                       int64_t dil, int64_t ntaps, int shift_a, float* scratch, int64_t scratch_elems, void* stream) {
  if (!a || !b || !out || D <= 0 || H <= 0 || W <= 0 || Ca <= 0 || Cb <= 0 || dil <= 0 || (ntaps != 1 && ntaps != 27) ||
      (Ca % 8) != 0 || (Cb % 8) != 0 || Ca < 64 || Cb < 64) {
    set_error("wgrad_mn_det: bad arguments (D=%lld H=%lld W=%lld Ca=%lld Cb=%lld dil=%lld taps=%lld): channels >= 64, multiples of 8",
              (long long)D, (long long)H, (long long)W, (long long)Ca, (long long)Cb, (long long)dil, (long long)ntaps);
    return CVIT_ERR_INVALID;
  }
  if (int rc = det_check_scratch(scratch, scratch_elems, cvit_wgrad_mn_ndhwc_det_partials(D, H, W, Ca, Cb, ntaps), "wgrad_mn_det")) return rc;
  if (((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15u) != 0) {
    set_error("wgrad_mn_det: operands must be 16-byte aligned");
    return CVIT_ERR_INVALID;
  }
  int BW, bn;
  const int64_t ksplit = wgrad_mn_ksplit(D, H, W, Ca, Cb, ntaps, &BW, &bn);
  WmArgs args;
  args.out = scratch;
  args.M = (int)Ca;
  args.N = (int)Cb;
  args.D = (int)D;
  args.H = (int)H;
  args.W = (int)W;
  args.dil = (int)dil;
  args.ntaps = (int)ntaps;
  args.shift_a = shift_a ? 1 : 0;
  args.BW = BW;
  args.BH = 64 / BW;
  args.ksplit = (int)ksplit;
  CUtensorMap tmA, tmB;
  {
    uint64_t dims[4] = {(uint64_t)Ca, (uint64_t)W, (uint64_t)H, (uint64_t)D};
    uint64_t strides[4] = {0, (uint64_t)Ca * 2, (uint64_t)W * Ca * 2, (uint64_t)H * W * Ca * 2};
    uint32_t box[4] = {64, (uint32_t)args.BW, (uint32_t)args.BH, 1};
    int rc = encode_tmap(&tmA, TmapDtype::BF16, 4, a, dims, strides, box, 128);
    if (rc) return rc;
  }
  {
    uint64_t dims[4] = {(uint64_t)Cb, (uint64_t)W, (uint64_t)H, (uint64_t)D};
    uint64_t strides[4] = {0, (uint64_t)Cb * 2, (uint64_t)W * Cb * 2, (uint64_t)H * W * Cb * 2};
    uint32_t box[4] = {64, (uint32_t)args.BW, (uint32_t)args.BH, 1};
    int rc = encode_tmap(&tmB, TmapDtype::BF16, 4, b, dims, strides, box, 128);
    if (rc) return rc;
  }
  cudaStream_t st = (cudaStream_t)stream;
  int rc;
  switch (bn) {
    case 256: rc = launch_wgrad_mn<256, true>(tmA, tmB, args, st); break;
    case 192: rc = launch_wgrad_mn<192, true>(tmA, tmB, args, st); break;
    case 128: rc = launch_wgrad_mn<128, true>(tmA, tmB, args, st); break;
    default: rc = launch_wgrad_mn<64, true>(tmA, tmB, args, st); break;
  }
  if (rc) return rc;
  const int64_t n = ntaps * Ca * Cb;
  return det_finalize(scratch, ksplit, n, n, out, true, st);
}
