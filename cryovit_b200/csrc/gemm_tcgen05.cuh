// Persistent, warp-specialised tcgen05 GEMM for sm_100a with fused epilogues.
//
//   D[M,N] = A[M,K] (bf16, K-major) x B[N,K]^T (bf16, K-major, i.e. torch Linear weight layout)
//   (GemmArgs::fmt: both operands IEEE fp16 instead, and/or the 16-bit output stored as fp16)
//   OPK = OPK_TF32: A and B are fp32 holding TF32 values, tcgen05.mma kind::tf32 (half the kind::f16 rate); the
//   bias(+GELU / SwiGLU) epilogues then store TF32-rounded fp32 for the next TF32 GEMM (EPI_BIAS stays 16-bit)
//
// One CTA per SM, 320 threads:
//   warp 0      TMA producer  (one lane): cp.async.bulk.tensor -> 128B/64B/32B-swizzled smem ring
//   warp 1      MMA issuer    (one lane): tcgen05.mma 128 x BN x 16, fp32 accumulators in TMEM,
//                                          two accumulator buffers so tile i+1 overlaps epilogue i
//   warps 2..9  epilogue (two warps per TMEM lane quarter, alternating 32-column chunks, so every scheduler
//               has two epilogue warps to hide latency): tcgen05.ld (32 lanes x 32 cols) -> warp-private
//               swizzled smem transpose -> fused math -> row-contiguous vector stores
//
// A-operand addressing modes:
//   AMODE_ROWS  plain 2-D [M,K] matrix (ViT linears, 1x1x1 conv, transposed conv)
//   AMODE_CONV3 implicit-GEMM 3x3x3 dilated "same" convolution over a channels-last [D,H,W,C] volume:
//               the K loop walks (tap, channel-chunk); each A tile is one 4-D TMA box shifted by the
//               tap offset, and TMA's out-of-bounds zero fill IS the zero padding (no im2col, no halo
//               staging code). Taps whose depth offset falls outside [0,D) are skipped outright.
//   AMODE_ROWS_MN  the same [M,K] matrix stored TRANSPOSED in memory ([K,M], M contiguous): the head's projection reads
//               the on-disk feature layout (C, D*h*w) directly as an MN-major A operand (two 64-row x 64-channel
//               128B-swizzled boxes per stage), so no channels-last copy of the features is ever written.
//
// Epilogues (what the reference computes around each GEMM, SURVEY.md 2.2 K5-K17):
//   EPI_BIAS            out_bf16 = acc + bias                               (qkv)
//   EPI_BIAS_GELU       out_bf16 = gelu_erf(acc + bias)                     (ViT-S/B/L fc1, head convs)
//   EPI_BIAS_SWIGLU     out_bf16 = silu(acc1 + b1) * (acc2 + b2)            (ViT-g w12; weights row-interleaved
//                                                                            per BN tile: [BN/2 of x1 | BN/2 of x2])
//   EPI_SCALE_RESIDUAL  x_f32   += gamma * (acc + bias)                     (attn.proj + ls1, w3/fc2 + ls2)
//   EPI_PATCH_EMBED     x_f32[b, off + p] = acc + table[p]                  (patch embed + bias + pos-embed)
//   EPI_CONVT_GELU      pixel-shuffle store of ConvTranspose3d(1,2,2) + bias + GELU
#pragma once
#include "ptx.cuh"

namespace cvit {

#ifndef CONVT_DIRECT
#define CONVT_DIRECT 1  // -DCONVT_DIRECT=0: the transposing epilogue for the plain transposed convolution too (A/B)
#endif
enum { EPI_BIAS = 0, EPI_BIAS_GELU = 1, EPI_BIAS_SWIGLU = 2, EPI_SCALE_RESIDUAL = 3, EPI_PATCH_EMBED = 4, EPI_CONVT_GELU = 5 };
enum { AMODE_ROWS = 0, AMODE_CONV3 = 1, AMODE_ROWS_MN = 2 };

struct GemmArgs {
  int M, N, K;        // rows, output columns, reduction length (per tap for AMODE_CONV3)
  void* out;          // bf16 or fp32, see epilogues
  int ldo;            // leading dimension of out, in elements
  const float* bias;  // [N] (interleaved like the weights for SWIGLU); may be null for PATCH_EMBED
  const float* gamma; // [N] LayerScale (SCALE_RESIDUAL)
  const float* table; // [pe_np, N] fp32 pos-embed(+bias) table (PATCH_EMBED)
  int pe_np, pe_tokens, pe_offset;  // patches per slice, tokens per slice, first patch token index
  int D, H, W, dil;   // AMODE_CONV3 geometry (M == D*H*W); dilation applies to depth only
  int BW, BH;         // AMODE_CONV3 tile footprint, BW*BH == 128
  int c3;             // EPI_CONVT_GELU: output channels per sub-pixel (N == 4*c3); uses H, W too
  int n_valid;        // columns >= n_valid are computed (zero-padded weights) but never stored
  int act;            // EPI_BIAS_GELU / EPI_CONVT_GELU: ACT_* of ptx.cuh (1 = GELU: inference; 0 / 2 / 3: training); EPI_BIAS reads
                      // only ACT_GELU_GRAD
  void* aux;          // ACT_DUAL: bf16 activation output; ACT_GELU_GRAD: bf16 saved pre-activation (indexed like out)
  int fmt;            // GEMM_FMT_* bits: 16-bit type of the operands / of the stored output (0 = bf16 everywhere)
  // GroupNorm fused into its neighbours (head inference, models/cryovit.py:56 SynthesisBlock.layers[0]):
  //  * PRODUCER side (EPI_BIAS_GELU on plain rows, EPI_CONVT_GELU): gn_partials != null -> every epilogue warp also
  //    writes, per 32-row block and per group of gn_cpg consecutive output columns, the (sum, sum of squares) of the
  //    values it stores: fp32 [ceil(M/32)][N / gn_cpg][2], one plain store per entry (each entry has exactly one
  //    owner, so the later fixed-order reduction is deterministic). N == n_valid is required.
  //  * CONSUMER side (EPI_BIAS_GELU with AMODE_CONV3): bias_table != null -> the bias of an output voxel is row
  //    ((dm*4 + hm)*4 + wm) of fp32 [64][N], where the 2-bit masks say which of the taps -1 / +1 along depth (dilated),
  //    height and width fall inside the volume. With the GroupNorm affine folded into the weights (w' = w * a_c) the
  //    shift b_c contributes  sum over the IN-BOUNDS taps of sum_c w[tap][c] * b_c, which depends on exactly that.
  float* gn_partials;
  int gn_cpg;
  int gn_direct;      // EPI_CONVT_GELU with 32 channels in groups of 4: every epilogue thread keeps the 8 group sums of everything it
                      // stores in registers and writes ONE partials row [8][2] at the end of the kernel (row = block * 256 + thread)
  const float* bias_table;
};
// A and B hold IEEE fp16 instead of bf16 (same type on both sides: tcgen05 kind::f16 rule); EPI_BIAS / _GELU / _SWIGLU
// store fp16 instead of bf16. fp16 keeps three more mantissa bits than bf16 for operands whose range is bounded
// (LayerNorm output, q/k/v, attention output and the weights they meet).
// GEMM_FMT_OPERANDS_TF32: A and B are fp32 holding TF32 values (the OPK_TF32 kernels); GEMM_FMT_OUT_F32: EPI_BIAS_GELU /
// EPI_BIAS_SWIGLU of those kernels store TF32-rounded fp32. The host picks kernels from these bits; the kernel body reads
// only GEMM_FMT_OUT_F16 at run time.
enum { GEMM_FMT_OPERANDS_F16 = 1, GEMM_FMT_OUT_F16 = 2, GEMM_FMT_OPERANDS_TF32 = 4, GEMM_FMT_OUT_F32 = 8 };
// Operand kind of a kernel instantiation: kind::f16 (bf16 or fp16 by GemmArgs::fmt) or kind::tf32 (fp32 containers).
enum { OPK_F16 = 0, OPK_TF32 = 1 };

constexpr int GEMM_BM = 128;
constexpr int GEMM_THREADS = 320;
constexpr int GEMM_EPI_WARPS = 8;

// SUB > 1 ("tall" tiles, plain-rows GEMMs with a single short K chunk: the transposed convolutions of the head, K = 16
// .. 64): one pipeline stage carries SUB consecutive 128-row blocks of A, the issuer runs one MMA chain per block into
// its own TMEM column range, and the epilogue warps share the SUB x (BN / 32) column chunks. With K this short a
// 128-row tile is a few hundred cycles of tensor work, so the per-tile barrier round trips (and, for BN = 32, half of
// the epilogue warps having no chunk at all) dominated; SUB amortises them.
template <int BN, int KSPAN, bool PAIR = false, int SUB = 1>
struct GemmCfg {
  static constexpr int A_BLOCK_BYTES = GEMM_BM * KSPAN;
  static constexpr int A_BYTES = SUB * A_BLOCK_BYTES;
  static constexpr int B_BYTES = (PAIR ? BN / 2 : BN) * KSPAN;  // a CTA pair splits the B tile half/half
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES_RAW = (192 * 1024) / STAGE_BYTES;
  static constexpr int STAGES = STAGES_RAW > 8 ? 8 : STAGES_RAW;
  static constexpr int STG_BYTES_PER_WARP = 4096;  // one 32x32 fp32 transpose buffer per epilogue warp
  static constexpr int ACC_STRIDE = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;
  static constexpr int TMEM_COLS = 2 * SUB * ACC_STRIDE;
  static_assert(TMEM_COLS <= 512, "SUB x accumulator width exceeds TMEM");
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + GEMM_EPI_WARPS * STG_BYTES_PER_WARP + 256 /*barriers*/ + 1024 /*align slack*/;
  static_assert(SMEM_BYTES <= 232448, "exceeds 227 KB of shared memory per CTA");
  static_assert(BN % 32 == 0 && BN >= 32 && BN <= 256, "BN must be a multiple of 32 in [32,256]");
  // every stage base must stay 1024-aligned for the swizzle pattern to line up with the descriptor
  static_assert(A_BYTES % 1024 == 0 && B_BYTES % 1024 == 0, "operand tiles must be 1024B multiples");
};

struct TileCoord {
  int m0, n0;        // first output row / column of this tile
  int d, h0, w0;     // AMODE_CONV3: depth plane and spatial origin
};

// MB_MUL / mb_add: a CTA pair in AMODE_CONV3 walks PAIRS of row tiles (row tile = 2 * pair tile + cluster rank)
template <int BN, int AMODE>
__device__ __forceinline__ TileCoord tile_coord(int tile, int num_n, const GemmArgs& a, int mb_mul = 1, int mb_add = 0) {
  TileCoord t;
  int mb = tile / num_n;
  t.n0 = (tile - mb * num_n) * BN;
  mb = mb * mb_mul + mb_add;
  t.m0 = mb * GEMM_BM;
  t.d = t.h0 = t.w0 = 0;
  if (AMODE == AMODE_CONV3) {
    int tiles_w = (a.W + a.BW - 1) / a.BW, tiles_h = (a.H + a.BH - 1) / a.BH;
    int per_plane = tiles_w * tiles_h;
    t.d = mb / per_plane;
    int r = mb - t.d * per_plane;
    int th = r / tiles_w;
    t.h0 = th * a.BH;
    t.w0 = (r - th * tiles_w) * a.BW;
  }
  return t;
}

// Row r (0..127) of a tile -> linear output row (voxel index for conv), or -1 when out of range.
template <int AMODE>
__device__ __forceinline__ int tile_row_to_global(const TileCoord& t, int r, const GemmArgs& a) {
  if (AMODE == AMODE_CONV3) {
    int hl = r / a.BW, wl = r - hl * a.BW;
    int h = t.h0 + hl, w = t.w0 + wl;
    // partial tiles at the plane border (or the odd last tile of a CTA pair, d == D): TMA zero-filled the loads, the
    // rows are simply not stored
    if (h >= a.H || w >= a.W || t.d >= a.D) return -1;
    return (t.d * a.H + h) * a.W + w;
  }
  int g = t.m0 + r;
  return g < a.M ? g : -1;
}

// PAIR = true (AMODE_ROWS only): the kernel is launched as clusters of two CTAs (the two SMs of a TPC). A pair owns a
// 256 x BN output tile: CTA rank r loads A rows [m0 + 128 r, +128) and B rows [n0 + BN/2 r, +BN/2), the leader (rank 0)
// issues tcgen05.mma.cta_group::2 (M = 256) that reads both CTAs' shared memory and writes each CTA's 128 accumulator
// rows into its own TMEM, and each CTA runs its own epilogue. Per SM and per FLOP this halves the B-operand shared
// memory traffic (TMA writes and MMA reads) against the single-CTA kernel. Barriers: the "full" barriers that count
// TMA bytes live in the leader (both producers signal them), "empty"/"accumulator full" are multicast commits to both
// CTAs, "accumulator empty" collects the epilogue warps of both CTAs in the leader.
template <int BN, int EPI, int AMODE, int KSPAN, bool PAIR = false, int SUB = 1, int OPK = OPK_F16>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const GemmArgs args) {
  // PAIR with AMODE_CONV3: the two CTAs take two consecutive row tiles of the SAME depth plane (the host only selects
  // the pair kernel when the number of tiles per plane is even), so both skip the same out-of-range depth taps and the
  // leader's MMA schedule matches both producers'.
  static_assert(SUB == 1 || (AMODE == AMODE_ROWS && !PAIR), "tall tiles are implemented for the single-CTA plain-rows GEMM only");
  static_assert(AMODE != AMODE_ROWS_MN || KSPAN == 128, "the MN-major A operand is staged in 128-byte swizzled rows");
  static_assert(OPK == OPK_F16 || (AMODE == AMODE_ROWS && SUB == 1 && (EPI <= EPI_PATCH_EMBED)),
                "TF32 operands are implemented for the plain-rows ViT GEMMs only");
  using Cfg = GemmCfg<BN, KSPAN, PAIR, SUB>;
  constexpr bool TF32 = OPK == OPK_TF32;
  constexpr int TILE_M = (PAIR ? 2 : SUB) * GEMM_BM;  // output rows per tile (per CTA pair with PAIR)
  constexpr int KC = KSPAN / (TF32 ? 4 : 2);  // elements of K per stage (16-bit, or fp32 for TF32)
  constexpr int MMAS_PER_STAGE = KC / (TF32 ? 8 : 16);  // 32 bytes of K per MMA either way
  constexpr int STAGES = Cfg::STAGES;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sA = smem_base;
  const uint32_t sB = smem_base + STAGES * Cfg::A_BYTES;
  const uint32_t sStg = smem_base + STAGES * Cfg::STAGE_BYTES;
  const uint32_t sBar = sStg + GEMM_EPI_WARPS * Cfg::STG_BYTES_PER_WARP;
  const uint32_t bar_full = sBar;                    // STAGES x 8B
  const uint32_t bar_empty = sBar + 8 * STAGES;      // STAGES x 8B
  const uint32_t bar_tfull = sBar + 16 * STAGES;     // 2 x 8B
  const uint32_t bar_tempty = bar_tfull + 16;        // 2 x 8B
  const uint32_t tmem_slot = bar_tempty + 16;        // 4B
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));  // generic alias of smem_base

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const int num_n = args.N / BN;
  const int num_m = AMODE == AMODE_CONV3
                        ? (args.D * ((args.H + args.BH - 1) / args.BH) * ((args.W + args.BW - 1) / args.BW) + (PAIR ? 1 : 0)) / (PAIR ? 2 : 1)
                        : (args.M + TILE_M - 1) / TILE_M;
  const int num_tiles = num_m * num_n;
  const int k_chunks = (args.K + KC - 1) / KC;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const int tile_first = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int tile_step = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  auto coord = [&](int tile) {
    if (PAIR && AMODE == AMODE_CONV3) return tile_coord<BN, AMODE>(tile, num_n, args, 2, (int)rank);
    TileCoord t = tile_coord<BN, AMODE>(tile, num_n, args);
    if (PAIR) t.m0 = 2 * t.m0 + (int)rank * GEMM_BM;
    if (SUB > 1) t.m0 *= SUB;
    return t;
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
      mbar_init(bar_tempty + 8 * i, (PAIR ? 2 : 1) * GEMM_EPI_WARPS);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    if (PAIR) tmem_alloc_pair<Cfg::TMEM_COLS>(tmem_slot);
    else tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  }
  tcgen05_fence_before();
  if (PAIR) cluster_sync_all();  // the peer's barriers must be initialised before anything is signalled on them
  else __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int tile = tile_first; tile < num_tiles; tile += tile_step) {
        const TileCoord t = coord(tile);
        const int taps = AMODE == AMODE_CONV3 ? 27 : 1;
        for (int tap = 0; tap < taps; ++tap) {
          int dz = 0, dy = 0, dx = 0;
          if (AMODE == AMODE_CONV3) {
            int kd = tap / 9, kr = tap - kd * 9, kh = kr / 3, kw = kr - kh * 3;
            dz = t.d + (kd - 1) * args.dil;
            dy = t.h0 + kh - 1;
            dx = t.w0 + kw - 1;
            if (dz < 0 || dz >= args.D) continue;  // whole tap is zero padding
          }
          for (int kc = 0; kc < k_chunks; ++kc) {
            mbar_wait(bar_empty + 8 * s, ph ^ 1u);
            if (PAIR) {
              // both producers report their bytes to the LEADER's full barrier, which expects the pair's total
              if (rank == 0) mbar_arrive_expect_tx(bar_full + 8 * s, 2 * Cfg::STAGE_BYTES);
              const uint32_t lead_full = mapa_cluster(bar_full + 8 * s, 0);
              if (AMODE == AMODE_CONV3) {
                tma_load_4d_pair(sA + s * Cfg::A_BYTES, &tmA, lead_full, kc * KC, dx, dy, dz);
                tma_load_2d_pair(sB + s * Cfg::B_BYTES, &tmB, lead_full, kc * KC, tap * args.N + t.n0 + (int)rank * (BN / 2));
                if (++s == STAGES) { s = 0; ph ^= 1u; }
                continue;
              }
              if (AMODE == AMODE_ROWS_MN) {  // two boxes of 64 rows (inner, contiguous) x KC channels
                tma_load_2d_pair(sA + s * Cfg::A_BYTES, &tmA, lead_full, t.m0, kc * KC);
                tma_load_2d_pair(sA + s * Cfg::A_BYTES + Cfg::A_BYTES / 2, &tmA, lead_full, t.m0 + 64, kc * KC);
              } else
              tma_load_2d_pair(sA + s * Cfg::A_BYTES, &tmA, lead_full, kc * KC, t.m0);
              tma_load_2d_pair(sB + s * Cfg::B_BYTES, &tmB, lead_full, kc * KC, t.n0 + (int)rank * (BN / 2));
              if (++s == STAGES) { s = 0; ph ^= 1u; }
              continue;
            }
            mbar_arrive_expect_tx(bar_full + 8 * s, Cfg::STAGE_BYTES);
            if (AMODE == AMODE_CONV3) {
              tma_load_4d(sA + s * Cfg::A_BYTES, &tmA, bar_full + 8 * s, kc * KC, dx, dy, dz);
              tma_load_2d(sB + s * Cfg::B_BYTES, &tmB, bar_full + 8 * s, kc * KC, tap * args.N + t.n0);
            } else if (AMODE == AMODE_ROWS_MN) {
              tma_load_2d(sA + s * Cfg::A_BYTES, &tmA, bar_full + 8 * s, t.m0, kc * KC);
              tma_load_2d(sA + s * Cfg::A_BYTES + Cfg::A_BYTES / 2, &tmA, bar_full + 8 * s, t.m0 + 64, kc * KC);
              tma_load_2d(sB + s * Cfg::B_BYTES, &tmB, bar_full + 8 * s, kc * KC, t.n0);
            } else {
#pragma unroll
              for (int sub = 0; sub < SUB; ++sub)  // blocks past the last row are zero-filled by TMA and never stored
                tma_load_2d(sA + s * Cfg::A_BYTES + sub * Cfg::A_BLOCK_BYTES, &tmA, bar_full + 8 * s, kc * KC, t.m0 + sub * GEMM_BM);
              tma_load_2d(sB + s * Cfg::B_BYTES, &tmB, bar_full + 8 * s, kc * KC, t.n0);
            }
            if (++s == STAGES) { s = 0; ph ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ------------------------------------------------------------------ MMA issuer (the pair's leader only)
    // The whole warp walks the tile / k-chunk schedule so control flow stays warp-uniform and the descriptors live
    // in uniform registers; one elected lane issues the MMAs and commits. (Issuing from a divergent `lane == 0`
    // region cost ~90 cycles per tcgen05.mma: every operand went through R2UR and a per-lane ELECT loop.)
    {
      const uint32_t idesc = TF32 ? umma_idesc_tf32_f32(PAIR ? 2 * GEMM_BM : GEMM_BM, BN)
                                  : umma_idesc_f16_f32(PAIR ? 2 * GEMM_BM : GEMM_BM, BN) |
                                        ((args.fmt & GEMM_FMT_OPERANDS_F16) ? 0u : UMMA_IDESC_BF16_BITS) |
                                        (AMODE == AMODE_ROWS_MN ? (1u << 15) : 0u);  // bit 15: A is MN-major
      int s = 0;
      uint32_t ph = 0;
      int acc = 0;
      uint32_t acc_ph = 0;
      for (int tile = tile_first; tile < num_tiles; tile += tile_step) {
        const TileCoord t = coord(tile);
        mbar_wait(bar_tempty + 8 * acc, acc_ph ^ 1u);
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + acc * SUB * Cfg::ACC_STRIDE;
        uint32_t accumulate = 0;
        const int taps = AMODE == AMODE_CONV3 ? 27 : 1;
        for (int tap = 0; tap < taps; ++tap) {
          if (AMODE == AMODE_CONV3) {
            int kd = tap / 9;
            int dz = t.d + (kd - 1) * args.dil;
            if (dz < 0 || dz >= args.D) continue;
          }
          for (int kc = 0; kc < k_chunks; ++kc) {
            mbar_wait(bar_full + 8 * s, ph);
            tcgen05_fence_after();
            if (elect_one_sync()) {
              const uint64_t bdesc = umma_smem_desc_kmajor<KSPAN>(sB + s * Cfg::B_BYTES);
#pragma unroll
              for (int sub = 0; sub < SUB; ++sub) {
                // K-major A: 16 elements of K = 32 bytes inside the swizzle span (+2 in 16-byte units). MN-major A: 16 K
                // rows of 128 bytes (+128); the two 64-row blocks of the tile are LBO = A_BYTES / 2 apart.
                const uint64_t adesc = AMODE == AMODE_ROWS_MN
                                           ? umma_smem_desc_mnmajor_sw128(sA + s * Cfg::A_BYTES, Cfg::A_BYTES / 2)
                                           : umma_smem_desc_kmajor<KSPAN>(sA + s * Cfg::A_BYTES + sub * Cfg::A_BLOCK_BYTES);
                constexpr int ASTEP = AMODE == AMODE_ROWS_MN ? 128 : 2;
#pragma unroll
                for (int k = 0; k < MMAS_PER_STAGE; ++k) {
                  // B: advance 16 bf16 (8 TF32) = 32 bytes along K inside the swizzle span: +2 in 16-byte units
                  if (TF32 && PAIR) umma_tf32_pair(d_tmem, adesc + ASTEP * k, bdesc + 2 * k, idesc, accumulate | (k > 0));
                  else if (TF32) umma_tf32(d_tmem, adesc + ASTEP * k, bdesc + 2 * k, idesc, accumulate | (k > 0));
                  else if (PAIR) umma_bf16_pair(d_tmem, adesc + ASTEP * k, bdesc + 2 * k, idesc, accumulate | (k > 0));
                  else umma_bf16(d_tmem + sub * Cfg::ACC_STRIDE, adesc + ASTEP * k, bdesc + 2 * k, idesc, accumulate | (k > 0));
                }
              }
              // smem slot reusable once these MMAs retire (in both CTAs of a pair)
              if (PAIR) umma_commit_pair(bar_empty + 8 * s);
              else umma_commit(bar_empty + 8 * s);
            }
            __syncwarp();
            accumulate = 1;
            if (++s == STAGES) { s = 0; ph ^= 1u; }
          }
        }
        if (elect_one_sync()) {  // accumulator complete
          if (PAIR) umma_commit_pair(bar_tfull + 8 * acc);
          else umma_commit(bar_tfull + 8 * acc);
        }
        __syncwarp();
        acc ^= 1;
        if (acc == 0) acc_ph ^= 1u;
      }
    }
  } else if (warp >= 2) {
    // ------------------------------------------------------------------ epilogue warps
    const int ew = warp - 2;   // 0..7
    const int q = warp & 3;    // TMEM lane quarter this warp may access (hardware rule: warp id % 4)
    const int half = ew >> 2;  // the two warps of a quarter take alternate 32-column chunks
    const uint32_t stg = sStg + ew * Cfg::STG_BYTES_PER_WARP;
    int acc = 0;
    uint32_t acc_ph = 0;
    constexpr int NCHUNK = (EPI == EPI_BIAS_SWIGLU ? BN / 2 : BN) / 32;
    const bool out_f16 = (args.fmt & GEMM_FMT_OUT_F16) != 0;
    const int jc = lane & 7;    // 16-byte column group handled by this lane on the way out
    const int rsub = lane >> 3; // row within each group of 4 rows
    // smem transpose addresses: thread == row on the way in, (4 rows x 8 column groups) per step on the way out
    const uint32_t st_addr = stg + lane * 128;
    const int st_sw = lane & 7;
    auto stage_in = [&](const uint32_t (&v)[32]) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(st_addr + ((j ^ st_sw) << 4)), "r"(v[4 * j]),
                     "r"(v[4 * j + 1]), "r"(v[4 * j + 2]), "r"(v[4 * j + 3])
                     : "memory");
      }
    };
    auto stage_out = [&](float4 (&x)[8]) {
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        const int r = it * 4 + rsub;
        const uint32_t addr = stg + r * 128 + ((jc ^ (r & 7)) << 4);
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(x[it].x), "=f"(x[it].y), "=f"(x[it].z), "=f"(x[it].w) : "r"(addr));
      }
    };
    // GroupNorm statistics of what this warp stores for one 32-column chunk: this lane's 4 columns x 8 rows, summed
    // over the rows of the lanes that share the columns (and over the lane pair that shares an 8-column group), one
    // (sum, sum of squares) store per group by its first lane. row0 = first of the warp's 32 rows (a multiple of 32).
    auto gn_stats = [&](const float4 (&v)[8], const int (&grow)[8], int row0, int ncol) {
      float sm = 0.f, sq = 0.f;
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        if (grow[it] >= 0) {
          sm += (v[it].x + v[it].y) + (v[it].z + v[it].w);
          sq += (v[it].x * v[it].x + v[it].y * v[it].y) + (v[it].z * v[it].z + v[it].w * v[it].w);
        }
      }
      sm += __shfl_xor_sync(0xffffffffu, sm, 8);
      sq += __shfl_xor_sync(0xffffffffu, sq, 8);
      sm += __shfl_xor_sync(0xffffffffu, sm, 16);
      sq += __shfl_xor_sync(0xffffffffu, sq, 16);
      if (args.gn_cpg == 8) {
        sm += __shfl_xor_sync(0xffffffffu, sm, 1);
        sq += __shfl_xor_sync(0xffffffffu, sq, 1);
      }
      if (rsub == 0 && (args.gn_cpg == 4 || (jc & 1) == 0)) {
        float2* dst = reinterpret_cast<float2*>(args.gn_partials) + (size_t)(row0 >> 5) * (args.N / args.gn_cpg) + ncol / args.gn_cpg;
        *dst = make_float2(sm, sq);
      }
    };
    float gsum[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, gsq[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // gn_direct
    for (int tile = tile_first; tile < num_tiles; tile += tile_step) {
      const TileCoord t = coord(tile);
      mbar_wait(bar_tfull + 8 * acc, acc_ph);
      tcgen05_fence_after();
      const uint32_t t_acc0 = tmem_base + acc * SUB * Cfg::ACC_STRIDE + (static_cast<uint32_t>(q * 32) << 16);
      // global row of this lane's first output row (rows mode: linear, 4 apart per step; conv mode: per row)
      int grow_it[8];
      if (SUB == 1) {
#pragma unroll
        for (int it = 0; it < 8; ++it) grow_it[it] = tile_row_to_global<AMODE>(t, q * 32 + it * 4 + rsub, args);
      }
#pragma unroll 1
      for (int idx = half; idx < SUB * NCHUNK; idx += 2) {
        const int sub = SUB == 1 ? 0 : idx / NCHUNK;
        const int ch = SUB == 1 ? idx : idx - sub * NCHUNK;
        const uint32_t t_acc = t_acc0 + sub * Cfg::ACC_STRIDE;
        if (SUB > 1) {
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            const int g = t.m0 + sub * GEMM_BM + q * 32 + it * 4 + rsub;
            grow_it[it] = g < args.M ? g : -1;
          }
        }
        const int c0 = ch * 32;
        if (EPI == EPI_CONVT_GELU && CONVT_DIRECT && args.c3 <= 32 && (!args.gn_partials || args.gn_direct)) {
          // Transposed convolution to 8 / 16 / 32 channels: NO shared-memory transpose. The thread keeps its accumulator row
          // (one input voxel, 32 output columns = whole channel blocks of 1..4 sub-pixels) and stores them where the pixel
          // shuffle puts them, 32 bytes (one full sector) per store: columns 0..15 and 16..31 of a chunk are contiguous in
          // the output for every channel count (8: sub-pixels (i,0),(i,1); 16 / 32: one sub-pixel). ~9 instructions per
          // output value instead of 19-25 (ncu: the transposing epilogue ran at 46 % issue utilisation, tensor pipe 1-2 %).
          // GroupNorm statistics (gn_direct): 32 columns = the 8 groups of 4 channels of one sub-pixel, the same 8 groups in
          // every chunk: two FMAs per value into 16 registers that live for the whole kernel.
          uint32_t v[32];
          tmem_ld_32x32(t_acc + c0, v);
          tmem_ld_wait();
          const int g = t.m0 + (SUB == 1 ? 0 : sub * GEMM_BM) + q * 32 + lane;
          if (g < args.M && t.n0 + c0 < args.n_valid) {
            const int dh = g / args.W, w = g - dh * args.W, W2 = 2 * args.W;
            int ij = (t.n0 + c0) / args.c3, co = (t.n0 + c0) - ij * args.c3;
            __nv_bfloat16* o1 = static_cast<__nv_bfloat16*>(args.out);
            __nv_bfloat16* o2 = static_cast<__nv_bfloat16*>(args.act == ACT_DUAL ? args.aux : args.out);
#pragma unroll
            for (int b16 = 0; b16 < 2; ++b16) {
              float y[16];
#pragma unroll
              for (int c4 = 0; c4 < 4; ++c4) {
                const float4 bq = __ldg(reinterpret_cast<const float4*>(args.bias + t.n0 + c0 + 16 * b16 + 4 * c4));
                y[4 * c4] = __uint_as_float(v[16 * b16 + 4 * c4]) + bq.x;
                y[4 * c4 + 1] = __uint_as_float(v[16 * b16 + 4 * c4 + 1]) + bq.y;
                y[4 * c4 + 2] = __uint_as_float(v[16 * b16 + 4 * c4 + 2]) + bq.z;
                y[4 * c4 + 3] = __uint_as_float(v[16 * b16 + 4 * c4 + 3]) + bq.w;
              }
              const size_t off = ((size_t)(2 * dh + (ij >> 1)) * W2 + 2 * w + (ij & 1)) * args.c3 + co;
              if (args.act == ACT_DUAL) {
                uint32_t pz[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) pz[i] = pack_bf16x2(y[2 * i], y[2 * i + 1]);
                st_global_v8(o1 + off, pz);
              }
              if (args.act) {
#pragma unroll
                for (int i = 0; i < 8; ++i) gelu_erf2(y[2 * i], y[2 * i + 1]);
              }
              if (args.gn_direct) {
#pragma unroll
                for (int gi = 0; gi < 4; ++gi) {
                  const float a0 = y[4 * gi], a1 = y[4 * gi + 1], a2 = y[4 * gi + 2], a3 = y[4 * gi + 3];
                  gsum[4 * b16 + gi] += (a0 + a1) + (a2 + a3);
                  gsq[4 * b16 + gi] += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
                }
              }
              uint32_t pk[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) pk[i] = pack_bf16x2(y[2 * i], y[2 * i + 1]);
              st_global_v8(o2 + off, pk);
              co += 16;
              while (co >= args.c3) {  // 16 columns on: the next sub-pixel(s) when a sub-pixel has 8 or 16 channels
                co -= args.c3;
                ++ij;
              }
            }
          }
          continue;
        }
        const int ncol = t.n0 + c0 + jc * 4;  // first of this lane's 4 accumulator columns
        float4 xs[8], ys[8];
        {
          uint32_t v[32];
          tmem_ld_32x32(t_acc + c0, v);
          tmem_ld_wait();
          stage_in(v);
          __syncwarp();
          stage_out(xs);
          if (EPI == EPI_BIAS_SWIGLU) {
            __syncwarp();
            tmem_ld_32x32(t_acc + BN / 2 + c0, v);
            tmem_ld_wait();
            stage_in(v);
            __syncwarp();
            stage_out(ys);
          }
          __syncwarp();  // staging buffer free for the next chunk
        }
        if (ncol >= args.n_valid) continue;
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f), g4 = b4, b4b = b4;
        if (args.bias) b4 = __ldg(reinterpret_cast<const float4*>(args.bias + ncol));
        if (EPI == EPI_SCALE_RESIDUAL) g4 = __ldg(reinterpret_cast<const float4*>(args.gamma + ncol));
        if (EPI == EPI_BIAS_SWIGLU) b4b = __ldg(reinterpret_cast<const float4*>(args.bias + ncol + BN / 2));
        if (EPI == EPI_BIAS || EPI == EPI_BIAS_GELU || EPI == EPI_BIAS_SWIGLU) {
          const int ocol = EPI == EPI_BIAS_SWIGLU ? (t.n0 >> 1) + c0 + jc * 4 : ncol;
          __nv_bfloat16* obase = static_cast<__nv_bfloat16*>(args.out) + ocol;
          // branch-free row loops (uniform switches hoisted, stores predicated) so the rows' chains interleave
          if (EPI == EPI_BIAS_GELU && AMODE == AMODE_CONV3 && args.bias_table) {
            // folded GroupNorm: the bias row depends on which taps of this voxel are inside the volume
            const int dm = (t.d >= args.dil ? 1 : 0) | (t.d + args.dil < args.D ? 2 : 0);
#pragma unroll
            for (int it = 0; it < 8; ++it) {
              const int r = q * 32 + it * 4 + rsub;
              const int hl = r / args.BW, h = t.h0 + hl, w = t.w0 + (r - hl * args.BW);
              const int hm = (h >= 1 ? 1 : 0) | (h + 1 < args.H ? 2 : 0), wm = (w >= 1 ? 1 : 0) | (w + 1 < args.W ? 2 : 0);
              const float4 tb = __ldg(reinterpret_cast<const float4*>(args.bias_table + ((dm * 4 + hm) * 4 + wm) * args.N + ncol));
              xs[it].x += tb.x - b4.x; xs[it].y += tb.y - b4.y; xs[it].z += tb.z - b4.z; xs[it].w += tb.w - b4.w;
            }
          }
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            xs[it].x += b4.x; xs[it].y += b4.y; xs[it].z += b4.z; xs[it].w += b4.w;
            if (EPI == EPI_BIAS_SWIGLU) {
              xs[it].x = silu(xs[it].x) * (ys[it].x + b4b.x);
              xs[it].y = silu(xs[it].y) * (ys[it].y + b4b.y);
              xs[it].z = silu(xs[it].z) * (ys[it].z + b4b.z);
              xs[it].w = silu(xs[it].w) * (ys[it].w + b4b.w);
            }
          }
          if (!TF32 && (EPI == EPI_BIAS_GELU || EPI == EPI_BIAS) && args.act == ACT_GELU_GRAD) {
            // input-gradient GEMM / convolution: times gelu'(z) of the layer below, z read where the result is stored
            const __nv_bfloat16* zbase = static_cast<const __nv_bfloat16*>(args.aux) + ocol;
            uint2 z2[8];
#pragma unroll
            for (int it = 0; it < 8; ++it) {
              z2[it] = make_uint2(0u, 0u);
              if (grow_it[it] >= 0) z2[it] = __ldg(reinterpret_cast<const uint2*>(zbase + (size_t)grow_it[it] * args.ldo));
            }
#pragma unroll
            for (int it = 0; it < 8; ++it) {
              xs[it].x *= gelu_grad(__uint_as_float(z2[it].x << 16));
              xs[it].y *= gelu_grad(__uint_as_float(z2[it].x & 0xffff0000u));
              xs[it].z *= gelu_grad(__uint_as_float(z2[it].y << 16));
              xs[it].w *= gelu_grad(__uint_as_float(z2[it].y & 0xffff0000u));
            }
          }
          if (!TF32 && EPI == EPI_BIAS_GELU && args.act == ACT_DUAL) {
            // training forward: the pre-activation stays in `out` for the backward pass, the activation goes to `aux`
#pragma unroll
            for (int it = 0; it < 8; ++it)
              if (grow_it[it] >= 0)
                *reinterpret_cast<uint2*>(obase + (size_t)grow_it[it] * args.ldo) =
                    make_uint2(pack_bf16x2(xs[it].x, xs[it].y), pack_bf16x2(xs[it].z, xs[it].w));
            obase = static_cast<__nv_bfloat16*>(args.aux) + ocol;
          }
          if (EPI == EPI_BIAS_GELU && (args.act == ACT_GELU || args.act == ACT_DUAL)) {
#pragma unroll
            for (int it = 0; it < 8; ++it) {
              gelu_erf2(xs[it].x, xs[it].y);
              gelu_erf2(xs[it].z, xs[it].w);
            }
          }
          if (!TF32 && EPI == EPI_BIAS_GELU && AMODE != AMODE_CONV3 && args.gn_partials)
            gn_stats(xs, grow_it, t.m0 + (SUB == 1 ? 0 : sub * GEMM_BM) + q * 32, ncol);
          if (TF32 && EPI != EPI_BIAS) {
            // the FFN hidden activations of the TF32 path: fp32, rounded to TF32 so the next GEMM reads them exactly
            float* of = static_cast<float*>(args.out) + ocol;
#pragma unroll
            for (int it = 0; it < 8; ++it)
              if (grow_it[it] >= 0)
                *reinterpret_cast<float4*>(of + (size_t)grow_it[it] * args.ldo) =
                    make_float4(round_tf32(xs[it].x), round_tf32(xs[it].y), round_tf32(xs[it].z), round_tf32(xs[it].w));
            continue;
          }
          uint2 pk[8];
          if (out_f16) {
#pragma unroll
            for (int it = 0; it < 8; ++it) pk[it] = make_uint2(pack_f16x2(xs[it].x, xs[it].y), pack_f16x2(xs[it].z, xs[it].w));
          } else {
#pragma unroll
            for (int it = 0; it < 8; ++it) pk[it] = make_uint2(pack_bf16x2(xs[it].x, xs[it].y), pack_bf16x2(xs[it].z, xs[it].w));
          }
#pragma unroll
          for (int it = 0; it < 8; ++it)
            if (grow_it[it] >= 0) *reinterpret_cast<uint2*>(obase + (size_t)grow_it[it] * args.ldo) = pk[it];
        } else if (EPI == EPI_SCALE_RESIDUAL) {
          float* xbase = static_cast<float*>(args.out) + ncol;
          float4 resid[8];
          // issue all residual loads up front so their latency overlaps (the stores below may alias them)
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            resid[it] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (grow_it[it] >= 0) resid[it] = *reinterpret_cast<const float4*>(xbase + (size_t)grow_it[it] * args.ldo);
          }
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            float4 r = resid[it];
            r.x += g4.x * (xs[it].x + b4.x);
            r.y += g4.y * (xs[it].y + b4.y);
            r.z += g4.z * (xs[it].z + b4.z);
            r.w += g4.w * (xs[it].w + b4.w);
            if (grow_it[it] >= 0) *reinterpret_cast<float4*>(xbase + (size_t)grow_it[it] * args.ldo) = r;
          }
        } else if (EPI == EPI_PATCH_EMBED) {
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            const int grow = grow_it[it];
            if (grow < 0) continue;
            const int b = grow / args.pe_np, p = grow - b * args.pe_np;
            const float4 tb = __ldg(reinterpret_cast<const float4*>(args.table + (size_t)p * args.N + ncol));
            const float4 o = make_float4(xs[it].x + tb.x + b4.x, xs[it].y + tb.y + b4.y, xs[it].z + tb.z + b4.z, xs[it].w + tb.w + b4.w);
            const size_t orow = (size_t)b * args.pe_tokens + args.pe_offset + p;
            *reinterpret_cast<float4*>(static_cast<float*>(args.out) + orow * args.ldo + ncol) = o;
          }
        } else if (EPI == EPI_CONVT_GELU) {
          // column n = (i*2 + j) * c3 + co ; voxel grow = (d*H + h)*W + w -> out[d, 2h+i, 2w+j, co]
          const int ij = ncol / args.c3, co = ncol - ij * args.c3;
          const int si = ij >> 1, sj = ij & 1;
          // rows of a chunk are 4 voxels apart (plain-rows GEMM): one division per chunk, then (w, dh) are stepped.
          // The loops below are kept free of branches (predicated selects, activation switch hoisted, stores predicated)
          // so that the eight rows' GELU chains interleave: with two epilogue warps per scheduler the kernel waited on
          // fixed-latency dependencies (ncu: 38 % stall_wait, 8 % branch resolving with a branchy row loop).
          size_t off_it[8];
          {
            const int g0 = t.m0 + (SUB == 1 ? 0 : sub * GEMM_BM) + q * 32 + rsub;
            int dh = g0 / args.W;  // dh = d*H + h
            int w = g0 - dh * args.W;
            const int W2 = 2 * args.W;
            if (args.W >= 4) {
#pragma unroll
              for (int it = 0; it < 8; ++it) {
                if (it > 0) {
                  w += 4;
                  const int wrap = w >= args.W ? 1 : 0;
                  w -= wrap * args.W;
                  dh += wrap;
                }
                off_it[it] = ((size_t)(2 * dh + si) * W2 + 2 * w + sj) * args.c3 + co;
              }
            } else {
#pragma unroll
              for (int it = 0; it < 8; ++it) {
                if (it > 0) {
                  w += 4;
                  while (w >= args.W) { w -= args.W; ++dh; }
                }
                off_it[it] = ((size_t)(2 * dh + si) * W2 + 2 * w + sj) * args.c3 + co;
              }
            }
          }
          uint2 pk[8];
          __nv_bfloat16* obaseT = static_cast<__nv_bfloat16*>(args.out);
          if (args.act == ACT_DUAL) {  // training forward: pre-activation -> out, activation -> aux
#pragma unroll
            for (int it = 0; it < 8; ++it)
              if (grow_it[it] >= 0)
                *reinterpret_cast<uint2*>(obaseT + off_it[it]) =
                    make_uint2(pack_bf16x2(xs[it].x + b4.x, xs[it].y + b4.y), pack_bf16x2(xs[it].z + b4.z, xs[it].w + b4.w));
            obaseT = static_cast<__nv_bfloat16*>(args.aux);
          }
          if (args.act) {
#pragma unroll
            for (int it = 0; it < 8; ++it) {
              float o0 = xs[it].x + b4.x, o1 = xs[it].y + b4.y, o2 = xs[it].z + b4.z, o3 = xs[it].w + b4.w;
              gelu_erf2(o0, o1);
              gelu_erf2(o2, o3);
              pk[it] = make_uint2(pack_bf16x2(o0, o1), pack_bf16x2(o2, o3));
              xs[it] = make_float4(o0, o1, o2, o3);
            }
            // statistics for the GroupNorm that follows: columns (i, j, co) -> groups of gn_cpg channels per sub-pixel
            if (args.gn_partials) gn_stats(xs, grow_it, t.m0 + (SUB == 1 ? 0 : sub * GEMM_BM) + q * 32, ncol);
          } else {
#pragma unroll
            for (int it = 0; it < 8; ++it)
              pk[it] = make_uint2(pack_bf16x2(xs[it].x + b4.x, xs[it].y + b4.y), pack_bf16x2(xs[it].z + b4.z, xs[it].w + b4.w));
          }
#pragma unroll
          for (int it = 0; it < 8; ++it)
            if (grow_it[it] >= 0) *reinterpret_cast<uint2*>(obaseT + off_it[it]) = pk[it];
        }
      }
      // all TMEM reads of this accumulator buffer are complete (every tcgen05.ld was waited on)
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) mbar_arrive_cluster(mapa_cluster(bar_tempty + 8 * acc, 0));  // the leader's issuer waits for both CTAs
        else mbar_arrive(bar_tempty + 8 * acc);
      }
      acc ^= 1;
      if (acc == 0) acc_ph ^= 1u;
    }
    if (EPI == EPI_CONVT_GELU && args.gn_partials && args.gn_direct) {
      // one partials row per epilogue thread: [8 groups][sum, sum of squares] of everything it stored
      float4* dst = reinterpret_cast<float4*>(args.gn_partials) + ((size_t)blockIdx.x * 256 + (ew * 32 + lane)) * 4;
#pragma unroll
      for (int i = 0; i < 4; ++i) dst[i] = make_float4(gsum[2 * i], gsq[2 * i], gsum[2 * i + 1], gsq[2 * i + 1]);
    }
  }

  tcgen05_fence_before();
  if (PAIR) cluster_sync_all();  // neither CTA may exit (or free TMEM) while the pair's MMAs / remote arrivals are in flight
  else __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tcgen05_fence_after();
    if (PAIR) tmem_dealloc_pair<Cfg::TMEM_COLS>(tmem_base);
    else tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

}  // namespace cvit
