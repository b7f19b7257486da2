// 3x3x3 "same" convolution (dilation 1) of an 8-channel channels-last volume into 8 channels, + bias (+ GELU): the
// full-resolution output_layer.0 of the CryoVIT head (models/cryovit.py:30-32) and its two input gradients in training,
// with A ROW OF VOXELS AS THE ROWS OF ONE MMA AND NO RE-LAYOUT (the idea of csrc/wgrad_tc.cu turned around).
//
// Why. conv3d_wpack packs 8 output voxels into an MMA row and pays for it with banded weights: 3 of every 10 multiplies
// are useful, 15 MMAs (N = 192) per 1024 voxels and input plane, 0.40 ms for 33.5 M voxels (tensor pipe 44 % busy, all of
// it streaming A). Here an MMA row is ONE voxel x and K runs over its three column taps:
//
//   A[x][k = (kw, ci)] = X[z', y', x - 1 + kw][ci]   -- 8 channels of a channels-last voxel are 16 bytes, so the row segment as
//       it lies in shared memory is a K-major SWIZZLE_NONE operand whose rows are 16 bytes apart (a core matrix = 8 voxels
//       x 16 bytes = 128 contiguous bytes, SBO = 128) and whose next K chunk -- the next column tap -- is the SAME bytes one
//       voxel further on (LBO = 16). K = 32: taps kw = 0..3, the fourth against zero weights.
//   B[n = (yr, p, co)][k] = w[co][ci][kd][kh = 2 - yr][kw]   -- one input row (z', y') feeds the nine output rows
//       (z' - (kd-1), y' - (kh-1)); yr = 0..2 counts the output rows y' - 1 + yr, p the output planes.
//   D[x][n]: 128 voxels x 72 numbers per input row, 2 MMAs (K = 32) -- 16 MMAs (N = 80) per 1024 voxels and input plane, all
//       multiplies useful.
//
// The nine partial sums of an output voxel come from nine different input rows. They meet IN TENSOR MEMORY: an accumulator
// column is (output row slot r, output plane slot p, co), r-major, so the 72 columns an input row writes are one
// contiguous window that slides by 24 columns per input row, and the MMAs of consecutive rows accumulate into overlapping
// windows. Output plane zo lives in plane slot zo mod 3; which kd an input plane contributes to which slot depends on
// z' mod 3, so the weights are kept as three images. When input plane z' is done, output plane z' - 1 is complete: the
// epilogue warps read its slot (thread = voxel: 16 contiguous bytes per thread, 512 per warp), add bias, apply GELU, store,
// and ZERO the slot for plane z' + 2. Rows at the edge of the tile use shorter windows (N = 32 / 64 / 48 / 32 from image
// rows 48 / 24 / 0 / 0; zero rows behind the image make the overhang add zeros, a pad slot takes the last row's).
//
// A work unit is (16 output planes, 8 output rows, two 128-voxel segments): the two segments own half of TMEM each and
// alternate plane by plane, so one's epilogue runs under the other's MMAs. One CTA per SM, 320 threads: warp 0 TMA producer
// (ONE box of whole 128-byte lines for the ten input rows of a (plane, segment) -- with a box per row the TMA issue rate
// bounded the kernel at 0.46 ms -- zero fill = padding), warp 1 MMA issuer (row loop unrolled, descriptors = base + constant),
// warps 2-9 epilogue (two warps per TMEM lane quarter, half of the tile's rows each).
#include "ptx.cuh"
#include "tmap.h"

namespace cvit {

constexpr int CR_THREADS = 320;
constexpr int CR_HT = 8;                       // output rows per unit
constexpr int CR_ZC = 16;                      // output planes per unit
constexpr int CR_SEG = 128;                    // voxels per segment
constexpr int CR_XARR = (CR_SEG + 16) * 16;    // input row array: voxels x0 - 8 .. x0 + 135 (18 lines of 128 bytes)
constexpr int CR_ROWS = CR_HT + 2;             // input rows per (plane, segment): one TMA box, one pipeline stage
constexpr int CR_STAGE = CR_ROWS * CR_XARR;    // 23040 bytes
constexpr int CR_STAGES = 6;
constexpr int CR_IMG_ROWS = 96;                // 72 weight rows + 24 zero rows
constexpr int CR_IMG_KSTEP = 2 * CR_IMG_ROWS * 16;  // [chunk][row][8]: 3072 bytes
constexpr int CR_IMG_BYTES = 3 * 2 * CR_IMG_KSTEP;  // [z' mod 3][K step]: 18432 bytes
constexpr int CR_SLOT = 24;                    // columns per output row slot: 3 plane slots x 8 channels
constexpr int CR_SEG_COLS = 256;               // TMEM columns per segment ((HT + 1) * 24 = 216 used)
constexpr int CR_SMEM = CR_STAGES * CR_STAGE + CR_IMG_BYTES + 512 + 1024;

// Order in which the HT + 2 input rows of a (plane, segment) are loaded and multiplied: i = y' - yt0 in [-1, HT].
#ifndef CR_ORDER
#define CR_ORDER 0
#endif
__device__ __forceinline__ int cr_row(int k) {
#if CR_ORDER == 1
  // consecutive MMAs write windows at least four row slots apart (no column of one in the next): 0 4 8 1 5 -1 2 6 3 7
  constexpr int order[CR_HT + 2] = {0, 4, 8, 1, 5, -1, 2, 6, 3, 7};
  return order[k];
#else
  return k - 1;
#endif
}

struct CrArgs {
  const __nv_bfloat16* w_img;  // CR_IMG_BYTES, host-arranged (cryovit_b200.head.rows8_weight_image)
  const float* bias;           // [8] (FINAL: only bias[0] is used)
  __nv_bfloat16* out;          // [D, H, W, 8]
  __nv_bfloat16* aux;          // act = ACT_DUAL: gelu(out); ACT_GELU_GRAD: the pre-activation z whose gelu' scales the result
  float* db;                   // ACT_GELU_GRAD: fp32 [8] column sums of what is stored are added here (may be null)
  float* logits;               // FINAL: [D, H, W] clipped logits (may be null)
  float* probs;                // FINAL: [D, H, W] sigmoid of the clipped logits (may be null)
  int D, H, W, act;
  const int8_t* labels;        // SCORE: [D, H, W], -1 = ignore
  double* partials;            // SCORE: [gridDim.x][8], one row per CTA
  float thr;                   // SCORE: threshold of sums 3 and 4
};

__device__ __forceinline__ uint64_t cr_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) {  // K-major SWIZZLE_NONE
  return static_cast<uint64_t>((addr & 0x3ffffu) >> 4) | (static_cast<uint64_t>(lbo >> 4) << 16) |
         (static_cast<uint64_t>(sbo >> 4) << 32) | (1ull << 46);
}
__device__ __forceinline__ void cr_tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}

// R8_FINAL: output_layer.2 (8 -> 1): the same MMAs on a weight image whose channels 1..7 are zero (an M = 128 MMA costs the
// same for any N <= 128), the epilogue keeps column 0: clip(-5, 5) (+ sigmoid), fp32, 128 contiguous bytes per warp.
// R8_SCORE: the same MMAs, clip and sigmoid, but the epilogue stores nothing: it reads the voxel's int8 label and
// accumulates the eight masked sums of cvit_seg_stats (csrc/head_elementwise.cu) over the voxels whose label is > -1.
//   - Exact counts: labels are integers, so sums 1 and 3..7 are integer counts. They are accumulated in integers (per
//     thread), then reduced in fp64, which is exact below 2^53. The soft sums 0 and 2 accumulate per thread in fp32 over
//     one work unit (64 voxels), then in fp64.
//   - Deterministic: each CTA reduces its threads in a fixed order (shuffle tree, then warp by warp) and writes ONE fp64 row
//     of 8 into args.partials; cvit_conv3d_rows8_score's one-block finalize kernel adds the rows in a fixed order. No
//     atomics: two runs give bit-identical sums.
enum Rows8Mode { R8_CONV = 0, R8_FINAL = 1, R8_SCORE = 2 };

template <int MODE>
__global__ void __launch_bounds__(CR_THREADS, 1) conv3d_rows8_kernel(const __grid_constant__ CUtensorMap tmX, const CrArgs args) {
  constexpr bool FINAL = MODE != R8_CONV;  // one output channel (R8_FINAL, R8_SCORE)
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sX = smem_base, sW = smem_base + CR_STAGES * CR_STAGE, sBar = sW + CR_IMG_BYTES;
  const uint32_t bar_full = sBar, bar_empty = sBar + 8 * CR_STAGES;
  const uint32_t bar_done = sBar + 16 * CR_STAGES, bar_free = bar_done + 16, tmem_slot = bar_free + 16;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const int seg_pairs = (args.W + 2 * CR_SEG - 1) / (2 * CR_SEG), ytiles = (args.H + CR_HT - 1) / CR_HT;
  const int zchunks = (args.D + CR_ZC - 1) / CR_ZC;
  const int num_units = seg_pairs * ytiles * zchunks;
  auto unit_of = [&](int u, int& xp, int& yt0, int& za, int& zb) {  // z chunk fastest: neighbours in time share input planes in L2
    const int zc = u % zchunks, r = u / zchunks;
    xp = (r % seg_pairs) * 2 * CR_SEG;
    yt0 = (r / seg_pairs) * CR_HT;
    za = zc * CR_ZC;
    zb = min(za + CR_ZC, args.D);
  };

  // weights -> shared memory (generic proxy), barriers, TMEM
  for (int i = threadIdx.x; i < CR_IMG_BYTES / 16; i += CR_THREADS)
    reinterpret_cast<uint4*>(smem_gen + (sW - smem_base))[i] = __ldg(reinterpret_cast<const uint4*>(args.w_img) + i);
  fence_proxy_async_smem();
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmX);
    for (int s = 0; s < CR_STAGES; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    for (int g = 0; g < 2; ++g) {
      mbar_init(bar_done + 8 * g, 1);  // MMA -> epilogue: the segment's MMAs of one input plane have retired
      mbar_init(bar_free + 8 * g, 8);  // epilogue -> MMA: the slot is drained and zeroed (one arrival per warp)
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer: input rows in the order the MMAs want them
    if (lane == 0) {
      uint32_t it = 0;
      for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
        int xp, yt0, za, zb;
        unit_of(u, xp, yt0, za, zb);
        for (int zi = za - 1; zi <= zb; ++zi) {
          if (zi < 0 || zi >= args.D) continue;
          for (int g = 0; g < 2; ++g, ++it) {  // the HT + 2 input rows of (plane, segment): ONE box (one TMA per 2 MMAs bounded v1)
            const uint32_t s = it % CR_STAGES;
            mbar_wait(bar_empty + 8 * s, ((it / CR_STAGES) & 1) ^ 1u);
            mbar_arrive_expect_tx(bar_full + 8 * s, CR_STAGE);
            tma_load_4d(sX + s * CR_STAGE, &tmX, bar_full + 8 * s, 0, (xp + g * CR_SEG) / 8 - 1, yt0 - 1, zi);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t id32 = umma_idesc_bf16_f32(128, 32), id48 = umma_idesc_bf16_f32(128, 48), id64 = umma_idesc_bf16_f32(128, 64),
                       id80 = umma_idesc_bf16_f32(128, 80);
    uint32_t it = 0, np[2] = {0, 0};  // stage counter; planes issued per segment (phase of bar_free)
    const uint64_t a_base = cr_desc(sX + 7 * 16, 16, 128);  // stage 0, voxel x0 - 1; LBO = 16: the next column tap = the next voxel
    for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
      int xp, yt0, za, zb;
      unit_of(u, xp, yt0, za, zb);
      for (int zi = za - 1; zi <= zb; ++zi) {
        const bool real = zi >= 0 && zi < args.D;
        const uint32_t img = sW + ((zi + 3) % 3) * (2 * CR_IMG_KSTEP);
        for (int g = 0; g < 2; ++g) {
#ifndef CR_DEBUG_NOWAIT  // (timing experiment only: wrong results)
          mbar_wait(bar_free + 8 * g, np[g] & 1);  // every slot this plane's windows touch is zero or live
#endif
          tcgen05_fence_after();
          ++np[g];
          if (real) {
            // The row loop is unrolled: window (image rows from r0, n columns from row slot `slot`) and instruction descriptor
            // of every row are compile-time constants, the operand descriptors are a base plus a constant -- the issuing
            // thread's own instruction stream was the bottleneck of the first version (460 cycles per row for two MMAs).
            const uint32_t d_seg = tmem_base + g * CR_SEG_COLS;
            const uint64_t b_base = cr_desc(img, CR_IMG_ROWS * 16, 128);
            const uint32_t s = it % CR_STAGES;
            mbar_wait(bar_full + 8 * s, (it / CR_STAGES) & 1);
            tcgen05_fence_after();
            ++it;
            if (elect_one_sync()) {
              const uint64_t a_stage = a_base + s * (CR_STAGE >> 4);
#pragma unroll
              for (int k = 0; k < CR_ROWS; ++k) {
                const int i = cr_row(k);
                const int r0 = i == -1 ? 48 : i == 0 ? 24 : 0;
                const int slot = i <= 0 ? 0 : i - 1;
                const uint32_t idesc = i == -1 ? id32 : i == 0 ? id64 : i == CR_HT - 1 ? id48 : i == CR_HT ? id32 : id80;
                const uint64_t ad = a_stage + (i + 1) * (CR_XARR >> 4);
#pragma unroll
                for (int ks = 0; ks < 2; ++ks)  // column taps (0, 1) and (2, 3: zero weights)
                  umma_bf16(d_seg + slot * CR_SLOT, ad + 2 * ks, b_base + ks * (CR_IMG_KSTEP >> 4) + r0, idesc, 1u);
              }
              umma_commit(bar_empty + 8 * s);
            }
            __syncwarp();
          }
          if (elect_one_sync()) umma_commit(bar_done + 8 * g);
          __syncwarp();
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue: all eight warps drain every (plane, segment):
    // warps 2-5 the output rows 0..3 of the tile, warps 6-9 rows 4..7 (the drain sits between "plane z' done" and "plane
    // z' + 1 may start" of its segment, so its latency, not its throughput, is what the other segment's MMAs have to cover)
    const int half = (warp - 2) >> 2, q = warp & 3;
    constexpr int RH = CR_HT / 2;
    float bias[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) bias[c] = __ldg(args.bias + c);
    const uint32_t zeros[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
    auto seg_addr = [&](int g) { return tmem_base + g * CR_SEG_COLS + (static_cast<uint32_t>(q * 32) << 16); };
    auto zero_all = [&](int g) {  // this half's row slots (the second half takes the pad slot too)
      const int c0 = half * RH * CR_SLOT, c1 = half ? (CR_HT + 1) * CR_SLOT : RH * CR_SLOT;
#pragma unroll 1
      for (int c = c0; c < c1; c += 8) tmem_st_32x8(seg_addr(g) + c, zeros);
    };
    auto hand_back = [&](int g) {
      tmem_st_wait();
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_free + 8 * g);
    };
    for (int g = 0; g < 2; ++g) {
      zero_all(g);
      hand_back(g);
    }
    uint32_t nd = 0;  // planes drained per segment (phase of bar_done)
    float bsum[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // ACT_GELU_GRAD: column sums of what this thread stores
    // R8_SCORE: soft sums 0, 2 (fp32 over the current unit, fp64 over all) and the counts 1, 3, 4, 5, 6, 7
    float soft32[2] = {0.f, 0.f};
    double soft64[2] = {0.0, 0.0};
    int cnt[6] = {0, 0, 0, 0, 0, 0};
    for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
      int xp, yt0, za, zb;
      unit_of(u, xp, yt0, za, zb);
      for (int zi = za - 1; zi <= zb; ++zi, ++nd) {
        const int zo = zi - 1, p = (zo + 3) % 3;
        for (int g = 0; g < 2; ++g) {
          const uint32_t t_seg = seg_addr(g);
          const int x = xp + g * CR_SEG + q * 32 + lane;
          // ACT_GELU_GRAD: the z values of the plane about to be drained are requested before the wait for its MMAs
          uint4 zz[RH];
          // R8_SCORE: so are the labels
          int lab[RH];
          if constexpr (MODE == R8_SCORE) {
#pragma unroll
            for (int r = 0; r < RH; ++r) {
              const int y = yt0 + half * RH + r;
              lab[r] = -1;
              if (zo >= za && zo < zb && y < args.H && x < args.W) lab[r] = __ldg(args.labels + ((size_t)zo * args.H + y) * args.W + x);
            }
          }
          if (!FINAL && args.act == ACT_GELU_GRAD && zo >= za && zo < zb) {
#pragma unroll
            for (int r = 0; r < RH; ++r) {
              const int y = yt0 + half * RH + r;
              zz[r] = make_uint4(0u, 0u, 0u, 0u);
              if (y < args.H && x < args.W) zz[r] = __ldg(reinterpret_cast<const uint4*>(args.aux + (((size_t)zo * args.H + y) * args.W + x) * 8));
            }
          }
          mbar_wait(bar_done + 8 * g, nd & 1);
          tcgen05_fence_after();
          // Read this half's rows of the finished plane, zero the slot and hand it back BEFORE the math and the stores: the other
          // segment's MMAs cover the drain's TMEM round trips, not its GELUs.
          const bool live = zo >= za && zo < zb;
          uint32_t v[RH][8];
          if (live) {
#pragma unroll
            for (int r = 0; r < RH; ++r) cr_tmem_ld8(t_seg + (half * RH + r) * CR_SLOT + p * 8, v[r]);
            tmem_ld_wait();
          }
          if (zi == zb) {
            zero_all(g);  // the unit's last plane: everything (the halo planes' leftovers too) is cleared for the next unit
          } else {
#pragma unroll
            for (int r = 0; r < RH; ++r) tmem_st_32x8(t_seg + (half * RH + r) * CR_SLOT + p * 8, zeros);  // slot p: plane zo + 3 next
          }
          hand_back(g);
          if (live) {
#pragma unroll
            for (int r = 0; r < RH; ++r) {
              const int y = yt0 + half * RH + r;
              if (y < args.H && x < args.W) {
                if constexpr (MODE == R8_SCORE) {
                  if (lab[r] > -1) {
                    const float lg = fminf(fmaxf(__uint_as_float(v[r][0]) + bias[0], -5.0f), 5.0f);
                    const float p = 1.0f / (1.0f + __expf(-lg));
                    const int yl = lab[r], hge = p >= args.thr, hgt = p > 0.5f;
                    soft32[0] += p;
                    soft32[1] += p * (float)yl;
                    cnt[0] += yl;
                    cnt[1] += yl * hge;
                    cnt[2] += hge;
                    cnt[3] += yl * hgt;
                    cnt[4] += (1 - yl) * hgt;
                    cnt[5] += yl * (1 - hgt);
                  }
                  continue;
                } else if (FINAL) {
                  const size_t vox = ((size_t)zo * args.H + y) * args.W + x;
                  const float lg = fminf(fmaxf(__uint_as_float(v[r][0]) + bias[0], -5.0f), 5.0f);
                  if (args.logits) args.logits[vox] = lg;
                  if (args.probs) args.probs[vox] = 1.0f / (1.0f + __expf(-lg));
                  continue;
                }
                const size_t off = (((size_t)zo * args.H + y) * args.W + x) * 8;
                float o[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) o[c] = __uint_as_float(v[r][c]) + bias[c];
                if (args.act == ACT_GELU_GRAD) {
                  const uint32_t zw[4] = {zz[r].x, zz[r].y, zz[r].z, zz[r].w};
                  uint32_t pk[4];
#pragma unroll
                  for (int c = 0; c < 4; ++c) {
                    pk[c] = act_gelu_grad_pair(o[2 * c], o[2 * c + 1], zw[c]);
                    bsum[2 * c] += __uint_as_float(pk[c] << 16);  // sums over the STORED gradient
                    bsum[2 * c + 1] += __uint_as_float(pk[c] & 0xffff0000u);
                  }
                  *reinterpret_cast<uint4*>(args.out + off) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                  continue;
                }
                if (args.act == ACT_DUAL)
                  *reinterpret_cast<uint4*>(args.out + off) =
                      make_uint4(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]), pack_bf16x2(o[4], o[5]), pack_bf16x2(o[6], o[7]));
                if (args.act) {
                  gelu_erf2(o[0], o[1]);
                  gelu_erf2(o[2], o[3]);
                  gelu_erf2(o[4], o[5]);
                  gelu_erf2(o[6], o[7]);
                }
                __nv_bfloat16* dst = args.act == ACT_DUAL ? args.aux : args.out;
                *reinterpret_cast<uint4*>(dst + off) =
                    make_uint4(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]), pack_bf16x2(o[4], o[5]), pack_bf16x2(o[6], o[7]));
              }
            }
          }
        }
      }
      if constexpr (MODE == R8_SCORE) {
        soft64[0] += soft32[0];
        soft64[1] += soft32[1];
        soft32[0] = soft32[1] = 0.f;
      }
    }
    if constexpr (MODE == R8_SCORE) {  // this warp's eight sums -> shared memory (summed per CTA below, in warp order)
      double t[8] = {soft64[0], (double)cnt[0], soft64[1], (double)cnt[1], (double)cnt[2], (double)cnt[3], (double)cnt[4],
                     (double)cnt[5]};
#pragma unroll
      for (int k = 0; k < 8; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t[k] += __shfl_xor_sync(0xffffffffu, t[k], o);
      }
      if (lane < 8) {
        double mine = t[0];
#pragma unroll
        for (int k = 1; k < 8; ++k)
          if (lane == k) mine = t[k];
        reinterpret_cast<double*>(smem_gen + (sX - smem_base))[(warp - 2) * 8 + lane] = mine;  // stages idle: every MMA retired
      }
    }
    if (!FINAL && args.act == ACT_GELU_GRAD && args.db) {  // bias gradient: one shuffle tree and 8 atomics per warp
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const float tot = warp_sum(bsum[c]);
        if (lane == 0) atomicAdd(args.db + c, tot);
      }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if constexpr (MODE == R8_SCORE) {
    if (threadIdx.x < 8) {
      const double* red = reinterpret_cast<const double*>(smem_gen + (sX - smem_base));
      double s = 0.0;
      for (int w = 0; w < 8; ++w) s += red[w * 8 + threadIdx.x];
      args.partials[(size_t)blockIdx.x * 8 + threadIdx.x] = s;
    }
  }
  if (warp == 1) {
    __syncwarp();
    tcgen05_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// R8_SCORE's second step: out8[k] = the sum of partials[r][k] over the rows r = 0 .. rows - 1, in a fixed order.
__global__ void __launch_bounds__(256) rows8_score_finalize_kernel(const double* __restrict__ partials, int rows, double* __restrict__ out8) {
  __shared__ double red[32][8];
  const int k = threadIdx.x & 7, j = threadIdx.x >> 3;
  double s = 0.0;
  for (int r = j; r < rows; r += 32) s += partials[(size_t)r * 8 + k];
  red[j][k] = s;
  __syncthreads();
  if (threadIdx.x < 8) {
    double t = 0.0;
    for (int i = 0; i < 32; ++i) t += red[i][threadIdx.x];
    out8[threadIdx.x] = t;
  }
}

}  // namespace cvit

using namespace cvit;

extern "C" int64_t cvit_conv3d_rows8_weight_bytes() { return CR_IMG_BYTES; }

// out (bf16 [D,H,W,8]) = conv3d(x bf16 [D,H,W,8], 3x3x3, "same", dilation 1) + bias, act: 0 none, 1 GELU, 2 out = pre-activation
// and aux = GELU of it, 3 out = result * gelu'(aux) with db (fp32 [8], may be null) += the column sums of what is stored (ptx.cuh ACT_*). w_img: cvit_conv3d_rows8_weight_bytes() bytes in the layout of
// cryovit_b200.head.rows8_weight_image. W must be a multiple of 8.
static int64_t rows8_units(int64_t D, int64_t H, int64_t W) {
  return ((W + 2 * CR_SEG - 1) / (2 * CR_SEG)) * ((H + CR_HT - 1) / CR_HT) * ((D + CR_ZC - 1) / CR_ZC);
}

static int rows8_launch(const void* x, CrArgs a, int mode, cudaStream_t stream, double* out8 = nullptr) {
  CUtensorMap tmX;
  uint64_t dims[4] = {64, (uint64_t)(a.W / 8), (uint64_t)a.H, (uint64_t)a.D};
  uint64_t strides[4] = {0, 128, (uint64_t)a.W * 16, (uint64_t)a.H * a.W * 16};
  uint32_t box[4] = {64, CR_SEG / 8 + 2, CR_ROWS, 1};
  int rc = encode_tmap(&tmX, TmapDtype::BF16, 4, x, dims, strides, box, 0);
  if (rc) return rc;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(conv3d_rows8_kernel<R8_CONV>, cudaFuncAttributeMaxDynamicSharedMemorySize, CR_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3d_rows8_kernel<R8_FINAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, CR_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3d_rows8_kernel<R8_SCORE>, cudaFuncAttributeMaxDynamicSharedMemorySize, CR_SMEM);
    if (e != cudaSuccess) {
      set_error("conv3d_rows8: cudaFuncSetAttribute(smem=%d): %s", CR_SMEM, cudaGetErrorString(e));
      return CVIT_ERR_CUDA;
    }
    configured = true;
  }
  const int64_t units = rows8_units(a.D, a.H, a.W);
  int grid = num_sms();
  if (grid > units) grid = (int)units;
  if (mode == R8_SCORE) {
    conv3d_rows8_kernel<R8_SCORE><<<grid, CR_THREADS, CR_SMEM, stream>>>(tmX, a);
    if (int rc2 = check_launch("conv3d_rows8_kernel<score>")) return rc2;
    rows8_score_finalize_kernel<<<1, 256, 0, stream>>>(a.partials, grid, out8);
    return check_launch("rows8_score_finalize_kernel");
  }
  if (mode == R8_FINAL) conv3d_rows8_kernel<R8_FINAL><<<grid, CR_THREADS, CR_SMEM, stream>>>(tmX, a);
  else conv3d_rows8_kernel<R8_CONV><<<grid, CR_THREADS, CR_SMEM, stream>>>(tmX, a);
  return check_launch("conv3d_rows8_kernel");
}

static int rows8_check(const void* x, const void* w_img, const float* bias, int64_t D, int64_t H, int64_t W) {
  if (!x || !w_img || !bias || D <= 0 || H <= 0 || W <= 0) {
    set_error("conv3d_rows8: bad arguments (D=%lld H=%lld W=%lld)", (long long)D, (long long)H, (long long)W);
    return CVIT_ERR_INVALID;
  }
  if (W % 8) {
    set_error("conv3d_rows8: W=%lld must be a multiple of 8 (use cvit_conv3d_wpack8_* / cvit_conv3d_halo_ndhwc otherwise)", (long long)W);
    return CVIT_ERR_UNSUPPORTED;
  }
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(w_img)) & 15u) {
    set_error("conv3d_rows8: x and w_img must be 16-byte aligned");
    return CVIT_ERR_INVALID;
  }
  return CVIT_OK;
}

extern "C" int cvit_conv3d_rows8(const void* x, const void* w_img, const float* bias, void* out, int64_t D, int64_t H, int64_t W,
                                 int act, void* aux, float* db, void* stream) {
  if (int rc = rows8_check(x, w_img, bias, D, H, W)) return rc;
  if (!out || act < 0 || act > 3 || (act >= 2 && !aux) || ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(aux)) & 15u)) {
    set_error("conv3d_rows8: act must be 0, 1, 2 or 3 (2, 3 with aux); out and aux 16-byte aligned bf16 [D,H,W,8]");
    return CVIT_ERR_INVALID;
  }
  CrArgs a;
  a.w_img = static_cast<const __nv_bfloat16*>(w_img);
  a.bias = bias;
  a.out = static_cast<__nv_bfloat16*>(out);
  a.aux = static_cast<__nv_bfloat16*>(aux);
  a.db = db;
  a.logits = nullptr;
  a.probs = nullptr;
  a.D = (int)D;
  a.H = (int)H;
  a.W = (int)W;
  a.act = act;
  a.labels = nullptr;
  a.partials = nullptr;
  a.thr = 0.f;
  return rows8_launch(x, a, R8_CONV, (cudaStream_t)stream);
}

// output_layer.2 (8 -> 1) + bias + clip(-5, 5) -> logits fp32 [D,H,W] and/or sigmoid of them -> probs; w_img: the rows8 image of
// the [1, 8, 3, 3, 3] weight (channels 1..7 zero), bias fp32 [>= 1].
extern "C" int cvit_conv3d_rows8_final(const void* x, const void* w_img, const float* bias, float* logits, float* probs, int64_t D,
                                       int64_t H, int64_t W, void* stream) {
  if (int rc = rows8_check(x, w_img, bias, D, H, W)) return rc;
  if (!logits && !probs) {
    set_error("conv3d_rows8_final: need logits and/or probs");
    return CVIT_ERR_INVALID;
  }
  CrArgs a;
  a.w_img = static_cast<const __nv_bfloat16*>(w_img);
  a.bias = bias;
  a.out = nullptr;
  a.aux = nullptr;
  a.db = nullptr;
  a.logits = logits;
  a.probs = probs;
  a.D = (int)D;
  a.H = (int)H;
  a.W = (int)W;
  a.act = 0;
  a.labels = nullptr;
  a.partials = nullptr;
  a.thr = 0.f;
  return rows8_launch(x, a, R8_FINAL, (cudaStream_t)stream);
}

// Doubles of the partials buffer cvit_conv3d_rows8_score needs for a [D, H, W] volume (one row of 8 per work unit: at least
// one per CTA of any grid); depends on the shape only.
extern "C" int64_t cvit_conv3d_rows8_score_partials(int64_t D, int64_t H, int64_t W) {
  if (D <= 0 || H <= 0 || W <= 0) return 0;
  return 8 * rows8_units(D, H, W);
}

// output_layer.2 (8 -> 1) + bias + clip(-5, 5) + sigmoid as cvit_conv3d_rows8_final, scored instead of stored: out8 (fp64 [8],
// overwritten) = the eight masked sums of cvit_seg_stats of (probabilities, labels) with labels int8 [D,H,W] (-1 = ignore).
// partials: cvit_conv3d_rows8_score_partials(D, H, W) doubles of scratch. Counts (1, 3..7) exact; bit-identical across runs.
extern "C" int cvit_conv3d_rows8_score(const void* x, const void* w_img, const float* bias, const int8_t* labels, int64_t D,
                                       int64_t H, int64_t W, float threshold, double* partials, double* out8, void* stream) {
  if (int rc = rows8_check(x, w_img, bias, D, H, W)) return rc;
  if (!labels || !partials || !out8) {
    set_error("conv3d_rows8_score: need labels, partials and out8");
    return CVIT_ERR_INVALID;
  }
  CrArgs a;
  a.w_img = static_cast<const __nv_bfloat16*>(w_img);
  a.bias = bias;
  a.out = nullptr;
  a.aux = nullptr;
  a.db = nullptr;
  a.logits = nullptr;
  a.probs = nullptr;
  a.D = (int)D;
  a.H = (int)H;
  a.W = (int)W;
  a.act = 0;
  a.labels = labels;
  a.partials = partials;
  a.thr = threshold;
  return rows8_launch(x, a, R8_SCORE, (cudaStream_t)stream, out8);
}
