// C-ABI launchers for the tcgen05 GEMM family (ViT linears, patch embed, head 1x1x1 / 3x3x3 /
// transposed convolutions). See include/cryovit_b200.h for the contracts.
#include <string.h>

#include "gemm_tcgen05.cuh"
#include "tmap.h"

namespace cvit {

// 1 = large plain-rows GEMMs with 256-wide N tiles run as CTA pairs (tcgen05 cta_group::2); 0 = single-CTA kernel
// everywhere. Process-wide switch for A/B measurements (tools/kernel_probe.py); the default is pairs.
static int g_gemm_pair = 1;

template <int BN, int EPI, int AMODE, int KSPAN, bool PAIR = false, int SUB = 1, int OPK = OPK_F16>
static int launch_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmArgs& args, int num_tiles,
                       cudaStream_t stream) {
  using Cfg = GemmCfg<BN, KSPAN, PAIR, SUB>;
  auto kern = gemm_tcgen05_kernel<BN, EPI, AMODE, KSPAN, PAIR, SUB, OPK>;
  static bool configured = false;  // per instantiation; attribute is per function, setting twice is harmless
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) {
      set_error("cudaFuncSetAttribute(smem=%d): %s", Cfg::SMEM_BYTES, cudaGetErrorString(e));
      return CVIT_ERR_CUDA;
    }
    configured = true;
  }
  if (PAIR) {
    // num_tiles counts 256-row pair tiles; one cluster of two CTAs per TPC
    int pairs = num_sms() / 2;
    if (pairs > num_tiles) pairs = num_tiles;
    if (pairs < 1) return CVIT_OK;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(2 * pairs);
    cfg.blockDim = dim3(GEMM_THREADS);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, tmA, tmB, args);
    if (e != cudaSuccess) {
      set_error("gemm_tcgen05_kernel<pair>: %s", cudaGetErrorString(e));
      return CVIT_ERR_CUDA;
    }
    return check_launch("gemm_tcgen05_kernel<pair>");
  }
  int grid = num_sms();
  if (grid > num_tiles) grid = num_tiles;
  if (grid < 1) return CVIT_OK;
  kern<<<grid, GEMM_THREADS, Cfg::SMEM_BYTES, stream>>>(tmA, tmB, args);
  return check_launch("gemm_tcgen05_kernel");
}

static int make_tmap_rows(CUtensorMap* tm, const void* base, int64_t rows, int64_t K, int64_t ld, int box_rows,
                          int kspan, TmapDtype dt = TmapDtype::BF16) {
  const int esz = dt == TmapDtype::F32 ? 4 : 2;
  uint64_t dims[2] = {(uint64_t)K, (uint64_t)rows};
  uint64_t strides[2] = {0, (uint64_t)ld * esz};
  uint32_t box[2] = {(uint32_t)(kspan / esz), (uint32_t)box_rows};
  return encode_tmap(tm, dt, 2, base, dims, strides, box, kspan);
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

#define CVIT_GEMM_CASE(BN_, EPI_, AMODE_, KSPAN_)                                     \
  if (bn == BN_ && epi == EPI_ && kspan == KSPAN_)                                    \
    return launch_gemm<BN_, EPI_, AMODE_, KSPAN_>(tmA, tmB, args, num_tiles, stream);
// tall tiles (SUB_ consecutive 128-row blocks per pipeline stage) for single-K-chunk GEMMs with many rows
#define CVIT_GEMM_TALL_CASE(BN_, EPI_, KSPAN_, SUB_)                                                     \
  if (bn == BN_ && epi == EPI_ && kspan == KSPAN_ && K <= KSPAN_ / 2 && M >= 8 * SUB_ * GEMM_BM)         \
    return launch_gemm<BN_, EPI_, AMODE_ROWS, KSPAN_, false, SUB_>(tmA, tmB, args, (int)((M + SUB_ * GEMM_BM - 1) / (SUB_ * GEMM_BM)) * (int)(N / bn), stream);
#define CVIT_GEMM_PAIR_CASE(EPI_)                                                     \
  if (pair && epi == EPI_)                                                            \
    return launch_gemm<256, EPI_, AMODE_ROWS, 128, true>(tmA, tmB, args, num_tiles, stream);
// TF32 operands (fp32 containers, 32 values per 128-byte swizzle span): the ViT linears and the patch embedding
#define CVIT_GEMM_TF32_CASE(BN_, EPI_)                                                \
  if (bn == BN_ && epi == EPI_)                                                       \
    return launch_gemm<BN_, EPI_, AMODE_ROWS, 128, false, 1, OPK_TF32>(tmA, tmB, args, num_tiles, stream);
#define CVIT_GEMM_TF32_PAIR_CASE(EPI_)                                                \
  if (pair && epi == EPI_)                                                            \
    return launch_gemm<256, EPI_, AMODE_ROWS, 128, true, 1, OPK_TF32>(tmA, tmB, args, num_tiles, stream);

// [M,K] x [N,K]^T with TF32 operands: K and lda in fp32 elements (multiples of 4, K >= 32: one 128-byte span per stage).
static int gemm_rows_tf32(const void* A, int64_t lda, const void* B, GemmArgs args, int epi, cudaStream_t stream) {
  const int64_t M = args.M, N = args.N, K = args.K;
  if (!A || !B || !args.out || !aligned16(A) || !aligned16(B) || !aligned16(args.out) || (lda % 4) != 0 || (K % 4) != 0 || K < 32) {
    set_error("gemm tf32: null/unaligned operand (A,B,out need 16B alignment; lda and K multiples of 4, K >= 32)");
    return CVIT_ERR_INVALID;
  }
  const int bn = (epi == EPI_BIAS_SWIGLU) ? ((N % 256 == 0) ? 256 : 0) : (N % 256 == 0) ? 256 : (N % 128 == 0) ? 128 : 0;
  if (bn == 0) {
    set_error("gemm tf32: N=%lld not tileable for epilogue %d (multiple of 128; 256 for SwiGLU)", (long long)N, epi);
    return CVIT_ERR_UNSUPPORTED;
  }
  CUtensorMap tmA, tmB;
  int rc = make_tmap_rows(&tmA, A, M, K, lda, GEMM_BM, 128, TmapDtype::F32);
  if (rc) return rc;
  const bool pair = g_gemm_pair && bn == 256 && M > GEMM_BM && epi != EPI_PATCH_EMBED;
  rc = make_tmap_rows(&tmB, B, N, K, K, pair ? bn / 2 : bn, 128, TmapDtype::F32);
  if (rc) return rc;
  const int bm = pair ? 2 * GEMM_BM : GEMM_BM;
  const int num_tiles = (int)(((M + bm - 1) / bm) * (N / bn));
  CVIT_GEMM_TF32_PAIR_CASE(EPI_BIAS)
  CVIT_GEMM_TF32_PAIR_CASE(EPI_BIAS_GELU)
  CVIT_GEMM_TF32_PAIR_CASE(EPI_BIAS_SWIGLU)
  CVIT_GEMM_TF32_PAIR_CASE(EPI_SCALE_RESIDUAL)
  CVIT_GEMM_TF32_CASE(256, EPI_BIAS)
  CVIT_GEMM_TF32_CASE(128, EPI_BIAS)
  CVIT_GEMM_TF32_CASE(256, EPI_BIAS_GELU)
  CVIT_GEMM_TF32_CASE(128, EPI_BIAS_GELU)
  CVIT_GEMM_TF32_CASE(256, EPI_BIAS_SWIGLU)
  CVIT_GEMM_TF32_CASE(256, EPI_SCALE_RESIDUAL)
  CVIT_GEMM_TF32_CASE(128, EPI_SCALE_RESIDUAL)
  CVIT_GEMM_TF32_CASE(256, EPI_PATCH_EMBED)
  CVIT_GEMM_TF32_CASE(128, EPI_PATCH_EMBED)
  set_error("gemm tf32: no kernel instantiated for BN=%d epilogue=%d", bn, epi);
  return CVIT_ERR_UNSUPPORTED;
}

// Plain [M,K] x [N,K]^T GEMM with a fused epilogue.
static int gemm_rows(const void* A, int64_t lda, const void* B, GemmArgs args, int epi, cudaStream_t stream) {
  const int64_t M = args.M, N = args.N, K = args.K;
  if (M <= 0 || N <= 0 || K <= 0) {
    set_error("gemm: non-positive dimension M=%lld N=%lld K=%lld", (long long)M, (long long)N, (long long)K);
    return CVIT_ERR_INVALID;
  }
  if (args.fmt & GEMM_FMT_OPERANDS_TF32) return gemm_rows_tf32(A, lda, B, args, epi, stream);
  if (!A || !B || !args.out || !aligned16(A) || !aligned16(B) || !aligned16(args.out) || (lda % 8) != 0 || (K % 8) != 0) {
    set_error("gemm: null/unaligned operand (A,B,out need 16B alignment; lda and K multiples of 8)");
    return CVIT_ERR_INVALID;
  }
  int kspan = K >= 64 ? 128 : K >= 32 ? 64 : 32;
  if (K < 64 && (K != 32 && K != 16)) {
    set_error("gemm: K=%lld unsupported (need K>=64, or K in {16,32})", (long long)K);
    return CVIT_ERR_UNSUPPORTED;
  }
  int bn;
  if (epi == EPI_BIAS_SWIGLU) bn = (N % 256 == 0) ? 256 : 0;
  else bn = (N % 256 == 0) ? 256 : (N % 128 == 0) ? 128 : (N % 64 == 0) ? 64 : (N % 32 == 0) ? 32 : 0;
  if (bn == 0) {
    set_error("gemm: N=%lld not tileable for epilogue %d", (long long)N, epi);
    return CVIT_ERR_UNSUPPORTED;
  }
  if (kspan != 128 && bn > 128) bn = 128;
  CUtensorMap tmA, tmB;
  const TmapDtype dt = (args.fmt & GEMM_FMT_OPERANDS_F16) ? TmapDtype::F16 : TmapDtype::BF16;
  int rc = make_tmap_rows(&tmA, A, M, K, lda, GEMM_BM, kspan, dt);
  if (rc) return rc;
  // CTA pairs (256 x 256 output tile per TPC) whenever there is more than one 128-row tile to share a B tile over
  const bool pair = g_gemm_pair && bn == 256 && kspan == 128 && M > GEMM_BM &&
                    (epi == EPI_BIAS || epi == EPI_BIAS_GELU || epi == EPI_BIAS_SWIGLU || epi == EPI_SCALE_RESIDUAL);
  rc = make_tmap_rows(&tmB, B, N, K, K, pair ? bn / 2 : bn, kspan, dt);
  if (rc) return rc;
  const int bm = pair ? 2 * GEMM_BM : GEMM_BM;
  const int num_tiles = (int)(((M + bm - 1) / bm) * (N / bn));
  CVIT_GEMM_TALL_CASE(32, EPI_CONVT_GELU, 32, 8)    // ConvTranspose 16 -> 8 (K = 16, N = 32)
  CVIT_GEMM_TALL_CASE(128, EPI_CONVT_GELU, 64, 2)   // ConvTranspose 32 -> 32 (K = 32, N = 128)
  CVIT_GEMM_TALL_CASE(128, EPI_CONVT_GELU, 128, 2)  // ConvTranspose 64 -> 32 (K = 64, N = 128)
  CVIT_GEMM_PAIR_CASE(EPI_BIAS)
  CVIT_GEMM_PAIR_CASE(EPI_BIAS_GELU)
  CVIT_GEMM_PAIR_CASE(EPI_BIAS_SWIGLU)
  CVIT_GEMM_PAIR_CASE(EPI_SCALE_RESIDUAL)
  CVIT_GEMM_CASE(256, EPI_BIAS, AMODE_ROWS, 128)
  CVIT_GEMM_CASE(128, EPI_BIAS, AMODE_ROWS, 128)
  CVIT_GEMM_CASE(64, EPI_BIAS, AMODE_ROWS, 128)   // transposed-convolution input gradients (training)
  CVIT_GEMM_CASE(32, EPI_BIAS, AMODE_ROWS, 128)
  CVIT_GEMM_CASE(32, EPI_BIAS, AMODE_ROWS, 64)
  CVIT_GEMM_CASE(256, EPI_BIAS_GELU, AMODE_ROWS, 128)
  CVIT_GEMM_CASE(128, EPI_BIAS_GELU, AMODE_ROWS, 128)
  CVIT_GEMM_CASE(256, EPI_BIAS_SWIGLU, AMODE_ROWS, 128)
  CVIT_GEMM_CASE(256, EPI_SCALE_RESIDUAL, AMODE_ROWS, 128)
  CVIT_GEMM_CASE(128, EPI_SCALE_RESIDUAL, AMODE_ROWS, 128)
  CVIT_GEMM_CASE(256, EPI_PATCH_EMBED, AMODE_ROWS, 128)
  CVIT_GEMM_CASE(128, EPI_PATCH_EMBED, AMODE_ROWS, 128)
  CVIT_GEMM_CASE(256, EPI_CONVT_GELU, AMODE_ROWS, 128)
  CVIT_GEMM_CASE(128, EPI_CONVT_GELU, AMODE_ROWS, 128)
  CVIT_GEMM_CASE(128, EPI_CONVT_GELU, AMODE_ROWS, 64)
  CVIT_GEMM_CASE(32, EPI_CONVT_GELU, AMODE_ROWS, 32)
  set_error("gemm: no kernel instantiated for BN=%d epilogue=%d kspan=%d", bn, epi, kspan);
  return CVIT_ERR_UNSUPPORTED;
}

// out[M,N] = At[K,M]^T x B[N,K]^T + bias (+ GELU): A is read from its TRANSPOSED storage (M contiguous) as an MN-major
// operand. fp16 operands (the feature volume on disk is fp16), bf16 output.
static int gemm_rows_mn(const void* At, int64_t ldat, const void* B, GemmArgs args, cudaStream_t stream) {
  const int64_t M = args.M, N = args.N, K = args.K;
  if (M <= 0 || N <= 0 || K <= 0) {
    set_error("gemm_mn: non-positive dimension M=%lld N=%lld K=%lld", (long long)M, (long long)N, (long long)K);
    return CVIT_ERR_INVALID;
  }
  if (!At || !B || !args.out || !aligned16(At) || !aligned16(B) || !aligned16(args.out) || (ldat % 8) != 0 || (K % 8) != 0 || K < 64) {
    set_error("gemm_mn: null/unaligned operand (At,B,out need 16B alignment; ldat and K multiples of 8, K >= 64)");
    return CVIT_ERR_INVALID;
  }
  const int bn = (N % 256 == 0) ? 256 : (N % 128 == 0) ? 128 : 0;
  if (!bn) {
    set_error("gemm_mn: N=%lld must be a multiple of 128", (long long)N);
    return CVIT_ERR_UNSUPPORTED;
  }
  const int epi = EPI_BIAS_GELU, kspan = 128;
  CUtensorMap tmA, tmB;
  {
    uint64_t dims[2] = {(uint64_t)M, (uint64_t)K};
    uint64_t strides[2] = {0, (uint64_t)ldat * 2};
    uint32_t box[2] = {64u, 64u};  // 64 rows (128 bytes, contiguous) x 64 channels
    int rc = encode_tmap(&tmA, TmapDtype::F16, 2, At, dims, strides, box, 128);
    if (rc) return rc;
  }
  const bool pair = g_gemm_pair && bn == 256 && M > GEMM_BM;
  int rc = make_tmap_rows(&tmB, B, N, K, K, pair ? bn / 2 : bn, kspan, TmapDtype::F16);
  if (rc) return rc;
  const int bm = pair ? 2 * GEMM_BM : GEMM_BM;
  const int num_tiles = (int)(((M + bm - 1) / bm) * (N / bn));
  if (pair) return launch_gemm<256, EPI_BIAS_GELU, AMODE_ROWS_MN, 128, true>(tmA, tmB, args, num_tiles, stream);
  CVIT_GEMM_CASE(256, EPI_BIAS_GELU, AMODE_ROWS_MN, 128)
  CVIT_GEMM_CASE(128, EPI_BIAS_GELU, AMODE_ROWS_MN, 128)
  set_error("gemm_mn: no kernel instantiated for BN=%d", bn);
  return CVIT_ERR_UNSUPPORTED;
}

// 3x3x3 depth-dilated "same" convolution over a channels-last bf16 volume, + bias + GELU.
static int conv3_rows(const void* x, const void* w, GemmArgs args, cudaStream_t stream) {
  const int D = args.D, H = args.H, W = args.W, Cin = args.K, Cout = args.N;
  if (D <= 0 || H <= 0 || W <= 0 || Cin <= 0 || Cout <= 0 || args.dil <= 0) {
    set_error("conv3: bad geometry D=%d H=%d W=%d Cin=%d Cout=%d dil=%d", D, H, W, Cin, Cout, args.dil);
    return CVIT_ERR_INVALID;
  }
  if (!x || !w || !args.out || !aligned16(x) || !aligned16(w) || !aligned16(args.out)) {
    set_error("conv3: null/unaligned operand");
    return CVIT_ERR_INVALID;
  }
  int kspan = (Cin % 64 == 0) ? 128 : (Cin == 32) ? 64 : (Cin == 16) ? 32 : 0;
  if (!kspan) {
    set_error("conv3: Cin=%d unsupported (need multiple of 64, or 32, or 16)", Cin);
    return CVIT_ERR_UNSUPPORTED;
  }
  // tile footprint: BW*BH = 128 output voxels of one depth plane; BW = smallest power of two covering
  // min(W,128) (>= 8). Planes that are not a multiple of the footprint get partial border tiles.
  int BW = 8;
  while (BW < W && BW < 128) BW <<= 1;
  const int BH = 128 / BW;
  args.BW = BW;
  args.BH = BH;
  // one N tile for the forward layers' channel counts; wider outputs (input gradients: Cout = the layer's Cin) tile N
  const int bn = (Cout == 192 || Cout == 64 || Cout == 32) ? Cout : (Cout % 256 == 0) ? 256 : (Cout % 128 == 0) ? 128 : 0;
  if (!bn) {
    set_error("conv3: Cout=%d unsupported", Cout);
    return CVIT_ERR_UNSUPPORTED;
  }
  const int epi = EPI_BIAS_GELU;
  CUtensorMap tmA, tmB;
  {
    uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)W, (uint64_t)H, (uint64_t)D};
    uint64_t strides[4] = {0, (uint64_t)Cin * 2, (uint64_t)W * Cin * 2, (uint64_t)H * W * Cin * 2};
    uint32_t box[4] = {(uint32_t)(kspan / 2), (uint32_t)BW, (uint32_t)BH, 1u};
    int rc = encode_tmap(&tmA, TmapDtype::BF16, 4, x, dims, strides, box, kspan);
    if (rc) return rc;
  }
  // CTA pairs (two consecutive row tiles of one depth plane share every B tile, half each) for the wide layers: the
  // single-CTA kernel re-fetches the tap's whole weight tile for every 128 voxels and is bound by L2 -> SM traffic
  const int per_plane = ((H + BH - 1) / BH) * ((W + BW - 1) / BW);
  const bool pair = g_gemm_pair && kspan == 128 && (bn == 192 || bn == 256) && (per_plane % 2) == 0;
  int rc = make_tmap_rows(&tmB, w, (int64_t)27 * Cout, Cin, Cin, pair ? bn / 2 : bn, kspan);
  if (rc) return rc;
  const int num_tiles = D * per_plane * (Cout / bn);
  if (pair && bn == 192) return launch_gemm<192, EPI_BIAS_GELU, AMODE_CONV3, 128, true>(tmA, tmB, args, num_tiles / 2, stream);
  if (pair && bn == 256) return launch_gemm<256, EPI_BIAS_GELU, AMODE_CONV3, 128, true>(tmA, tmB, args, num_tiles / 2, stream);
  CVIT_GEMM_CASE(256, EPI_BIAS_GELU, AMODE_CONV3, 128)
  CVIT_GEMM_CASE(128, EPI_BIAS_GELU, AMODE_CONV3, 128)
  CVIT_GEMM_CASE(192, EPI_BIAS_GELU, AMODE_CONV3, 128)
  CVIT_GEMM_CASE(64, EPI_BIAS_GELU, AMODE_CONV3, 128)
  CVIT_GEMM_CASE(32, EPI_BIAS_GELU, AMODE_CONV3, 64)
  CVIT_GEMM_CASE(32, EPI_BIAS_GELU, AMODE_CONV3, 32)
  set_error("conv3: no kernel instantiated for Cout=%d kspan=%d", bn, kspan);
  return CVIT_ERR_UNSUPPORTED;
}

}  // namespace cvit

using namespace cvit;

static GemmArgs base_args(int64_t M, int64_t N, int64_t K, void* out, int64_t ldo) {
  GemmArgs a;
  memset(&a, 0, sizeof(a));
  a.M = (int)M;
  a.N = (int)N;
  a.K = (int)K;
  a.out = out;
  a.ldo = (int)ldo;
  a.n_valid = (int)N;
  a.act = 1;
  return a;
}

extern "C" {

int64_t cvit_convT_gn_partial_rows(int64_t Cout, int64_t gn_cpg);
int cvit_linear_bias_bf16_nvalid_aux(const void* A, int64_t lda, const void* W, const float* bias, void* out, int64_t ldo,
                                     int64_t M, int64_t N, int64_t K, int64_t n_valid, int act, const void* aux, void* stream);
int cvit_linear_bias_cfirst_f16_aux(const void* At, int64_t ldat, const void* W, const float* bias, void* out, int64_t ldo,
                                    int64_t M, int64_t N, int64_t K, int act, void* aux, void* stream);
int cvit_conv3d_dilated_ndhwc_aux(const void* x, const void* w_taps, const float* bias, void* out, int64_t D,
                                  int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t Cout_valid, int64_t dil,
                                  int act, void* aux, void* stream);
int cvit_convT_1x2x2_ndhwc_aux(const void* x, const void* w_sub, const float* bias4, void* out, int64_t D, int64_t H,
                               int64_t W, int64_t Cin, int64_t Cout, int act, void* aux, void* stream);

int cvit_set_gemm_pair(int enable) {
  const int prev = cvit::g_gemm_pair;
  cvit::g_gemm_pair = enable ? 1 : 0;
  return prev;
}

// tf32_out_f32: with TF32 operands this entry point's epilogue stores TF32-rounded fp32 (GELU / SwiGLU), so
// CVIT_FMT_OUT_F32 is required; otherwise (EPI_BIAS: 16-bit qkv output; the fp32 residual stream) it is refused.
static int check_fmt(int fmt, const char* who, bool tf32_out_f32) {
  if (fmt & ~(GEMM_FMT_OPERANDS_F16 | GEMM_FMT_OUT_F16 | GEMM_FMT_OPERANDS_TF32 | GEMM_FMT_OUT_F32)) {
    set_error("%s: unknown format flags 0x%x", who, fmt);
    return CVIT_ERR_INVALID;
  }
  const bool tf32 = (fmt & GEMM_FMT_OPERANDS_TF32) != 0, f32 = (fmt & GEMM_FMT_OUT_F32) != 0;
  // instantiated: 16-bit operands with 16-bit outputs; TF32 operands with fp32 GELU / SwiGLU output or 16-bit EPI_BIAS
  // output. Everything else is refused rather than run in some other format.
  if ((tf32 && (fmt & GEMM_FMT_OPERANDS_F16)) || (f32 && !tf32) || (tf32 && f32 != tf32_out_f32) ||
      (f32 && (fmt & GEMM_FMT_OUT_F16))) {
    set_error("%s: format flags 0x%x are not instantiated (TF32 operands need %s)", who, fmt,
              tf32_out_f32 ? "CVIT_FMT_OUT_F32 and no fp16 flag" : "no CVIT_FMT_OUT_F32 and no fp16 operands");
    return CVIT_ERR_UNSUPPORTED;
  }
  return CVIT_OK;
}

int cvit_linear_bias_fmt(const void* A, int64_t lda, const void* W, const float* bias, void* out, int64_t ldo,
                         int64_t M, int64_t N, int64_t K, int gelu, int fmt, void* stream) {
  if (!bias) { set_error("linear_bias: bias is required"); return CVIT_ERR_INVALID; }
  if (int rc = check_fmt(fmt, "linear_bias", gelu != 0)) return rc;
  GemmArgs a = base_args(M, N, K, out, ldo);
  a.bias = bias;
  a.fmt = fmt;
  return gemm_rows(A, lda, W, a, gelu ? EPI_BIAS_GELU : EPI_BIAS, (cudaStream_t)stream);
}

int cvit_linear_bias_bf16(const void* A, int64_t lda, const void* W, const float* bias, void* out, int64_t ldo,
                          int64_t M, int64_t N, int64_t K, int gelu, void* stream) {
  return cvit_linear_bias_fmt(A, lda, W, bias, out, ldo, M, N, K, gelu, 0, stream);
}

// Same as cvit_linear_bias_bf16 for an output narrower than the (zero-row-padded) weight: columns >= n_valid are
// computed but not stored, ldo is the true row pitch (transposed-convolution input gradient with 16 channels).
int cvit_linear_bias_bf16_nvalid(const void* A, int64_t lda, const void* W, const float* bias, void* out, int64_t ldo,
                                 int64_t M, int64_t N, int64_t K, int64_t n_valid, void* stream) {
  return cvit_linear_bias_bf16_nvalid_aux(A, lda, W, bias, out, ldo, M, N, K, n_valid, 0, nullptr, stream);
}

// act = 0: the plain entry point; act = 3 (ACT_GELU_GRAD): out = (A W^T + bias) * gelu'(aux), aux bf16 [M, n_valid] with
// row pitch ldo -- the transposed convolution's input gradient handed on as the gradient of the pre-activation below it.
int cvit_linear_bias_bf16_nvalid_aux(const void* A, int64_t lda, const void* W, const float* bias, void* out, int64_t ldo,
                                     int64_t M, int64_t N, int64_t K, int64_t n_valid, int act, const void* aux, void* stream) {
  if (!bias) { set_error("linear_bias: bias is required"); return CVIT_ERR_INVALID; }
  if ((act != ACT_NONE && act != ACT_GELU_GRAD) || (act == ACT_GELU_GRAD && (!aux || (reinterpret_cast<uintptr_t>(aux) & 7u)))) {
    set_error("linear_bias_nvalid_aux: act must be 0 or 3 (with an 8-byte aligned aux)");
    return CVIT_ERR_INVALID;
  }
  GemmArgs a = base_args(M, N, K, out, ldo);
  a.bias = bias;
  a.n_valid = (int)n_valid;
  a.act = act;
  a.aux = const_cast<void*>(aux);
  return gemm_rows(A, lda, W, a, EPI_BIAS, (cudaStream_t)stream);
}

static int check_act_aux(const char* who, int act, const void* aux, bool grad_ok) {
  const bool known = act == ACT_NONE || act == ACT_GELU || act == ACT_DUAL || (grad_ok && act == ACT_GELU_GRAD);
  if (!known || ((act == ACT_DUAL || act == ACT_GELU_GRAD) && (!aux || (reinterpret_cast<uintptr_t>(aux) & 15u)))) {
    set_error("%s: act=%d unsupported here, or aux missing / not 16-byte aligned (0 none, 1 GELU, 2 out=z aux=gelu(z)%s)", who, act,
              grad_ok ? ", 3 out=y*gelu'(aux)" : "");
    return CVIT_ERR_INVALID;
  }
  return CVIT_OK;
}

int cvit_linear_bias_cfirst_f16(const void* At, int64_t ldat, const void* W, const float* bias, void* out, int64_t ldo,
                                int64_t M, int64_t N, int64_t K, int gelu, void* stream) {
  return cvit_linear_bias_cfirst_f16_aux(At, ldat, W, bias, out, ldo, M, N, K, gelu ? 1 : 0, nullptr, stream);
}

int cvit_linear_bias_cfirst_f16_aux(const void* At, int64_t ldat, const void* W, const float* bias, void* out, int64_t ldo,
                                    int64_t M, int64_t N, int64_t K, int act, void* aux, void* stream) {
  if (!bias) { set_error("linear_bias_cfirst: bias is required"); return CVIT_ERR_INVALID; }
  if (int rc = check_act_aux("linear_bias_cfirst", act, aux, false)) return rc;
  GemmArgs a = base_args(M, N, K, out, ldo);
  a.bias = bias;
  a.act = act;
  a.aux = aux;
  a.fmt = GEMM_FMT_OPERANDS_F16;
  return gemm_rows_mn(At, ldat, W, a, (cudaStream_t)stream);
}

// GroupNorm-producer variants (see GemmArgs::gn_partials): same GEMM, plus per-(32-row block, group) statistics.
static int check_gn(const float* partials, int64_t cpg, int64_t N) {
  if (!partials || (cpg != 4 && cpg != 8) || (N % 32) != 0 || (reinterpret_cast<uintptr_t>(partials) & 7u)) {
    set_error("gn producer: partials must be a non-null 8-byte aligned buffer, channels per group 4 or 8 (got %lld)", (long long)cpg);
    return CVIT_ERR_INVALID;
  }
  return CVIT_OK;
}

int cvit_linear_bias_cfirst_f16_gn(const void* At, int64_t ldat, const void* W, const float* bias, void* out, int64_t ldo,
                                   int64_t M, int64_t N, int64_t K, int gelu, float* gn_partials, int64_t gn_cpg, void* stream) {
  if (!bias) { set_error("linear_bias_cfirst: bias is required"); return CVIT_ERR_INVALID; }
  if (int rc = check_gn(gn_partials, gn_cpg, N)) return rc;
  GemmArgs a = base_args(M, N, K, out, ldo);
  a.bias = bias;
  a.act = gelu ? 1 : 0;
  a.fmt = GEMM_FMT_OPERANDS_F16;
  a.gn_partials = gn_partials;
  a.gn_cpg = (int)gn_cpg;
  return gemm_rows_mn(At, ldat, W, a, (cudaStream_t)stream);
}

int cvit_linear_bias_gelu_bf16_gn(const void* A, int64_t lda, const void* W, const float* bias, void* out, int64_t ldo,
                                  int64_t M, int64_t N, int64_t K, float* gn_partials, int64_t gn_cpg, void* stream) {
  if (!bias) { set_error("linear_bias: bias is required"); return CVIT_ERR_INVALID; }
  if (int rc = check_gn(gn_partials, gn_cpg, N)) return rc;
  GemmArgs a = base_args(M, N, K, out, ldo);
  a.bias = bias;
  a.gn_partials = gn_partials;
  a.gn_cpg = (int)gn_cpg;
  return gemm_rows(A, lda, W, a, EPI_BIAS_GELU, (cudaStream_t)stream);
}

int cvit_linear_swiglu_fmt(const void* A, int64_t lda, const void* W12i, const float* bias12i, void* out,
                           int64_t ldo, int64_t M, int64_t N2, int64_t K, int fmt, void* stream) {
  if (!bias12i) { set_error("linear_swiglu: bias is required"); return CVIT_ERR_INVALID; }
  if (int rc = check_fmt(fmt, "linear_swiglu", true)) return rc;
  GemmArgs a = base_args(M, N2, K, out, ldo);
  a.bias = bias12i;
  a.fmt = fmt;
  return gemm_rows(A, lda, W12i, a, EPI_BIAS_SWIGLU, (cudaStream_t)stream);
}

int cvit_linear_swiglu_bf16(const void* A, int64_t lda, const void* W12i, const float* bias12i, void* out,
                            int64_t ldo, int64_t M, int64_t N2, int64_t K, void* stream) {
  return cvit_linear_swiglu_fmt(A, lda, W12i, bias12i, out, ldo, M, N2, K, 0, stream);
}

int cvit_linear_scale_residual_fmt(const void* A, int64_t lda, const void* W, const float* bias, const float* gamma,
                                   float* x, int64_t ldx, int64_t M, int64_t N, int64_t K, int fmt, void* stream) {
  if (!bias || !gamma) { set_error("linear_scale_residual: bias and gamma are required"); return CVIT_ERR_INVALID; }
  if (int rc = check_fmt(fmt & ~GEMM_FMT_OUT_F16, "linear_scale_residual", false)) return rc;
  GemmArgs a = base_args(M, N, K, x, ldx);
  a.bias = bias;
  a.gamma = gamma;
  a.fmt = fmt & (GEMM_FMT_OPERANDS_F16 | GEMM_FMT_OPERANDS_TF32);
  return gemm_rows(A, lda, W, a, EPI_SCALE_RESIDUAL, (cudaStream_t)stream);
}

int cvit_linear_scale_residual_f32(const void* A, int64_t lda, const void* W, const float* bias, const float* gamma,
                                   float* x, int64_t ldx, int64_t M, int64_t N, int64_t K, void* stream) {
  return cvit_linear_scale_residual_fmt(A, lda, W, bias, gamma, x, ldx, M, N, K, 0, stream);
}

int cvit_patch_embed_gemm_fmt(const void* patches, int64_t lda, const void* W, const float* pos_bias_table, float* x,
                              int64_t ldx, int64_t n_slices, int64_t n_patches, int64_t tokens_per_slice,
                              int64_t first_patch_token, int64_t N, int64_t K, int fmt, void* stream);

int cvit_patch_embed_gemm(const void* patches, int64_t lda, const void* W, const float* pos_bias_table, float* x,
                          int64_t ldx, int64_t n_slices, int64_t n_patches, int64_t tokens_per_slice,
                          int64_t first_patch_token, int64_t N, int64_t K, void* stream) {
  return cvit_patch_embed_gemm_fmt(patches, lda, W, pos_bias_table, x, ldx, n_slices, n_patches, tokens_per_slice,
                                   first_patch_token, N, K, 0, stream);
}

int cvit_patch_embed_gemm_fmt(const void* patches, int64_t lda, const void* W, const float* pos_bias_table, float* x,
                              int64_t ldx, int64_t n_slices, int64_t n_patches, int64_t tokens_per_slice,
                              int64_t first_patch_token, int64_t N, int64_t K, int fmt, void* stream) {
  if (!pos_bias_table) { set_error("patch_embed: table is required"); return CVIT_ERR_INVALID; }
  if (fmt != 0 && fmt != GEMM_FMT_OPERANDS_TF32) {
    set_error("patch_embed: format flags 0x%x are not instantiated (0: bf16 patches and weight, CVIT_FMT_OPERANDS_TF32)", fmt);
    return CVIT_ERR_UNSUPPORTED;
  }
  GemmArgs a = base_args(n_slices * n_patches, N, K, x, ldx);
  a.fmt = fmt;
  a.table = pos_bias_table;
  a.pe_np = (int)n_patches;
  a.pe_tokens = (int)tokens_per_slice;
  a.pe_offset = (int)first_patch_token;
  return gemm_rows(patches, lda, W, a, EPI_PATCH_EMBED, (cudaStream_t)stream);
}

int cvit_conv3d_dilated_ndhwc_act(const void* x, const void* w_taps, const float* bias, void* out, int64_t D,
                                  int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t Cout_valid, int64_t dil,
                                  int act, void* stream);

int cvit_conv3d_dilated_ndhwc(const void* x, const void* w_taps, const float* bias, void* out, int64_t D,
                              int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t Cout_valid, int64_t dil,
                              void* stream) {
  return cvit_conv3d_dilated_ndhwc_act(x, w_taps, bias, out, D, H, W, Cin, Cout, Cout_valid, dil, 1, stream);
}

int cvit_conv3d_dilated_ndhwc_act(const void* x, const void* w_taps, const float* bias, void* out, int64_t D,
                                  int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t Cout_valid, int64_t dil,
                                  int act, void* stream) {
  return cvit_conv3d_dilated_ndhwc_aux(x, w_taps, bias, out, D, H, W, Cin, Cout, Cout_valid, dil, act ? 1 : 0, nullptr, stream);
}

int cvit_conv3d_dilated_ndhwc_aux(const void* x, const void* w_taps, const float* bias, void* out, int64_t D,
                                  int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t Cout_valid, int64_t dil,
                                  int act, void* aux, void* stream) {
  if (!bias) { set_error("conv3d: bias is required"); return CVIT_ERR_INVALID; }
  if (int rc = check_act_aux("conv3d_dilated", act, aux, true)) return rc;
  GemmArgs a = base_args(D * H * W, Cout, Cin, out, Cout_valid);
  a.aux = aux;
  a.bias = bias;
  a.D = (int)D;
  a.H = (int)H;
  a.W = (int)W;
  a.dil = (int)dil;
  a.n_valid = (int)Cout_valid;
  a.act = act;
  return conv3_rows(x, w_taps, a, (cudaStream_t)stream);
}

int cvit_convT_1x2x2_ndhwc_act(const void* x, const void* w_sub, const float* bias4, void* out, int64_t D, int64_t H,
                               int64_t W, int64_t Cin, int64_t Cout, int act, void* stream);

int cvit_convT_1x2x2_ndhwc(const void* x, const void* w_sub, const float* bias4, void* out, int64_t D, int64_t H,
                           int64_t W, int64_t Cin, int64_t Cout, void* stream) {
  return cvit_convT_1x2x2_ndhwc_act(x, w_sub, bias4, out, D, H, W, Cin, Cout, 1, stream);
}

int cvit_convT_1x2x2_ndhwc_act(const void* x, const void* w_sub, const float* bias4, void* out, int64_t D, int64_t H,
                               int64_t W, int64_t Cin, int64_t Cout, int act, void* stream) {
  return cvit_convT_1x2x2_ndhwc_aux(x, w_sub, bias4, out, D, H, W, Cin, Cout, act ? 1 : 0, nullptr, stream);
}

int cvit_convT_1x2x2_ndhwc_aux(const void* x, const void* w_sub, const float* bias4, void* out, int64_t D, int64_t H,
                               int64_t W, int64_t Cin, int64_t Cout, int act, void* aux, void* stream) {
  if (!bias4) { set_error("convT: bias is required"); return CVIT_ERR_INVALID; }
  if (int rc = check_act_aux("convT", act, aux, false)) return rc;
  GemmArgs a = base_args(D * H * W, 4 * Cout, Cin, out, Cout);
  a.aux = aux;
  a.bias = bias4;
  a.H = (int)H;
  a.W = (int)W;
  a.c3 = (int)Cout;
  a.act = act;
  return gemm_rows(x, Cin, w_sub, a, EPI_CONVT_GELU, (cudaStream_t)stream);
}

int cvit_convT_1x2x2_ndhwc_gn(const void* x, const void* w_sub, const float* bias4, void* out, int64_t D, int64_t H,
                              int64_t W, int64_t Cin, int64_t Cout, float* gn_partials, int64_t gn_cpg, void* stream) {
  if (!bias4) { set_error("convT: bias is required"); return CVIT_ERR_INVALID; }
  if (int rc = check_gn(gn_partials, gn_cpg, 4 * Cout)) return rc;
  if (Cout % gn_cpg) { set_error("convT_gn: %lld channels do not split into groups of %lld", (long long)Cout, (long long)gn_cpg); return CVIT_ERR_INVALID; }
  GemmArgs a = base_args(D * H * W, 4 * Cout, Cin, out, Cout);
  a.bias = bias4;
  a.H = (int)H;
  a.W = (int)W;
  a.c3 = (int)Cout;
  a.act = 1;
  a.gn_partials = gn_partials;
  a.gn_cpg = (int)gn_cpg;
  if (cvit_convT_gn_partial_rows(Cout, gn_cpg) > 0) {
    // register-accumulated statistics: one partials row per epilogue thread of every CTA that could run; rows of CTAs that
    // are not launched (fewer tiles than SMs) must read as zero
    a.gn_direct = 1;
    cudaError_t e = cudaMemsetAsync(gn_partials, 0, (size_t)cvit_convT_gn_partial_rows(Cout, gn_cpg) * 8 * 2 * sizeof(float), (cudaStream_t)stream);
    if (e != cudaSuccess) { set_error("convT_gn: cudaMemsetAsync: %s", cudaGetErrorString(e)); return CVIT_ERR_CUDA; }
  }
  return gemm_rows(x, Cin, w_sub, a, EPI_CONVT_GELU, (cudaStream_t)stream);
}

// Rows of the statistics buffer cvit_convT_1x2x2_ndhwc_gn writes for this layer when it keeps the group sums in registers
// (32 output channels in groups of 4): [rows][8 groups][2] fp32, to be folded with rows32 = rows, partial columns = 8.
// 0: the per-32-voxel layout of the other producers ([ceil(voxels / 32)][4 Cout / cpg][2]).
int64_t cvit_convT_gn_partial_rows(int64_t Cout, int64_t gn_cpg) {
  return (CONVT_DIRECT && Cout == 32 && gn_cpg == 4) ? (int64_t)num_sms() * 256 : 0;
}

// Consumer variant (see GemmArgs::bias_table): the convolution after a folded GroupNorm.
int cvit_conv3d_dilated_ndhwc_tab(const void* x, const void* w_taps, const float* bias_table, void* out, int64_t D,
                                  int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t Cout_valid, int64_t dil,
                                  void* stream) {
  if (!bias_table || (reinterpret_cast<uintptr_t>(bias_table) & 15u)) { set_error("conv3d_tab: a 16-byte aligned bias table is required"); return CVIT_ERR_INVALID; }
  GemmArgs a = base_args(D * H * W, Cout, Cin, out, Cout_valid);
  a.bias = bias_table + 63 * Cout;  // the all-taps-inside row; the kernel swaps in the voxel's own row
  a.bias_table = bias_table;
  a.D = (int)D;
  a.H = (int)H;
  a.W = (int)W;
  a.dil = (int)dil;
  a.n_valid = (int)Cout_valid;
  a.act = 1;
  return conv3_rows(x, w_taps, a, (cudaStream_t)stream);
}

}  // extern "C"
