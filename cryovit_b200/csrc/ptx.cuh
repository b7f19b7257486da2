// Thin inline-PTX wrappers for the sm_100a primitives the CryoVIT hot path uses:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM alloc / TMEM load), and
// the legacy warp-level mma.sync + ldmatrix used by the attention kernel.
//
// Everything here is device code; the host-side tensor-map encoder lives in tmap.h.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace cvit {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ----------------------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t tx_bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(tx_bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must trap instead of hanging the GPU (a hung box is a lost box).
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = clock64();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3ffu) == 0 && (clock64() - t0) > 8000000000ll) {
      printf("cvit: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n", blockIdx.x,
             threadIdx.x, bar, parity);
      __trap();
    }
  }
}

// ----------------------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0,
                                            int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4}], [%2];" ::"r"(dst),
      "l"(m), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0,
                                            int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4, %5}], [%2];" ::"r"(dst),
      "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0,
                                            int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4, %5, %6}], [%2];" ::"r"(dst),
      "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0,
                                            int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4, %5, %6, %7}], [%2];" ::"r"(dst),
      "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

// One lane of a converged warp (the same lane every time): tcgen05.mma / commit are issued under this predicate
// so that the surrounding control flow stays warp-uniform and descriptors live in uniform registers.
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .b32 rx;\n"
      ".reg .pred px;\n"
      "elect.sync rx|px, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, px;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ----------------------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tcgen05_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// Whole warp. Writes the TMEM base address (lane<<16 | column) to *dst_smem.
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem) {
  static_assert(NCOLS >= 32 && NCOLS <= 512 && (NCOLS & (NCOLS - 1)) == 0, "TMEM columns: pow2 in [32,512]");
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem),
               "n"(NCOLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS)
               : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same with the A operand read from TMEM (lane = row, 16-bit elements packed two per 32-bit column).
__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrives (count 1) on the mbarrier once every previously issued tcgen05.mma of this thread retired.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread t of the warp gets row (lane base + t).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]),
        "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]),
        "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]),
        "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// Stores: thread t of the warp writes N consecutive 32-bit columns of TMEM lane (lane base + t).
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ----------------------------------------------------------------------------- CTA pair (cta_group::2)
// Two CTAs of a cluster on the two SMs of one TPC share every MMA: each supplies its 128 rows of A and HALF of the
// B tile from its own shared memory, each receives its 128 accumulator rows in its own TMEM. Only the leader (cluster
// rank 0) issues; shared-memory and TMEM offsets must be identical in both CTAs.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> shared::cluster address of the same offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_cluster(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
// TMA load into THIS CTA's shared memory whose completion bytes are signalled on a barrier that may live in the
// peer CTA of the pair (`cluster_bar` is a shared::cluster address).
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* m, uint32_t cluster_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4}], [%2];" ::"r"(dst),
      "l"(m), "r"(cluster_bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(uint32_t dst, const CUtensorMap* m, uint32_t cluster_bar, int c0, int c1,
                                                 int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, "
      "%5, %6}], [%2];" ::"r"(dst),
      "l"(m), "r"(cluster_bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// Executed by the SAME warp index in both CTAs of the pair; both receive the same TMEM address.
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t dst_smem) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "n"(NCOLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
// D[tmem, both CTAs] (+)= A * B over the pair: M = 256 (128 rows per CTA), B's N split half/half; leader thread only.
__device__ __forceinline__ void umma_bf16_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// The CTA-pair form with TF32 operands (see umma_tf32).
__device__ __forceinline__ void umma_tf32_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrives (count 1) on the barrier at this shared-memory offset in BOTH CTAs once the leader's MMAs retired.
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile(
      "{\n"
      ".reg .b16 m;\n"
      "mov.b16 m, 3;\n"
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], m;\n"
      "}\n" ::"r"(bar)
      : "memory");
}

// Shared-memory matrix descriptor for a K-major operand tile whose rows are exactly one swizzle span
// (SWIZZLE_BYTES = 128/64/32 bytes of K per row, rows packed back to back, tile base 1024-aligned).
// Field layout follows cute::UMMA::SmemDescriptor (cute/arch/mma_sm100_desc.hpp): start>>4 @[0,14),
// LBO>>4 @[16,30), SBO>>4 @[32,46), version=1 @[46,48), layout type @[61,64).
template <int SWIZZLE_BYTES>
__device__ __forceinline__ uint64_t umma_smem_desc_kmajor(uint32_t smem_addr) {
  constexpr uint64_t layout = SWIZZLE_BYTES == 128 ? 2ull : SWIZZLE_BYTES == 64 ? 4ull : 6ull;
  constexpr uint64_t sbo = (8ull * SWIZZLE_BYTES) >> 4;  // 8-row core-matrix group stride
  return static_cast<uint64_t>((smem_addr & 0x3ffffu) >> 4) | (1ull << 16) | (sbo << 32) | (1ull << 46) |
         (layout << 61);
}
// MN-major B operand (the contiguous dimension is N, e.g. a V tile [keys][head_dim]) in 128-byte-swizzled rows:
// canonical layout ((8,8,m),(8,k)):((1,8,LBO),(64,SBO)) in elements -- 64 N-elements per 128-byte row, rows are
// consecutive K indices, 8-row groups SBO = 1024 bytes apart (cute/atom/mma_traits_sm100.hpp, make_umma_desc<MN>).
__device__ __forceinline__ uint64_t umma_smem_desc_mnmajor_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
  return static_cast<uint64_t>((smem_addr & 0x3ffffu) >> 4) | (static_cast<uint64_t>((lbo_bytes >> 4) & 0x3fff) << 16) |
         (static_cast<uint64_t>(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// Instruction descriptor, kind::f16, BF16 x BF16 -> FP32, both operands K-major
// (cute::UMMA::InstrDescriptor: c_format @[4,6), a/b_format @[7,10)/[10,13), N>>3 @[17,23), M>>4 @[24,29)).
__host__ __device__ constexpr uint32_t umma_idesc_bf16_f32(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}
// Same with IEEE fp16 operands (a/b_format = 0). Both operands of a kind::f16 MMA must have the SAME 16-bit type on
// sm_100a: a bf16 x fp16 descriptor raises cudaErrorIllegalInstruction (profiles/r01_attention_notes.md).
__host__ __device__ constexpr uint32_t umma_idesc_f16_f32(int M, int N) {
  return (1u << 4) | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}
// format bits that turn umma_idesc_f16_f32 into umma_idesc_bf16_f32
constexpr uint32_t UMMA_IDESC_BF16_BITS = (1u << 7) | (1u << 10);
// Instruction descriptor, kind::tf32, TF32 x TF32 -> FP32, both operands K-major: the same fields as kind::f16 with
// a_format = b_format = 2 (TF32) (PTX ISA, instruction descriptor table for .kind::f16 / .kind::tf32; cute::UMMA::
// UMMAFormat::TF32). Each MMA consumes K = 8 fp32 values = 32 bytes of a K-major row, the same bytes as K = 16 of a
// 16-bit operand, so the shared-memory descriptors and their per-MMA advance do not change.
__host__ __device__ constexpr uint32_t umma_idesc_tf32_f32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}
// D[tmem] (+)= A * B with TF32 operands (fp32 containers; the tensor core reads the upper 19 bits); ONE thread.
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// ----------------------------------------------------------------------------- misc
__device__ __forceinline__ float gelu_erf_exact(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// GELU(erf) = x Phi(x). Two evaluations:
//
// gelu_erf_as (the first one used here; kept as the accuracy reference of tests/test_oracle.py): erf from
// Abramowitz-Stegun 7.1.26, 11 FMA-pipe instructions and two MUFU (rcp, ex2), |error| <= 5e-7 absolute.
//
// gelu_erf (what every epilogue calls): Phi(x) = sigmoid(x q(x^2)) with q an even cubic fitted to logit(Phi(x)) / x --
// the "tanh approximation" 0.5 (1 + tanh(u)) = sigmoid(2u) with one more term and re-fitted coefficients. 7 FMA-pipe
// instructions and the same two MUFU: the head's narrow layers and transposed convolutions are bound by exactly this
// epilogue math (268 M activations per layer at 512 x 512, ~29 instructions per output before). |error| <= 2.6e-5
// absolute over the whole real line and <= 2.1e-4 relative wherever |gelu| >= 0.1 (tests/test_oracle.py::
// test_fast_gelu_formula): a ninth of the 2^-9 rounding step of the bf16 value every consumer stores.
// x^2 is clamped at 36 (the cubic turns over near x^2 = 52); beyond |x| = 6, sigmoid(3.35 |x|) is 0 or 1 to 2e-9.
__device__ __forceinline__ float gelu_erf_as(float x) {
  const float z = fabsf(x) * 0.70710678118654752f;
  const float t = rcp_approx(fmaf(0.3275911f, z, 1.0f));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  p *= t;
  const float e = ex2_approx(z * z * -1.4426950408889634f);
  const float erf_abs = fmaf(-p, e, 1.0f);
  const float h = 0.5f * x;
  return fmaf(h, copysignf(erf_abs, x), h);
}
__device__ __forceinline__ float gelu_erf(float x) {
  constexpr float L2E = 1.4426950408889634f;
  const float x2 = fminf(x * x, 36.0f);
  float q = fmaf(7.030335764e-4f * L2E, x2, -7.401129204e-2f * L2E);   // -log2(e) q(x^2)
  q = fmaf(q, x2, -1.5950157686f * L2E);
  const float e = ex2_approx(q * x);        // exp(-x q): inf for very negative x, then rcp(inf) = 0
  return x * rcp_approx(1.0f + e);
}
// The same for two values at once on the packed fp32 pipe (Blackwell FFMA2 / FMUL2 / FADD2: one issue slot per PAIR);
// the clamp and the two MUFU stay scalar. Bit-identical to two gelu_erf calls (same roundings in the same order).
__device__ __forceinline__ void gelu_erf2(float& a, float& b) {
  constexpr float L2E = 1.4426950408889634f;
  uint64_t x, x2, q, t;
  asm("mov.b64 %0, {%1, %2};" : "=l"(x) : "f"(a), "f"(b));
  asm("mul.rn.f32x2 %0, %1, %1;" : "=l"(x2) : "l"(x));
  float x2a, x2b;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(x2a), "=f"(x2b) : "l"(x2));
  x2a = fminf(x2a, 36.0f);
  x2b = fminf(x2b, 36.0f);
  asm("mov.b64 %0, {%1, %2};" : "=l"(x2) : "f"(x2a), "f"(x2b));
  uint64_t c2, c1, c0, one;
  asm("mov.b64 %0, {%1, %1};" : "=l"(c2) : "f"(7.030335764e-4f * L2E));
  asm("mov.b64 %0, {%1, %1};" : "=l"(c1) : "f"(-7.401129204e-2f * L2E));
  asm("mov.b64 %0, {%1, %1};" : "=l"(c0) : "f"(-1.5950157686f * L2E));
  asm("mov.b64 %0, {%1, %1};" : "=l"(one) : "f"(1.0f));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(q) : "l"(c2), "l"(x2), "l"(c1));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(q) : "l"(q), "l"(x2), "l"(c0));
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(t) : "l"(q), "l"(x));
  float ta, tb;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(ta), "=f"(tb) : "l"(t));
  uint64_t e;
  asm("mov.b64 %0, {%1, %2};" : "=l"(e) : "f"(ex2_approx(ta)), "f"(ex2_approx(tb)));
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(e) : "l"(e), "l"(one));
  float da, db;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(da), "=f"(db) : "l"(e));
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(rcp_approx(da)), "f"(rcp_approx(db)));
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(x), "l"(r));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(r));
}
// d/dz [ 0.5 z (1 + erf(z / sqrt 2)) ] = Phi(z) + z phi(z). erf from Abramowitz-Stegun 7.1.26 (|error| <= 1.5e-7, see
// gelu_erf in ptx.cuh); its exp(-z^2 / 2) is the one phi(z) needs, so the whole derivative costs one ex2 and one rcp.
__device__ __forceinline__ float gelu_grad(float z) {
  const float u = fabsf(z) * 0.70710678118654752f;
  const float t = rcp_approx(fmaf(0.3275911f, u, 1.0f));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  p *= t;
  const float e = ex2_approx(u * u * -1.4426950408889634f);  // exp(-z^2 / 2)
  const float cdf = fmaf(0.5f, copysignf(fmaf(-p, e, 1.0f), z), 0.5f);
  return fmaf(z * 0.3989422804014327f, e, cdf);
}

// Activation modes of the head kernels' epilogues (`act` in the C ABI). Training fuses the element-wise passes into the
// convolutions: ACT_DUAL keeps the pre-activation for the backward pass and hands the activation to the next layer in
// one epilogue; ACT_GELU_GRAD turns an input-gradient convolution into "gradient of the previous pre-activation".
enum { ACT_NONE = 0, ACT_GELU = 1, ACT_DUAL = 2, ACT_GELU_GRAD = 3 };
//   ACT_NONE       out = y
//   ACT_GELU       out = gelu(y)
//   ACT_DUAL       out = y, aux = gelu(y)           (aux: bf16, same shape / indexing as out)
//   ACT_GELU_GRAD  out = y * gelu'(aux)             (aux: the saved pre-activation z of the layer below)
// Pair form used by every epilogue: (a, b) are two neighbouring channels, z2 / a2 point at their packed bf16 pair.
__device__ __forceinline__ uint32_t act_gelu_grad_pair(float a, float b, uint32_t z2) {
  const float z0 = __uint_as_float(z2 << 16), z1 = __uint_as_float(z2 & 0xffff0000u);
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b * gelu_grad(z1)), "f"(a * gelu_grad(z0)));
  return r;
}
// x * sigmoid(x) with ex2.approx + rcp.approx (both ~2^-22 relative error): 4 instructions instead of an IEEE division
__device__ __forceinline__ float silu(float x) { return __fdividef(x, 1.0f + ex2_approx(-1.4426950408889634f * x)); }
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  __half2 v = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
// fp32 -> the nearest TF32 value, ties away from zero (cvt.rna), in an fp32 container with the 13 low mantissa bits
// zero: what a producer stores for a kind::tf32 GEMM, so the tensor core consumes exactly the stored value. The mask
// makes the container's low bits zero whatever the conversion leaves in them.
__device__ __forceinline__ float round_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r & 0xffffe000u);
}
// two fp32 -> one packed pair of the 16-bit operand type (F16: IEEE fp16, else bf16)
template <bool F16>
__device__ __forceinline__ uint32_t pack_16x2(float lo, float hi) {
  return F16 ? pack_f16x2(lo, hi) : pack_bf16x2(lo, hi);
}
// 32-byte store (one full sector per lane; sm_100: STG.256). p must be 32-byte aligned.
__device__ __forceinline__ void st_global_v8(void* p, const uint32_t (&v)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]),
               "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace cvit
