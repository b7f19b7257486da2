// Flash-style self-attention of one ViT slice on tcgen05 / TMEM (head_dim 64, bf16 in/out, fp32 softmax).
// Restates upstream MemEffAttention: softmax(q k^T / 8) v, q,k,v = qkv.reshape(B, N, 3, H, 64) (SURVEY.md K9).
//
// Persistent kernel, one CTA per SM, 512 threads = four warpgroups; registers are re-balanced with setmaxnreg
// (softmax warps hold a whole 128-wide S row). A work item is (slice, head, 256 query rows) = two 128-row query
// tiles A and B that share every K/V tile; items are walked query-pair fastest so co-running CTAs share K/V in L2.
// Barrier phases, the K/V ring and the S/P/O buffers run across items: the tile stream never drains at an item end.
//   warps 0-3   softmax group A, warps 4-7 softmax group B; one thread per query row (TMEM lane = row). The whole
//               128-wide S row is held in registers: row max (3-input FMNMX), lazy rescale (O and l are only rescaled
//               when the max grows by more than 2^8), p = exp2(s*c - m*c) with packed f32x2 FMA/ADD -> bf16 pairs
//               -> TMEM. P(j) is published to the MMA warp only after the loads of S(j+1) were issued, so the TMEM
//               store drain (300-600 cycles when the tensor pipe is busy) is off the critical path.
//   warps 8-11  epilogue: O_g / l -> bf16 -> global, while the softmax warps already run the next item.
//   warp 12     TMA producer: Q_A|Q_B once per item, (K, V) tiles of 128 keys through a 4-stage ring. The tensor map
//               is 3-D (column, token, slice): tokens past the end of a slice are zero-filled, never the next slice.
//   warps 13,14 MMA issuers, one per query tile (whole warp walks the schedule, one elected lane issues):
//                   S_g = Q_g K^T  (SS: K-major operands in 128B-swizzled smem, N = 128 keys)
//                   O_g += P_g V   (TS: P read from TMEM as packed bf16, V tile as an MN-major B operand)
//               Each issues S_g(t+1) as soon as its group has pulled S_g(t) into registers (so the next S is ready
//               before the softmax of the current one ends), then PV_g(t) when P_g(t) is published.
// TMEM (512 columns): S_A [0,128) S_B [128,256) | P_A [256,320) P_B [320,384) | O_A [384,448) O_B [448,512).
// The ragged tail (1029 = 8*128 + 5 keys) runs as an N=16 MMA with the 11 padding keys masked to -inf.
// A slice whose query-tile count is odd ends with an A-only item (group B idles through it).
#include "ptx.cuh"
#include "tmap.h"

namespace cvit {

constexpr int FA_BQ = 128, FA_BK = 128, FA_D = 64;
constexpr int FA_THREADS = 512;
// setmaxnreg budget per scheduler (one warp of each warpgroup): 2 x softmax + epilogue + control <= 512
constexpr int FA_REGS_SOFTMAX = 184, FA_REGS_EPILOGUE = 72, FA_REGS_CONTROL = 72;
constexpr int FA_STAGES = 4;
constexpr int FA_TILE_BYTES = 128 * 128;  // 128 rows x 64 bf16
constexpr int FA_SMEM = (4 + 2 * FA_STAGES) * FA_TILE_BYTES + 4096 /* row sums, maxima */ + 512 /* barriers */ + 1024;
constexpr int FA_TMEM_COLS = 512;
constexpr uint32_t FA_COL_S = 0, FA_COL_P = 256, FA_COL_O = 384;

// Optional per-phase cycle accounting (tools/fa_trace.py builds with -DCVIT_FA_TRACE): every warp accumulates the
// cycles it spends in each phase in registers and dumps the totals once at the end (a timeline of global stores
// proved too intrusive: it moved the phases it was measuring).
#ifdef CVIT_FA_TRACE
__device__ __forceinline__ unsigned long long fa_globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define FA_PROF_DECL uint32_t prof_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}; const unsigned long long prof_t0 = fa_globaltimer(); uint32_t prof_last = clock()
#define FA_PROF(slot) do { const uint32_t now_ = clock(); prof_acc[slot] += now_ - prof_last; prof_last = now_; } while (0)
#define FA_PROF_DUMP(tiles) do { if (args.trace && blockIdx.x < 4 && lane == 0) {                      \
    long long* d_ = args.trace + (blockIdx.x * 16 + warp) * 10;                                        \
    for (int i_ = 0; i_ < 8; ++i_) d_[i_] = prof_acc[i_];                                              \
    d_[8] = (tiles); d_[9] = (long long)(fa_globaltimer() - prof_t0); } } while (0)
#else
#define FA_PROF_DECL do { } while (0)
#define FA_PROF(slot) do { } while (0)
#define FA_PROF_DUMP(tiles) do { } while (0)
#endif
struct FaArgs {
  long long* trace;    // debug accounting (tools/fa_trace.py), normally null
  __nv_bfloat16* out;  // [B*T, C]
  int T, heads, C, slices;
  float scale_log2e;   // head_dim^-0.5 * log2(e)
};

// packed fp32 pairs (Blackwell FFMA2 / FADD2): halves the issue slots of the softmax inner loop
__device__ __forceinline__ uint64_t pack_f32x2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack_f32x2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fma_f32x2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ uint64_t add_f32x2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}

// F16: q/k/v and P are IEEE fp16 instead of bf16 (P <= 2^8 under the lazy rescale, far inside the fp16 range);
// OUT16: the output is stored as IEEE fp16 instead of bf16 (independent of F16: the output only has to match the
// operand type of the projection GEMM that reads it). Everything else is identical.
// OUT32: the output is stored as TF32-rounded fp32 (the A operand of a kind::tf32 projection GEMM); the epilogue
// stores straight from registers (no shared-memory staging), 16 columns per TMEM load so its live registers stay
// within the 16-bit path's under the epilogue's setmaxnreg budget.
template <bool F16, bool OUT16, bool OUT32 = false>
__global__ void __launch_bounds__(FA_THREADS, 1)
attention_tcgen05_kernel(const __grid_constant__ CUtensorMap tmQKV, const FaArgs args) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sQ = smem_base;                                        // [item parity][Q_A | Q_B]: the next item's
                                                                        // query tiles land while this one runs
  const uint32_t sK = smem_base + 4 * FA_TILE_BYTES;                    // FA_STAGES tiles
  const uint32_t sV = smem_base + (4 + FA_STAGES) * FA_TILE_BYTES;      // FA_STAGES tiles
  const uint32_t sL = smem_base + (4 + 2 * FA_STAGES) * FA_TILE_BYTES;  // [item parity][group][sums 128 | maxima 128] fp32
  const uint32_t sBar = sL + 4096;
  const uint32_t bar_q = sBar, bar_q_empty = sBar + 16;   // 2 x 8 each (one per Q buffer)
  const uint32_t bar_kv_full = sBar + 32;                 // FA_STAGES x 8
  const uint32_t bar_kv_empty = sBar + 32 + 8 * FA_STAGES;
  const uint32_t bar_grp = sBar + 32 + 16 * FA_STAGES;    // per group (64 B apart): the seven barriers below
  constexpr uint32_t B_S = 0, B_SFREE = 8, B_P = 16, B_PV = 24, B_OFULL = 32, B_OEMPTY = 40, B_LFULL = 48;
  const uint32_t tmem_slot = bar_grp + 128;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int T = args.T;
  const int n_tiles = (T + FA_BK - 1) / FA_BK;   // K/V tiles per item
  const int n_qt = (T + FA_BQ - 1) / FA_BQ;      // query tiles per (slice, head)
  const int n_pairs = (n_qt + 1) >> 1;
  const int total_items = n_pairs * args.heads * args.slices;
  // K/V tiles are walked ragged-tile-first: the short tile's P is published at once and its PV retires under the
  // first full tile (walked last, the single P buffer would stall the softmax behind PV of the tile before it).
  const bool ragged = (T % FA_BK) != 0;
  auto kv_tile = [&](int j) { return ragged ? (j == 0 ? n_tiles - 1 : j - 1) : j; };
  // Item kinds. PAIRED: query tiles 2p (group A) and 2p+1 (group B). When the query-tile count is odd the last
  // item has a single tile; it is SPLIT between the groups by K/V tile (group g takes the walked tiles j = g mod 2,
  // each with its own running max / sum / O; the epilogue merges the two partial softmaxes) so that it costs half
  // an item instead of a whole one. With a single K/V tile there is nothing to split: SOLO (group A alone).
  enum { PAIRED = 0, SPLIT = 1, SOLO = 2 };
  auto pair_kind = [&](int pair) { return 2 * pair + 1 < n_qt ? PAIRED : n_tiles > 1 ? SPLIT : SOLO; };
  auto item_kind = [&](int item) { return pair_kind(item % n_pairs); };
  // does group g work on walked tile j of an item of this kind?
  auto mine = [&](int kind, int g, int j) { return kind == PAIRED || (kind == SPLIT ? (j & 1) == g : g == 0); };

  // Lazy rescale: O and l follow the running maximum only when it grew by more than 2^FA_RESCALE_LOG2, i.e. stored
  // probabilities reach at most that. fp16 probabilities (max 65504) keep 2^8; bf16 ones have fp32's range, and 2^16
  // makes the kernel's time independent of the score distribution (1.77 -> 1.54 ms on scores with std 2.25, where the
  // 2^8 threshold rescaled on most early tiles; profiles/r02_attention_notes.md).
  constexpr float FA_RESCALE_LOG2 = F16 ? 8.0f : 16.0f;
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQKV);
    for (int b = 0; b < 2; ++b) {
      mbar_init(bar_q + 8 * b, 1);
      mbar_init(bar_q_empty + 8 * b, 2);  // one commit per group (group A commits twice on SOLO items)
    }
    for (int s = 0; s < FA_STAGES; ++s) {
      mbar_init(bar_kv_full + 8 * s, 1);
      mbar_init(bar_kv_empty + 8 * s, 2);
    }
    for (int g = 0; g < 2; ++g) {
      mbar_init(bar_grp + 64 * g + B_S, 1);       // MMA -> softmax: S_g(t) complete
      mbar_init(bar_grp + 64 * g + B_SFREE, 4);   // softmax -> MMA: S_g(t) is in registers, the TMEM tile may be overwritten
      mbar_init(bar_grp + 64 * g + B_P, 4);       // softmax -> MMA: P_g(t) stored
      mbar_init(bar_grp + 64 * g + B_PV, 1);      // MMA -> softmax: PV_g(t) retired (P reusable, O consistent)
      mbar_init(bar_grp + 64 * g + B_OFULL, 1);   // MMA -> epilogue: the item's last PV_g retired, O_g complete
      mbar_init(bar_grp + 64 * g + B_OEMPTY, 4);  // epilogue -> MMA: O_g read out, the next item may overwrite it
      mbar_init(bar_grp + 64 * g + B_LFULL, 4);   // softmax -> epilogue: row sums of the item are in smem
    }
    fence_mbar_init();
  }
  if (warp == 13) tmem_alloc<FA_TMEM_COLS>(tmem_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  if (warp >= 12) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(FA_REGS_CONTROL));
    if (warp == 12) {
      // ------------------------------------------------------------------ TMA producer
      if (lane == 0) {
        uint32_t kv_it = 0, k = 0;
        for (int item = blockIdx.x; item < total_items; item += gridDim.x, ++k) {
          const int pair = item % n_pairs, bh = item / n_pairs;
          const int head = bh % args.heads, slice = bh / args.heads;
          const int cq = head * FA_D, ck = args.C + head * FA_D, cv = 2 * args.C + head * FA_D;
          const uint32_t qb_ = k & 1, sQk = sQ + qb_ * 2 * FA_TILE_BYTES, bq = bar_q + 8 * qb_;
          mbar_wait(bar_q_empty + 8 * qb_, ((k >> 1) & 1) ^ 1u);  // every S MMA of item k-2 has retired
          mbar_arrive_expect_tx(bq, 2 * FA_TILE_BYTES);
          tma_load_3d(sQk, &tmQKV, bq, cq, (2 * pair) * FA_BQ, slice);
          const int qb = item_kind(item) == PAIRED ? 2 * pair + 1 : 2 * pair;  // SPLIT: both groups work on tile 2p
          tma_load_3d(sQk + FA_TILE_BYTES, &tmQKV, bq, cq, qb * FA_BQ, slice);
          for (int j = 0; j < n_tiles; ++j, ++kv_it) {
            const uint32_t s = kv_it % FA_STAGES;
            mbar_wait(bar_kv_empty + 8 * s, ((kv_it / FA_STAGES) & 1) ^ 1u);
            mbar_arrive_expect_tx(bar_kv_full + 8 * s, 2 * FA_TILE_BYTES);
            tma_load_3d(sK + s * FA_TILE_BYTES, &tmQKV, bar_kv_full + 8 * s, ck, kv_tile(j) * FA_BK, slice);
            tma_load_3d(sV + s * FA_TILE_BYTES, &tmQKV, bar_kv_full + 8 * s, cv, kv_tile(j) * FA_BK, slice);
          }
        }
      }
    } else if (warp <= 14) {
      // ------------------------------------------------------------------ MMA issuers: warp 13 group A, warp 14 group B
      // One issuer warp per query tile: each walks its own stream  S_g(t+1), PV_g(t), S_g(t+2), PV_g(t+1) ...  and
      // never waits on the other group's softmax (a single issuer serving both in a fixed order coupled the two
      // groups through its blocking waits). tcgen05.commit only tracks the issuing thread's own MMAs, which is
      // exactly the per-group completion the softmax warps need. The whole warp walks the schedule (warp-uniform
      // control flow keeps the descriptors in uniform registers); one elected lane issues.
      // Shared barriers take one arrival per group: kv_empty (count 2) and q_empty (count 2); on A-only items
      // warp 13 commits twice, and warp 14 still waits every q / kv_full phase in order (a waiter that skipped
      // phases would alias on the parity bit).
      const int g = warp - 13;
      const uint32_t bg = bar_grp + 64 * g;
      constexpr uint32_t idesc_pv = (F16 ? umma_idesc_f16_f32(FA_BQ, FA_D) : umma_idesc_bf16_f32(FA_BQ, FA_D)) | (1u << 16);  // B is MN-major
      auto n_mma_of = [&](int j) {  // keys of the j-th walked tile rounded up to the MMA granularity (16)
        const int valid = min(FA_BK, T - kv_tile(j) * FA_BK);
        return (valid + 15) & ~15;
      };
      FA_PROF_DECL;
      // S_g for this group's tile number tg: walked tile j of the item whose first ring position is kv - j
      auto issue_s = [&](uint32_t tg, int j, uint32_t k, int commits_q) {
        const uint32_t kv = k * n_tiles + j;
        FA_PROF(7);
        if (tg > 0) mbar_wait(bg + B_SFREE, (tg - 1) & 1);
        FA_PROF(0);  // wait: S tile free
        const uint32_t s = kv % FA_STAGES;
        mbar_wait(bar_kv_full + 8 * s, (kv / FA_STAGES) & 1);
        tcgen05_fence_after();
        FA_PROF(1);  // wait: K/V landed
        if (elect_one_sync()) {
          const uint32_t idesc_s = F16 ? umma_idesc_f16_f32(FA_BQ, n_mma_of(j)) : umma_idesc_bf16_f32(FA_BQ, n_mma_of(j));
          const uint64_t qd = umma_smem_desc_kmajor<128>(sQ + ((k & 1) * 2 + g) * FA_TILE_BYTES);
          const uint64_t kd = umma_smem_desc_kmajor<128>(sK + s * FA_TILE_BYTES);
          const uint32_t tS = tmem_base + FA_COL_S + g * 128;
#pragma unroll
          for (int kk = 0; kk < FA_D / 16; ++kk) umma_bf16(tS, qd + 2 * kk, kd + 2 * kk, idesc_s, kk > 0);
          for (int i = 0; i < commits_q; ++i) umma_commit(bar_q_empty + 8 * (k & 1));  // this group's last S of the item
          umma_commit(bg + B_S);
        }
        __syncwarp();
        FA_PROF(2);  // issue S
      };
      auto issue_pv = [&](uint32_t tg, int j, uint32_t kv, bool first, bool last, uint32_t kg, int commits_kv) {
        FA_PROF(7);
        mbar_wait(bg + B_P, tg & 1);
        FA_PROF(3);  // wait: P stored
        if (first) mbar_wait(bg + B_OEMPTY, (kg & 1) ^ 1u);  // previous item's O_g has been read out of TMEM
        tcgen05_fence_after();
        FA_PROF(4);  // wait: O drained
        const uint32_t s = kv % FA_STAGES;
        if (elect_one_sync()) {
          const uint32_t tP = tmem_base + FA_COL_P + g * 64, tO = tmem_base + FA_COL_O + g * 64;
          const uint64_t vd = umma_smem_desc_mnmajor_sw128(sV + s * FA_TILE_BYTES, FA_TILE_BYTES);
          if (n_mma_of(j) == FA_BK) {
#pragma unroll
            for (int kk = 0; kk < FA_BK / 16; ++kk)  // 16 keys per step: 8 packed TMEM columns of P, 2 KB of the V tile
              umma_bf16_ts(tO, tP + 8 * kk, vd + 128 * kk, idesc_pv, !first || kk != 0);
          } else {
            for (int kk = 0; kk < n_mma_of(j) / 16; ++kk)
              umma_bf16_ts(tO, tP + 8 * kk, vd + 128 * kk, idesc_pv, !first || kk != 0);
          }
          for (int i = 0; i < commits_kv; ++i) umma_commit(bar_kv_empty + 8 * s);  // K(j), V(j) free once retired
          umma_commit(bg + B_PV);
          if (last) umma_commit(bg + B_OFULL);
        }
        __syncwarp();
        FA_PROF(5);  // issue PV
      };
      // Cursors over this group's tiles: (item, k = CTA-local item number, kind, j).
      struct Cur { int item; uint32_t k; int pair; int kind; int j; };
      const int pair_step = gridDim.x % n_pairs;  // pair index of item + gridDim.x without a division per tile
      auto cur_valid = [&](const Cur& c) { return c.item < total_items; };
      auto first_j = [&](int kind) { return kind == SPLIT ? g : 0; };
      auto last_j = [&](int kind) { return kind == SPLIT ? n_tiles - 1 - ((n_tiles - 1 - g) & 1) : n_tiles - 1; };
      auto advance = [&](Cur& c) {  // to the group's next tile
        for (;;) {
          ++c.j;
          if (c.j >= n_tiles) {
            c.item += gridDim.x;
            ++c.k;
            c.j = 0;
            if (c.item >= total_items) return;
            c.pair += pair_step;
            if (c.pair >= n_pairs) c.pair -= n_pairs;
            c.kind = pair_kind(c.pair);
          }
          if (mine(c.kind, g, c.j)) return;
        }
      };
      Cur cs{(int)blockIdx.x, 0u, (int)(blockIdx.x % n_pairs), 0, -1}, cp = cs;  // next S tile, next PV tile
      if (cur_valid(cs)) {
        cs.kind = cp.kind = pair_kind(cs.pair);
        advance(cs);
        advance(cp);
      }
      // The shared barriers (Q per item, kv_full per ring slot) must be observed phase by phase, also for the tiles
      // and items this group does not work on: (ok, oj) is the next ring position not yet observed.
      uint32_t ok = 0, obs_q = ~0u;  // obs_q: last item whose Q phase was observed
      int oj = 0;
      auto observe_up_to = [&](const Cur& c) {  // everything before tile (c.k, c.j), plus the Q phase of item c.k
        while (ok < c.k || (ok == c.k && oj < c.j)) {
          if (oj == 0) { mbar_wait(bar_q + 8 * (ok & 1), (ok >> 1) & 1); obs_q = ok; }
          const uint32_t kv = ok * n_tiles + oj;
          mbar_wait(bar_kv_full + 8 * (kv % FA_STAGES), (kv / FA_STAGES) & 1);
          if (++oj == n_tiles) { oj = 0; ++ok; }
        }
        if (oj == 0) { mbar_wait(bar_q + 8 * (ok & 1), (ok >> 1) & 1); obs_q = ok; }
        if (++oj == n_tiles) { oj = 0; ++ok; }  // the tile itself is waited for by issue_s
      };
      uint32_t ts = 0, tp = 0, kg = 0;  // S tiles issued, PV tiles issued, items finished (barrier phases)
      auto do_s = [&]() {
        FA_PROF(7);
        observe_up_to(cs);
        FA_PROF(6);  // observing shared barrier phases (incl. waiting for the next item's Q)
        const bool last = cs.j == last_j(cs.kind);
        issue_s(ts, cs.j, cs.k, last ? (cs.kind == SOLO ? 2 : 1) : 0);
        ++ts;
        advance(cs);
      };
      if (cur_valid(cs)) do_s();  // S(0)
      while (cur_valid(cp)) {
        // The next S tile first (it only needs the group's current S to be in registers) -- unless it belongs to
        // a later item whose Q has not landed yet (the other group is late): then this group's PV goes first.
        bool s_first = false;
        if (cur_valid(cs)) {
          if (cs.k == obs_q) s_first = true;
          else if (cs.k == obs_q + 1) s_first = __all_sync(0xffffffffu, mbar_try_wait(bar_q + 8 * (cs.k & 1), (cs.k >> 1) & 1));
        }
        if (s_first) do_s();
        const bool first = cp.j == first_j(cp.kind), last = cp.j == last_j(cp.kind);
        issue_pv(tp, cp.j, cp.k * n_tiles + cp.j, first, last, kg, cp.kind == PAIRED ? 1 : 2);
        ++tp;
        if (last) ++kg;
        advance(cp);
        if (!s_first && cur_valid(cs)) do_s();
      }
      FA_PROF(7);
      FA_PROF_DUMP(tp);
    }  // warp 15 idle
  } else if (warp >= 8) {
    // ------------------------------------------------------------------ epilogue: O / l -> bf16 -> global
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(FA_REGS_EPILOGUE));
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const float* sL_gen = reinterpret_cast<const float*>(smem_gen + (sL - smem_base));
    const float c = args.scale_log2e;
    uint32_t kg[2] = {0, 0};
    for (int item = blockIdx.x; item < total_items; item += gridDim.x) {
      const int pair = item % n_pairs, bh = item / n_pairs, kind = item_kind(item);
      __nv_bfloat16* out_bh = args.out + ((size_t)(bh / args.heads) * T) * args.C + (bh % args.heads) * FA_D;
      float* outf_bh = reinterpret_cast<float*>(args.out) + ((size_t)(bh / args.heads) * T) * args.C + (bh % args.heads) * FA_D;
      if (kind == SPLIT) {
        // two partial softmaxes of the same query tile (even / odd K/V tiles): merge, then normalise
        const int qt = 2 * pair;
        const uint32_t pa = kg[0] & 1, pb = kg[1] & 1;
        ++kg[0];
        ++kg[1];
        mbar_wait(bar_grp + B_LFULL, pa);
        mbar_wait(bar_grp + 64 + B_LFULL, pb);
        const float la = sL_gen[(pa * 2 + 0) * 256 + row], ma = sL_gen[(pa * 2 + 0) * 256 + 128 + row];
        const float lb = sL_gen[(pb * 2 + 1) * 256 + row], mb = sL_gen[(pb * 2 + 1) * 256 + 128 + row];
        const float mm = fmaxf(ma, mb);
        float wa = ex2_approx((ma - mm) * c), wb = ex2_approx((mb - mm) * c);
        const float inv = 1.0f / (wa * la + wb * lb);
        wa *= inv;
        wb *= inv;
        mbar_wait(bar_grp + B_OFULL, pa);
        mbar_wait(bar_grp + 64 + B_OFULL, pb);
        tcgen05_fence_after();
        const bool warp_active = qt * FA_BQ + q * 32 < T;  // warp-uniform
        if (OUT32 && warp_active) {
          const int tok = qt * FA_BQ + row;
          uint4* dst = reinterpret_cast<uint4*>(outf_bh + (size_t)tok * args.C);
#pragma unroll 1
          for (int hh = 0; hh < 4; ++hh) {
            uint32_t oa[16], o2[16];
            tmem_ld_32x16(t_row + FA_COL_O + hh * 16, oa);
            tmem_ld_32x16(t_row + FA_COL_O + 64 + hh * 16, o2);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i)
              oa[i] = __float_as_uint(round_tf32(__uint_as_float(oa[i]) * wa + __uint_as_float(o2[i]) * wb));
            if (tok < T) {
#pragma unroll
              for (int i = 0; i < 4; ++i) dst[4 * hh + i] = make_uint4(oa[4 * i], oa[4 * i + 1], oa[4 * i + 2], oa[4 * i + 3]);
            }
          }
        } else if (warp_active) {
          const int tok = qt * FA_BQ + row;
          uint4* dst = reinterpret_cast<uint4*>(out_bh + (size_t)tok * args.C);
#pragma unroll 1
          for (int hh = 0; hh < 4; ++hh) {  // 16 columns of both partial outputs at a time
            uint32_t oa[16], o2[16], ob[8];
            tmem_ld_32x16(t_row + FA_COL_O + hh * 16, oa);
            tmem_ld_32x16(t_row + FA_COL_O + 64 + hh * 16, o2);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 8; ++i)
              ob[i] = pack_16x2<OUT16>(__uint_as_float(oa[2 * i]) * wa + __uint_as_float(o2[2 * i]) * wb,
                                  __uint_as_float(oa[2 * i + 1]) * wa + __uint_as_float(o2[2 * i + 1]) * wb);
            if (tok < T) {
              dst[2 * hh] = make_uint4(ob[0], ob[1], ob[2], ob[3]);
              dst[2 * hh + 1] = make_uint4(ob[4], ob[5], ob[6], ob[7]);
            }
          }
        }
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(bar_grp + B_OEMPTY);
          mbar_arrive(bar_grp + 64 + B_OEMPTY);
        }
        continue;
      }
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        if (kind == SOLO && g == 1) continue;
        const int qt = 2 * pair + g;
        const uint32_t bg = bar_grp + 64 * g;
        const uint32_t par = kg[g] & 1;
        ++kg[g];
        mbar_wait(bg + B_LFULL, par);
        const float l = sL_gen[(par * 2 + g) * 256 + row];
        mbar_wait(bg + B_OFULL, par);
        tcgen05_fence_after();
        const bool warp_active = qt * FA_BQ + q * 32 < T;  // warp-uniform
        if (OUT32 && warp_active) {
          const float inv = 1.0f / l;
          const int tok = qt * FA_BQ + row;
          uint4* dst = reinterpret_cast<uint4*>(outf_bh + (size_t)tok * args.C);
#pragma unroll 1
          for (int hh = 0; hh < 4; ++hh) {
            uint32_t o[16];
            tmem_ld_32x16(t_row + FA_COL_O + g * 64 + hh * 16, o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(round_tf32(__uint_as_float(o[i]) * inv));
            if (tok < T) {
#pragma unroll
              for (int i = 0; i < 4; ++i) dst[4 * hh + i] = make_uint4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]);
            }
          }
        } else if (warp_active) {
          const float inv = 1.0f / l;
          const int tok = qt * FA_BQ + row;
          uint4* dst = reinterpret_cast<uint4*>(out_bh + (size_t)tok * args.C);
#pragma unroll 1
          for (int hh = 0; hh < 2; ++hh) {  // 32 of the row's 64 outputs at a time: normalise, pack, store
            uint32_t o[32];
            tmem_ld_32x32(t_row + FA_COL_O + g * 64 + hh * 32, o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) o[i] = pack_16x2<OUT16>(__uint_as_float(o[2 * i]) * inv, __uint_as_float(o[2 * i + 1]) * inv);
            if (tok < T) {
#pragma unroll
              for (int i = 0; i < 4; ++i) dst[4 * hh + i] = make_uint4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]);
            }
          }
        }
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bg + B_OEMPTY);  // O has left TMEM: the next item's first PV may overwrite it
      }
    }
  } else {
    // ------------------------------------------------------------------ softmax warps, thread == query row
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(FA_REGS_SOFTMAX));
    const int g = warp >> 2;        // 0 = group A, 1 = group B
    const int q = warp & 3;         // TMEM lane quarter this warp may access (hardware rule: warp id % 4)
    const int row = q * 32 + lane;
    const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t tS = t_row + FA_COL_S + g * 128, tP = t_row + FA_COL_P + g * 64, tO = t_row + FA_COL_O + g * 64;
    const uint32_t bg = bar_grp + 64 * g;
    const float c = args.scale_log2e;
    const uint64_t c2 = pack_f32x2(c, c);
    float* sL_gen = reinterpret_cast<float*>(smem_gen + (sL - smem_base));
    uint32_t tile_it = 0, kg = 0;
    bool pending = false;  // P of the previous tile is stored but not yet published to the MMA warp
    FA_PROF_DECL;
    auto publish = [&]() {
      tmem_st_wait();
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bg + B_P);
      pending = false;
    };
    for (int item = blockIdx.x; item < total_items; item += gridDim.x) {
      const int pair = item % n_pairs, kind = item_kind(item);
      if (kind == SOLO && g == 1) continue;  // nothing for group B here; its issuer skips the item too
      const int qt = kind == PAIRED ? 2 * pair + g : 2 * pair;
      const bool warp_active = qt * FA_BQ + q * 32 < T;  // warp-uniform: all-padding warps only keep the barriers moving
      float m = 0.f, l = 0.f;
      bool first = true;  // first tile this group works on in the item
      for (int j = 0; j < n_tiles; ++j) {
        if (!mine(kind, g, j)) continue;
        FA_PROF(7);  // loop
        mbar_wait(bg + B_S, tile_it & 1);
        tcgen05_fence_after();
        FA_PROF(0);  // wait for S
        const int valid = min(FA_BK, T - kv_tile(j) * FA_BK);
        bool pv_seen = tile_it == 0;  // PV(t-1) known retired: O may be rescaled, P overwritten
        if (warp_active && valid == FA_BK) {
          // The whole 128-wide S row lives in registers: one TMEM read per tile, four loads in flight.
          // The row max of each 32-column chunk is taken while the next chunk is still on its way from TMEM
          // (a TMEM read moves 64 B/clk per scheduler: 16 KB = 256 cycles for the row, more than the 64 FMNMX3).
          uint32_t v[128];
          float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
          tmem_ld_32x32(tS, *reinterpret_cast<uint32_t(*)[32]>(&v[0]));
          if (pending) publish();  // P(j-1): its TMEM store drained under the load above
#pragma unroll
          for (int ch = 0; ch < 4; ++ch) {
            tmem_ld_wait();
            if (ch < 3) tmem_ld_32x32(tS + (ch + 1) * 32, *reinterpret_cast<uint32_t(*)[32]>(&v[32 * (ch + 1)]));
#pragma unroll
            for (int i = 32 * ch; i < 32 * ch + 32; i += 8) {
#pragma unroll
              for (int u = 0; u < 4; ++u)
                mx[u] = fmax3(mx[u], __uint_as_float(v[i + 2 * u]), __uint_as_float(v[i + 2 * u + 1]));
            }
          }
          tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bg + B_SFREE);  // the MMA warp may start S(j+1) under this tile's softmax
          FA_PROF(1);  // TMEM -> registers + row max
          const float mt = fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3]));
          if (first) {
            m = mt;
          } else {
            const bool need = (mt - m) * c > FA_RESCALE_LOG2;
            if (__any_sync(0xffffffffu, need)) {
              mbar_wait(bg + B_PV, (tile_it - 1) & 1);
              tcgen05_fence_after();
              pv_seen = true;
              const float f = need ? ex2_approx((m - mt) * c) : 1.0f;
#pragma unroll 1
              for (int hh = 0; hh < 4; ++hh) {  // 16 columns at a time: the S row keeps 128 registers busy
                uint32_t o[16];
                tmem_ld_32x16(tO + hh * 16, o);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * f);
                tmem_st_32x16(tO + hh * 16, o);
              }
              l *= f;
              if (need) m = mt;
            }
          }
          FA_PROF(2);  // row max (+ rescale)
          // ---- probabilities, packed in place (element pair i -> register i); packed FMA + packed row sums
          const float nmc = -m * c;
          const uint64_t nmc2 = pack_f32x2(nmc, nmc);
          uint64_t ls[4] = {0ull, 0ull, 0ull, 0ull};
#pragma unroll
          for (int i = 0; i < 64; ++i) {
            const uint64_t t2 = fma_f32x2(pack_f32x2(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1])), c2, nmc2);
            float t0, t1;
            unpack_f32x2(t2, t0, t1);
            const float p0 = ex2_approx(t0), p1 = ex2_approx(t1);
            ls[i & 3] = add_f32x2(ls[i & 3], pack_f32x2(p0, p1));
            v[i] = pack_16x2<F16>(p0, p1);
          }
          {
            float a0, a1;
            unpack_f32x2(add_f32x2(add_f32x2(ls[0], ls[1]), add_f32x2(ls[2], ls[3])), a0, a1);
            l += a0 + a1;
          }
          FA_PROF(4);  // exp
          if (!pv_seen) {
            mbar_wait(bg + B_PV, (tile_it - 1) & 1);
            tcgen05_fence_after();
          }
#pragma unroll
          for (int ch = 0; ch < 4; ++ch)
            tmem_st_32x16(tP + ch * 16, *reinterpret_cast<uint32_t(*)[16]>(&v[16 * ch]));
          pending = true;
          if (j + 1 == n_tiles || (kind == SPLIT && j + 2 >= n_tiles)) publish();  // last one: the epilogue is waiting
          FA_PROF(5);  // wait PV(j-1), store P
        } else if (warp_active && valid <= 16 && first) {
          // ---- short ragged tile walked first (1029 = 8 * 128 + 5): its 16 columns stay in registers, S is released at
          // once, and the wait for the previous item's last PV (P is about to be overwritten) comes after the
          // exponentials instead of in front of the load; the publish is deferred like that of a full tile.
          uint32_t v[16];
          tmem_ld_32x16(tS, v);
          if (pending) publish();
          tmem_ld_wait();
          tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bg + B_SFREE);
          float mt = -INFINITY;
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (i < valid) mt = fmaxf(mt, __uint_as_float(v[i]));
          m = mt;
          const float nmc = -m * c;
          uint32_t pk[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float p0 = 2 * i < valid ? ex2_approx(fmaf(__uint_as_float(v[2 * i]), c, nmc)) : 0.f;
            const float p1 = 2 * i + 1 < valid ? ex2_approx(fmaf(__uint_as_float(v[2 * i + 1]), c, nmc)) : 0.f;
            l += p0 + p1;
            pk[i] = pack_16x2<F16>(p0, p1);
          }
          if (!pv_seen) {
            mbar_wait(bg + B_PV, (tile_it - 1) & 1);
            tcgen05_fence_after();
          }
          tmem_st_32x8(tP, pk);
          pending = true;
          if (j + 1 == n_tiles || (kind == SPLIT && j + 2 >= n_tiles)) publish();
          FA_PROF(6);  // ragged tile
        } else {
          if (pending) publish();
          if (!pv_seen) {
            mbar_wait(bg + B_PV, (tile_it - 1) & 1);
            tcgen05_fence_after();
          }
          if (warp_active) {
            // ---- ragged last tile: `valid` keys inside an N = roundup16(valid) MMA, 16-column chunks
            const int nch = (valid + 15) >> 4;
            float mt = -INFINITY;
            for (int ch = 0; ch < nch; ++ch) {
              uint32_t v[16];
              tmem_ld_32x16(tS + ch * 16, v);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 16; ++i)
                if (ch * 16 + i < valid) mt = fmaxf(mt, __uint_as_float(v[i]));
            }
            if (first) {
              m = mt;
            } else {
              const bool need = (mt - m) * c > FA_RESCALE_LOG2;
              if (__any_sync(0xffffffffu, need)) {
                const float f = need ? ex2_approx((m - mt) * c) : 1.0f;
#pragma unroll 1
                for (int hh = 0; hh < 2; ++hh) {
                  uint32_t o[32];
                  tmem_ld_32x32(tO + hh * 32, o);
                  tmem_ld_wait();
#pragma unroll
                  for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * f);
                  tmem_st_32x32(tO + hh * 32, o);
                }
                l *= f;
                if (need) m = mt;
              }
            }
            const float nmc = -m * c;
            for (int ch = 0; ch < nch; ++ch) {
              uint32_t v[16];
              tmem_ld_32x16(tS + ch * 16, v);
              tmem_ld_wait();
              uint32_t pk[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const int k0 = ch * 16 + 2 * i;
                const float p0 = k0 < valid ? ex2_approx(fmaf(__uint_as_float(v[2 * i]), c, nmc)) : 0.f;
                const float p1 = k0 + 1 < valid ? ex2_approx(fmaf(__uint_as_float(v[2 * i + 1]), c, nmc)) : 0.f;
                l += p0 + p1;
                pk[i] = pack_16x2<F16>(p0, p1);
              }
              tmem_st_32x8(tP + ch * 8, pk);
            }
          }
          tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bg + B_SFREE);
          publish();
          FA_PROF(6);  // ragged / padding tile
        }
        first = false;
        ++tile_it;
      }
      // hand the row sums (and, for the merge of a SPLIT item, the row maxima) to the epilogue warps; next item
      sL_gen[((kg & 1) * 2 + g) * 256 + row] = l;
      sL_gen[((kg & 1) * 2 + g) * 256 + 128 + row] = m;
      ++kg;
      __syncwarp();
      if (lane == 0) mbar_arrive(bg + B_LFULL);
    }  // item loop
    FA_PROF(7);
    FA_PROF_DUMP(tile_it);
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 13) {
    __syncwarp();
    tcgen05_fence_after();
    tmem_dealloc<FA_TMEM_COLS>(tmem_base);
  }
}

}  // namespace cvit

using namespace cvit;

#ifdef CVIT_FA_TRACE
static long long* g_fa_trace = nullptr;
extern "C" void cvit_fa_set_trace(long long* p) { g_fa_trace = p; }
#endif

template <bool F16, bool OUT16, bool OUT32 = false>
static int attention_fwd(const void* qkv, void* out, int64_t n_slices, int64_t tokens, int64_t heads, int64_t head_dim,
                         void* stream) {
  if (!qkv || !out || n_slices <= 0 || tokens <= 0 || heads <= 0) {
    set_error("attention: bad arguments");
    return CVIT_ERR_INVALID;
  }
  if (head_dim != FA_D) {
    set_error("attention: head_dim=%lld unsupported (64 only: every DINOv2 variant)", (long long)head_dim);
    return CVIT_ERR_UNSUPPORTED;
  }
  if (((tokens + FA_BQ - 1) / FA_BQ) * heads * n_slices > 0x7fffffffll) {
    set_error("attention: too many work items");
    return CVIT_ERR_UNSUPPORTED;
  }
  const int64_t C = heads * FA_D;
  CUtensorMap tm;
  uint64_t dims[3] = {(uint64_t)(3 * C), (uint64_t)tokens, (uint64_t)n_slices};
  uint64_t strides[3] = {0, (uint64_t)(3 * C) * 2, (uint64_t)tokens * 3 * C * 2};
  uint32_t box[3] = {FA_D, FA_BK, 1};
  int rc = encode_tmap(&tm, F16 ? TmapDtype::F16 : TmapDtype::BF16, 3, qkv, dims, strides, box, 128);
  if (rc) return rc;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(attention_tcgen05_kernel<F16, OUT16, OUT32>, cudaFuncAttributeMaxDynamicSharedMemorySize, FA_SMEM);
    if (e != cudaSuccess) {
      set_error("attention: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      return CVIT_ERR_CUDA;
    }
    configured = true;
  }
  FaArgs a;
#ifdef CVIT_FA_TRACE
  a.trace = g_fa_trace;
#else
  a.trace = nullptr;
#endif
  a.out = static_cast<__nv_bfloat16*>(out);
  a.T = (int)tokens;
  a.heads = (int)heads;
  a.C = (int)C;
  a.slices = (int)n_slices;
  a.scale_log2e = 0.125f * 1.4426950408889634f;
  const int n_qt = (int)((tokens + FA_BQ - 1) / FA_BQ);
  const int64_t items = (int64_t)((n_qt + 1) / 2) * heads * n_slices;
  int grid = num_sms();
  if (grid > items) grid = (int)items;
  attention_tcgen05_kernel<F16, OUT16, OUT32><<<grid, FA_THREADS, FA_SMEM, (cudaStream_t)stream>>>(tm, a);
  return check_launch("attention_tcgen05_kernel");
}

extern "C" int cvit_attention_fwd_bf16(const void* qkv, void* out, int64_t n_slices, int64_t tokens, int64_t heads,
                                       int64_t head_dim, void* stream) {
  return attention_fwd<false, false>(qkv, out, n_slices, tokens, heads, head_dim, stream);
}

// Same kernel with IEEE fp16 q/k/v, probabilities and output (the fp16-operand ViT path).
extern "C" int cvit_attention_fwd_f16(const void* qkv, void* out, int64_t n_slices, int64_t tokens, int64_t heads,
                                      int64_t head_dim, void* stream) {
  return attention_fwd<true, true>(qkv, out, n_slices, tokens, heads, head_dim, stream);
}

// fmt: CVIT_FMT_OPERANDS_F16 (q/k/v and the probabilities are fp16) | CVIT_FMT_OUT_F16 (the output is stored as fp16)
// | CVIT_FMT_OUT_F32 (bf16 q/k/v and probabilities, TF32-rounded fp32 output).
extern "C" int cvit_attention_fwd_fmt(const void* qkv, void* out, int64_t n_slices, int64_t tokens, int64_t heads,
                                      int64_t head_dim, int fmt, void* stream) {
  switch (fmt) {
    case 0: return attention_fwd<false, false>(qkv, out, n_slices, tokens, heads, head_dim, stream);
    case 2: return attention_fwd<false, true>(qkv, out, n_slices, tokens, heads, head_dim, stream);
    case 3: return attention_fwd<true, true>(qkv, out, n_slices, tokens, heads, head_dim, stream);
    case 8: return attention_fwd<false, false, true>(qkv, out, n_slices, tokens, heads, head_dim, stream);
    default:
      set_error("attention: unsupported format flags 0x%x (0, OUT_F16, OPERANDS_F16|OUT_F16, OUT_F32)", fmt);
      return CVIT_ERR_UNSUPPORTED;
  }
}
