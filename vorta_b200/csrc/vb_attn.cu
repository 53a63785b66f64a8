// vb_attn.cu — tcgen05 / TMEM / TMA flash-attention forward for sm_100a, driven by key/value *run lists*.
//
// One kernel serves all three VORTA branches (reference: vorta/attention/wan.py:103-149 SDPA, :243-270 coreset,
// :272-294 sliding tile).  A CTA owns up to two 128-row query tiles that attend to the same list of contiguous
// key ranges ("runs", in kernel order):
//     full     : one run [0, N)
//     coreset  : one run [0, S_c (+ text))   over the pooled sequence
//     sliding  : the <= 9 (+1 text) runs of the 3-D tile window, tile-major order
// so the block-sparse schedule is just a different table, and masked 3-D tiles are never visited.
//
// Warp roles (608 threads):
//     warps 0-15 : softmax + correction + epilogue; warp = 8 t + 4 h + q: query tile t, key / channel half h, row
//                  quarter q (TMEM lanes 32 q .. 32 q + 31) - two threads per query row
//     warp  16   : TMA producer (Q tiles once, then K/V blocks through a 5-slot ring of 32 KB)
//     warps 17,18: tcgen05.mma issuers, one per query tile (17 also allocates TMEM)
// TMEM (512 columns): S [0,128) shared by the two tiles | P0 [128,192) P1 [192,256) (bf16) | O0 [256,384) O1 [384,512).
// S = Q K^T is an SS UMMA (both operands K-major, SWIZZLE_128B as written by TMA), O += P V is a TS UMMA (P from
// TMEM, V from shared memory, MN-major).
//
// Decoupled pipeline.  P does not alias S, so QK_t(j+1) does not have to wait for softmax_t(j) -> PV_t(j): it is issued
// as soon as the softmax warps of tile t have their row maximum of block j (bar_qk_go) and the S region has been
// loaded into registers by its previous user (bar_s_free; the region alternates strictly between the tiles).  The
// softmax warps find S(j+1) complete when they finish block j and do not wait in steady state.  (With P aliased on S
// and one S per tile the chain softmax -> PV -> QK was serial per tile: 1600 + 300 + 1024 cycles per block, tensor pipe
// 61 % busy; profiles/r1g_timeline_dense16k.log vs r1l_timeline_decoupled.log.)
#include <algorithm>

#include "vb_common.cuh"
#include "vb_ptx.cuh"

namespace vb {

constexpr int kNumSlots = 5;                       // K/V ring
constexpr int kTileBytes = kBlockN * kHeadDim * 2; // 32 KB: one 128x128 bf16 block = two 128x64 swizzled halves
constexpr int kHalfBytes = kTileBytes / 2;
constexpr int kSoftmaxWarps = 16;                  // 2 tiles x 2 column halves x 4 row quarters
constexpr int kTmaWarp = kSoftmaxWarps;
constexpr int kMmaWarp = kSoftmaxWarps + 1;
constexpr int kMmaWarps = 2;                       // one issuer per query tile, on different schedulers
constexpr int kAttnThreads = (kSoftmaxWarps + 1 + kMmaWarps) * 32;
constexpr int kConsumerWarps = kSoftmaxWarps + kMmaWarps;   // warps that follow the producer's work-item queue
#ifndef VB_POLY_GROUPS
#define VB_POLY_GROUPS 0x02        // group 1 of every 8 groups of 4 keys: 1/8 of the exps on the FMA pipe (measured best of 0, 1/8, 2/8, 3/8)
#endif
constexpr unsigned kPolyGroups = VB_POLY_GROUPS;
constexpr float kRescaleThreshold = 8.0f;          // lazy rescale: tolerate 2^8 growth before touching O

struct SmemLayout {
  uint8_t q[2 * kTileBytes];                 // two query tiles
  uint8_t kv[kNumSlots * kTileBytes];        // K/V ring
  uint64_t bar_q_full[2];
  uint64_t bar_q_empty[2];      // every QK of the item that used Q_t completed: the next item's Q_t may land
  uint64_t bar_slot_full[kNumSlots];
  uint64_t bar_slot_empty[kNumSlots];
  uint64_t bar_s_full[2];
  uint64_t bar_p_half[2];
  uint64_t bar_p_ready[2];
  uint64_t bar_o_full[2];
  uint64_t bar_o_free[2];       // the epilogue of tile t holds O_t in registers: PV(0) of the next item may overwrite it
  uint64_t bar_s_free;          // the shared S region has been loaded into registers by its tile's softmax warps
  uint64_t bar_qk_go[2];        // softmax of tile t passed the trigger point of its block: QK of the next block may issue
  uint64_t bar_pv_done[2];      // PV of tile t completed: P_t is free again and O_t is quiescent
  uint64_t bar_item_full[2];    // the producer published the index of the CTA's next work item
  uint64_t bar_item_empty[2];   // all 18 consumer warps have read it
  int32_t item_idx[2];          // work-item queue (depth 2): item index, or -1 = no more work
  uint32_t tmem_base_slot;
  float xchg[2][2][kBlockM];                 // row max / row sum exchange between the two threads of a row
};
constexpr int kAttnSmemBytes = sizeof(SmemLayout);
static_assert(kAttnSmemBytes <= 232448, "exceeds the 227 KB shared memory of an sm_100 CTA");

// Walks the 128-key blocks of a run list that lives in global memory (<= a dozen 8-byte reads per work item, L1 hits
// after the first role touched them).
struct BlockWalker {
  const KvRun* runs;
  int n_runs, r, off, start, len;
  __device__ __forceinline__ BlockWalker(const KvRun* rr, int n) : runs(rr), n_runs(n), r(0), off(0), start(0), len(0) {
    if (n > 0) fetch();
  }
  __device__ __forceinline__ void fetch() {
    const int2 v = __ldg(reinterpret_cast<const int2*>(runs + r));
    start = v.x;
    len = v.y;
  }
  // next 128-key block: first key row and number of valid keys; false when exhausted
  __device__ __forceinline__ bool next(int& row0, int& valid) {
    while (r < n_runs) {
      if (off < len) {
        row0 = start + off;
        valid = min(kBlockN, len - off);
        off += kBlockN;
        return true;
      }
      ++r;
      off = 0;
      if (r < n_runs) fetch();
    }
    return false;
  }
};

#ifdef VB_TIMELINE               // perf experiment: clock stamps of the first item of CTA 0 -> p.dbg as int64[who][block][8]
#define VB_STAMP(who, j, slot)                                                                         \
  do {                                                                                                 \
    if (p.dbg != nullptr && item == 0 && (j) < 64)                                                     \
      reinterpret_cast<long long*>(p.dbg)[((who) * 64 + (j)) * 8 + (slot)] = clock64();                \
  } while (0)
#else
#define VB_STAMP(who, j, slot) do {} while (0)
#endif

#define VB_EXP2(x) fast_exp2(x)

// Work item -> (segment, pair, head, batch); segments are laid out longest items first by the host.  Every role of the
// CTA decodes the item itself (warp-uniform integer math + 48 bytes from global memory), so no hand-off is needed.
struct Item {
  int seg_idx, batch;
  QPair pair;
  AttnHead head;
};
__device__ __forceinline__ Item decode_item(const AttnParams& p, int item) {
  Item it;
  it.seg_idx = 0;
#pragma unroll
  for (int i = 1; i < kMaxSegments; ++i)
    if (i < p.n_seg && item >= p.seg[i].cta_begin) it.seg_idx = i;
  const AttnSeg& seg = p.seg[it.seg_idx];
  const int local = item - seg.cta_begin;
  const int4* src = reinterpret_cast<const int4*>(seg.pairs + local % seg.n_pairs);
  int4* dst = reinterpret_cast<int4*>(&it.pair);
  dst[0] = __ldg(src);
  dst[1] = __ldg(src + 1);
  dst[2] = __ldg(src + 2);
  it.head = p.heads[seg.head0 + (local / seg.n_pairs) % seg.n_heads];
  it.batch = local / (seg.n_pairs * seg.n_heads);
  return it;
}

// Persistent kernel, one CTA per SM.  Work items are handed out dynamically: the first item of CTA c is item c, every
// further one comes from a global counter (the TMA producer fetches it and publishes it to the other 18 warps through a
// two-entry queue in shared memory).  The host sorts items longest first, so this is greedy longest-processing-time
// scheduling: a layer's full, coreset and sliding items differ ~10x in length, and a static round-robin measured 5-9 %
// slower in-step (profiles/r2b_*).  The counter resets itself: n_items fetches in total, the last wraps it to 0.
// All pipelines run THROUGH the
// item boundary: the K/V ring and every mbarrier keep their running phase, the producer prefetches the next item's
// K/V and Q while the current item drains, and the issuer puts QK(0) of the next item on the tensor pipe while the
// softmax warps are still in the epilogue of the current one.  Per-item cost outside the steady state was ~11 us
// (CTA launch, TMEM allocation, barrier init, cold Q/K loads, pipeline fill, epilogue) against 3.4 us of work for a
// 512-key cross-attention item and 77 us for a Wan-14B sliding-tile item (profiles/r1t_attn_full_summary_wan14.md).
__global__ void __launch_bounds__(kAttnThreads, 1)
vb_attn_fwd_kernel(const __grid_constant__ AttnTmaps tmaps, const __grid_constant__ AttnParams p) {
  // Everything lives in dynamic shared memory (no static __shared__), so the operand area starts at the CTA's
  // shared window base, which is 1024-byte aligned as SWIZZLE_128B needs; checked below.
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  SmemLayout& sm = *reinterpret_cast<SmemLayout*>(smem_raw);
  uint64_t* bar_q_full = sm.bar_q_full;
  uint64_t* bar_slot_full = sm.bar_slot_full;
  uint64_t* bar_slot_empty = sm.bar_slot_empty;
  uint64_t* bar_s_full = sm.bar_s_full;
  uint64_t* bar_p_half = sm.bar_p_half;
  uint64_t* bar_p_ready = sm.bar_p_ready;
  uint64_t* bar_o_full = sm.bar_o_full;
  uint32_t& tmem_base_slot = sm.tmem_base_slot;
  float (*s_xchg)[2][kBlockM] = sm.xchg;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);   // provably warp-uniform: role / address math in uniform registers
  const int lane = threadIdx.x & 31;

  if ((smem_u32(smem_raw) & 1023u) != 0) {      // SWIZZLE_128B atoms are 8 rows x 128 B
    if (threadIdx.x == 0) printf("vb_attn_fwd_kernel: dynamic shared memory base is not 1024-byte aligned\n");
    __trap();
  }
  uint8_t* smem_q = sm.q;                       // 2 x 32 KB
  uint8_t* smem_kv = sm.kv;                     // kNumSlots x 32 KB

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bar_q_full[i], 1);
      mbar_init(&sm.bar_q_empty[i], 1);
      mbar_init(&bar_s_full[i], 1);
      mbar_init(&bar_p_half[i], kBlockM);    // 4 warps: column half 0 of P stored
      mbar_init(&bar_p_ready[i], kBlockM);   // 4 warps: column half 1 of P stored
      mbar_init(&bar_o_full[i], 1);
      mbar_init(&sm.bar_o_free[i], kSoftmaxWarps / 2);
    }
    for (int i = 0; i < kNumSlots; ++i) {
      mbar_init(&bar_slot_full[i], 1);
      mbar_init(&bar_slot_empty[i], 2);      // two commits per slot: one per tile that read it, or both by its only reader
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&sm.bar_item_full[i], 1);
      mbar_init(&sm.bar_item_empty[i], kConsumerWarps);
    }
    mbar_init(&sm.bar_s_free, kSoftmaxWarps / 2);        // lane 0 of the 8 warps of the loading tile
    for (int i = 0; i < 2; ++i) {
      mbar_init(&sm.bar_qk_go[i], kSoftmaxWarps / 2);
      mbar_init(&sm.bar_pv_done[i], 1);
    }
    fence_barrier_init();
  }
  if (warp == kTmaWarp && lane == 0) {
    for (int i = 0; i < p.n_seg; ++i) {
      tma_prefetch_desc(&tmaps.m[i][0]);
      tma_prefetch_desc(&tmaps.m[i][1]);
      tma_prefetch_desc(&tmaps.m[i][2]);
    }
  }
  if (warp == kMmaWarp) {
    tmem_alloc(&tmem_base_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_slot;
  // consumer side of the work-item queue: entry n lives in slot n & 1; -1 ends the loop (warp-uniform)
  auto next_item = [&](uint32_t n) -> int {
    mbar_wait(&sm.bar_item_full[n & 1u], (n >> 1) & 1u);
    const int item = *reinterpret_cast<volatile int32_t*>(&sm.item_idx[n & 1u]);
    __syncwarp();
    if (lane == 0) mbar_arrive(&sm.bar_item_empty[n & 1u]);
    return item;
  };

  if (warp == kTmaWarp) {
    // ======================================= TMA producer =======================================
    // The whole warp runs the loop converged; lane 0 owns the work counter, every expect_tx arrive and every load.
    uint32_t load_idx = 0;                 // position in the K/V ring, running through all items
    uint32_t q_uses[2] = {0, 0};           // items that used Q_t so far
    for (uint32_t n = 0;; ++n) {
      // fetch and publish: the first item is the CTA index, the rest come from the self-resetting global counter
      // (atomicInc wraps to 0 on the launch's n_items-th fetch: gridDim.x of the fetches are the "no more work" ones)
      int item = static_cast<int>(blockIdx.x);
      if (n > 0) {
        if (lane == 0) item = static_cast<int>(gridDim.x + atomicInc(p.work_counter, static_cast<unsigned>(p.n_items - 1)));
        item = __shfl_sync(0xffffffffu, item, 0);
      }
      if (item >= p.n_items) item = -1;
      mbar_wait(&sm.bar_item_empty[n & 1u], ((n >> 1) & 1u) ^ 1u);
      if (lane == 0) {
        *reinterpret_cast<volatile int32_t*>(&sm.item_idx[n & 1u]) = item;
        mbar_arrive(&sm.bar_item_full[n & 1u]);          // release semantics: the store above is visible to the waiters
      }
      if (item < 0) break;
      const Item it = decode_item(p, item);
      const AttnSeg& seg = p.seg[it.seg_idx];
      const CUtensorMap* tmap_q = &tmaps.m[it.seg_idx][0];
      const CUtensorMap* tmap_k = &tmaps.m[it.seg_idx][1];
      const CUtensorMap* tmap_v = &tmaps.m[it.seg_idx][2];
      const int nq = it.pair.nq, hk = it.head.hk, batch = it.batch;
      // 128 rows [row0, row0 + 128) of one operand -> dst (two 64-channel halves of 16 KB), completion on bar
      auto load_rows = [&](const CUtensorMap* m, int row0, uint8_t* dst, uint64_t* bar) {
        if (lane == 0) {
          mbar_arrive_expect_tx(bar, kTileBytes);
          tma_load_4d(dst, m, bar, 0, row0, hk, batch);
          tma_load_4d(dst + kHalfBytes, m, bar, 64, row0, hk, batch);
        }
      };
      auto load_kv = [&](const CUtensorMap* m, int row0) {
        const uint32_t slot = load_idx % kNumSlots;
        const uint32_t phase = (load_idx / kNumSlots) & 1u;
        mbar_wait(&bar_slot_empty[slot], phase ^ 1u);
        load_rows(m, row0, smem_kv + slot * kTileBytes, &bar_slot_full[slot]);
        ++load_idx;
      };
      auto load_q = [&]() {
        for (int t = 0; t < nq; ++t) {
          if (q_uses[t] > 0) mbar_wait(&sm.bar_q_empty[t], (q_uses[t] - 1) & 1u);
          ++q_uses[t];
          load_rows(tmap_q, it.pair.q_row0[t], smem_q + t * kTileBytes, &bar_q_full[t]);
        }
      };
      BlockWalker w0(seg.runs + it.pair.run_begin, it.pair.run_count);
      BlockWalker w1(seg.runs + it.pair.run_begin2, it.pair.split ? it.pair.run_count2 : 0);
      int row0, valid;
      // the first K block does not depend on the previous item having released Q: request it first
      for (int j = 0; w0.next(row0, valid); ++j) {
        load_kv(tmap_k, row0);
        if (j == 0) load_q();
        load_kv(tmap_v, row0);
        if (it.pair.split && w1.next(row0, valid)) {      // K1 V1 of the same block step
          load_kv(tmap_k, row0);
          load_kv(tmap_v, row0);
        }
      }
    }
  } else if (warp >= kMmaWarp) {
    // ======================================= MMA issuer =========================================
    // The whole warp runs this role converged and every address below is made warp-uniform, so descriptors live
    // in uniform registers and one elected lane issues; a single-lane role pays a register->uniform "waterfall"
    // per operand (measured: ~250 SASS instructions per 16 MMAs, the round-1 bottleneck).
    constexpr uint32_t idesc_qk0 = umma_idesc_bf16(kBlockM, 0, 0, 0);       // N filled in per block (tails are narrower)
    constexpr uint32_t idesc_pv = umma_idesc_bf16(kBlockM, kHeadDim, 0, 1);
    constexpr uint64_t desc_hi = static_cast<uint64_t>((1024u >> 4) | (1u << 14) | (2u << 29)) << 32;
    constexpr uint32_t lbo_k = 1u << 16;
    constexpr uint32_t lbo_v = (kHalfBytes >> 4) << 16;
    const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t q_lo = __shfl_sync(0xffffffffu, (smem_u32(smem_q) & 0x3FFFFu) >> 4, 0);
    const uint32_t kv_lo = __shfl_sync(0xffffffffu, (smem_u32(smem_kv) & 0x3FFFFu) >> 4, 0);
    const int t = warp - kMmaWarp;
    auto issue_qk = [&](uint32_t slot, int n_keys) {     // n_keys: multiple of 16 (a run's tail block is narrower)
      const uint32_t a0 = q_lo + t * (kTileBytes >> 4) + lbo_k;
      const uint32_t b0 = kv_lo + slot * (kTileBytes >> 4) + lbo_k;
      const uint32_t idesc = idesc_qk0 | (static_cast<uint32_t>(n_keys >> 3) << 17);
#pragma unroll
      for (int k = 0; k < kHeadDim / 16; ++k) {
        const uint32_t off = (k >> 2) * (kHalfBytes >> 4) + (k & 3) * 2;
        umma_ss(tb, desc_hi | (a0 + off), desc_hi | (b0 + off), idesc, k > 0);
      }
    };
    // 16-key steps [4 half, 4 half + 4) clipped to k_steps; full blocks (k_steps == 8) take the unrolled path: the
    // issuer crawls between MMA batches, every instruction it does not execute there is tensor-pipe time
    auto issue_pv = [&](uint32_t slot, uint32_t accumulate, int half, int k_steps) {
      const uint32_t b0 = kv_lo + slot * (kTileBytes >> 4) + lbo_v;
      const uint32_t d = tb + 2 * kBlockN + t * kHeadDim;
      const uint32_t a = tb + kBlockN + t * 64;
      if (k_steps == kBlockN / 16) {
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const int k = half * 4 + kk;
          umma_ts(d, a + k * 8, desc_hi | (b0 + k * (2048 >> 4)), idesc_pv, accumulate | (k > 0));
        }
      } else {
        for (int k = half * 4; k < min(k_steps, half * 4 + 4); ++k)
          umma_ts(d, a + k * 8, desc_hi | (b0 + k * (2048 >> 4)), idesc_pv, accumulate | (k > 0));
      }
    };
    // One issuer warp per query tile, on different schedulers: an issuer shares its scheduler with four busy softmax
    // warps and crawls through the ~40 instructions between two MMA batches (measured 220-600 cycles); with two
    // issuers one tile's gap overlaps the other tile's batch (one issuer for both tiles: 1230 TFLOP/s dense, two:
    // 1415; a polling event loop instead of in-order suspended waits starved completely: 1167).  Each issues, in
    // order, QK_t(0), then per block QK_t(j+1) and PV_t(j) in two halves of 64 keys.
    // The S region alternates strictly between the tiles through bar_s_free: use number u waits for completion u - 1.
    uint32_t ring0 = 0;      // K/V ring index of the item's first load
    uint32_t use0 = 0;       // S-region use number of the item's first QK
    uint32_t blk = 0;        // blocks this tile has processed so far (phase of its per-block barriers)
    uint32_t items_t = 0;    // items this tile has processed so far
    for (uint32_t n = 0;; ++n) {
      const int item = next_item(n);
      if (item < 0) break;
      const Item it = decode_item(p, item);
      const AttnSeg& seg = p.seg[it.seg_idx];
      const int nq = it.pair.nq, nblk = it.pair.n_blocks, split = it.pair.split;
      const uint32_t ring_stride = split ? 4u : 2u, ring_off = split ? 2u * t : 0u;
      const uint32_t empties = (nq == 2 && !split) ? 1u : 2u;      // commits this issuer owes a slot it read
      if (t < nq) {
        BlockWalker w(seg.runs + (split && t == 1 ? it.pair.run_begin2 : it.pair.run_begin),
                      split && t == 1 ? it.pair.run_count2 : it.pair.run_count);
        int row0, valid_next = 0, valid_cur = 0;
        w.next(row0, valid_next);
        mbar_wait(&bar_q_full[t], items_t & 1u);
        auto do_qk = [&](int j, int valid) {
          const uint32_t k_idx = ring0 + ring_stride * j + ring_off, k_slot = k_idx % kNumSlots,
                         k_phase = (k_idx / kNumSlots) & 1u;
          const uint32_t use = use0 + nq * j + t;
          if (blk + j > 0) mbar_wait(&sm.bar_qk_go[t], (blk + j - 1) & 1u);
          if (use > 0) mbar_wait(&sm.bar_s_free, (use - 1) & 1u);
          mbar_wait(&bar_slot_full[k_slot], k_phase);
          tc_fence_after();
          if (lane == 0) VB_STAMP(2 + t, j, 0);
          if (elect_one()) {
            issue_qk(k_slot, (valid + 15) & ~15);
            umma_commit(&bar_s_full[t]);
            umma_commit(&bar_slot_empty[k_slot]);
            if (empties == 2) umma_commit(&bar_slot_empty[k_slot]);
            if (j == nblk - 1) umma_commit(&sm.bar_q_empty[t]);
          }
          __syncwarp();
          if (lane == 0) VB_STAMP(2 + t, j, 3);
        };
        do_qk(0, valid_next);
        for (int j = 0; j < nblk; ++j) {
          const uint32_t v_idx = ring0 + ring_stride * j + ring_off + 1, v_slot = v_idx % kNumSlots,
                         v_phase = (v_idx / kNumSlots) & 1u;
          valid_cur = valid_next;
          if (j + 1 < nblk) {
            w.next(row0, valid_next);
            do_qk(j + 1, valid_next);
          }
          const int k_steps = (valid_cur + 15) >> 4;           // 16-key steps that hold real keys (tail blocks: < 8)
          mbar_wait(&bar_slot_full[v_slot], v_phase);
          mbar_wait(&bar_p_half[t], (blk + j) & 1u);
          if (j == 0 && items_t > 0) mbar_wait(&sm.bar_o_free[t], (items_t - 1) & 1u);
          tc_fence_after();
          if (lane == 0) VB_STAMP(2 + t, j, 1);
          if (elect_one()) issue_pv(v_slot, j > 0, 0, k_steps);
          __syncwarp();
          mbar_wait(&bar_p_ready[t], (blk + j) & 1u);
          tc_fence_after();
          if (elect_one()) {
            issue_pv(v_slot, j > 0, 1, k_steps);
            umma_commit(&sm.bar_pv_done[t]);
            umma_commit(&bar_slot_empty[v_slot]);
            if (empties == 2) umma_commit(&bar_slot_empty[v_slot]);
            if (j == nblk - 1) umma_commit(&bar_o_full[t]);
          }
          __syncwarp();
          if (lane == 0) VB_STAMP(2 + t, j, 2);
        }
        blk += nblk;
        ++items_t;
      }
      ring0 += ring_stride * nblk;
      use0 += nq * nblk;
    }
  } else {
    // ============================ softmax / correction / epilogue ===============================
    // TWO threads per query row: warp = 8 t + 4 h + q handles rows [32 q, 32 q + 32) of tile t, keys / channels
    // [64 h, 64 h + 64).  All warps with the same q sit on scheduler q and may touch TMEM lanes 32 q..32 q + 31, so
    // the pair (h = 0, 1) interleaves on one scheduler: a single warp per tile left the issue slot idle ~60 % of the
    // time on fixed-latency dependencies (round-1 timeline: 1550-1700 cycles per block for ~600 instructions).
    const int t = warp >> 3;
    const int h = (warp >> 2) & 1;
    const int q4 = warp & 3;
    const int row = (q4 << 5) + lane;               // query row inside the tile == TMEM lane
    const int pair_bar = 1 + t * 4 + q4;            // named barrier of the two warps sharing these rows
    const uint32_t lane_addr = static_cast<uint32_t>(q4 << 5) << 16;
    const uint32_t s_addr = tmem_base + lane_addr;                              // S region shared by both tiles
    const uint32_t p_addr = tmem_base + lane_addr + kBlockN + t * 64 + h * 32;  // P_t: its own 64 columns
    const uint32_t o_addr = tmem_base + lane_addr + 2 * kBlockN + t * kHeadDim + h * 64;
    const float scale = p.scale_log2;
    uint32_t blk = 0;        // blocks this tile has processed so far
    uint32_t items_t = 0;    // items this tile has processed so far
    for (uint32_t n = 0;; ++n) {
      const int item = next_item(n);
      if (item < 0) break;
      float m_ref = 0.f, l_sum = 0.f;
      const KvRun* run_ptr;
      int run_cnt;
      {   // only the run list is needed inside the block loop: the rest of the item is decoded again in the epilogue
          // instead of being carried through the loop in registers (the loop body sits at the register cap)
        const Item it = decode_item(p, item);
        if (t >= it.pair.nq) continue;
        const bool second = it.pair.split && t == 1;
        run_ptr = p.seg[it.seg_idx].runs + (second ? it.pair.run_begin2 : it.pair.run_begin);
        run_cnt = second ? it.pair.run_count2 : it.pair.run_count;
      }
      BlockWalker w(run_ptr, run_cnt);
      int row0, valid;
      for (int j = 0; w.next(row0, valid); ++j, ++blk) {
        if (row == 0 && h == 0) VB_STAMP(t, j, 0);
        mbar_wait(&bar_s_full[t], blk & 1u);
        tc_fence_after();
        if (row == 0 && h == 0) VB_STAMP(t, j, 1);
        uint32_t s[2][32];
#pragma unroll
        for (int c = 0; c < 2; ++c) tmem_ld32(s_addr + h * 64 + c * 32, s[c]);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&sm.bar_s_free);      // the S region may be overwritten by the next QK
        if (row == 0 && h == 0) VB_STAMP(t, j, 2);
        if (valid < kBlockN) {   // run tail: keys beyond the run do not exist for this query (the QK of a tail block is
                                 // issued for the valid keys rounded up to 16 only: the columns behind hold stale scores)
#pragma unroll
          for (int c = 0; c < 2; ++c)
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (h * 64 + c * 32 + i >= valid) s[c][i] = 0xff800000u;   // -inf
        }
        float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
        for (int c = 0; c < 2; ++c)
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            mx0 = fmaxf(mx0, __uint_as_float(s[c][i + 0]));
            mx1 = fmaxf(mx1, __uint_as_float(s[c][i + 1]));
            mx2 = fmaxf(mx2, __uint_as_float(s[c][i + 2]));
            mx3 = fmaxf(mx3, __uint_as_float(s[c][i + 3]));
          }
        // row maximum over both halves (exchange through shared memory + a 64-thread named barrier)
        s_xchg[t][h][row] = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
        named_bar_sync(pair_bar, 64);
        const float m_new = fmaxf(s_xchg[t][0][row], s_xchg[t][1][row]) * scale;   // block has >= 1 valid key: finite
        if (lane == 0) mbar_arrive(&sm.bar_qk_go[t]);          // the next QK of this tile (next block or next item) may issue
        if (row == 0 && h == 0) VB_STAMP(t, j, 6);

        if (j == 0) {
          m_ref = m_new;
        } else {
          const bool need = m_new > m_ref + kRescaleThreshold;
          if (__any_sync(0xffffffffu, need)) {             // identical in both warps of the pair (same rows)
            float alpha = 1.f;
            if (need) {
              alpha = fast_exp2(m_ref - m_new);
              m_ref = m_new;
            }
            // O_t must be quiescent: PV_t(j-1) may still be in flight (QK_t(j) was issued before it), PV_t(j) cannot
            // start before BOTH halves have arrived below.  Each thread rescales its 64 channels.
            mbar_wait(&sm.bar_pv_done[t], (blk - 1) & 1u);
            tc_fence_after();
#pragma unroll 1
            for (int c = 0; c < 4; ++c) {
              uint32_t o[16];
              tmem_ld16(o_addr + c * 16, o);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
              tmem_st16(o_addr + c * 16, o);
            }
            l_sum *= alpha;
            tmem_st_wait();
            named_bar_sync(pair_bar, 64);    // the half-0 arrive below releases PV over ALL channels
          }
        }

        {
          // p = exp2(s * scale - m_ref): packed fp32x2 FMA / ADD (one issue slot per two keys), MUFU ex2 per key
          const float neg_m = -m_ref;
          float sum0 = 0.f, sum1 = 0.f, sum2 = 0.f, sum3 = 0.f;
          uint32_t pk[32];
#pragma unroll
          for (int c = 0; c < 2; ++c) {
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              float x0, x1, x2, x3;
              ffma2(x0, x1, __uint_as_float(s[c][i + 0]), __uint_as_float(s[c][i + 1]), scale, scale, neg_m, neg_m);
              ffma2(x2, x3, __uint_as_float(s[c][i + 2]), __uint_as_float(s[c][i + 3]), scale, scale, neg_m, neg_m);
              float e0, e1, e2, e3;
              if ((kPolyGroups >> (i >> 2)) & 1) {      // compile-time pattern: this group of 4 keys skips the MUFU
                exp2_poly2(x0, x1, e0, e1);
                exp2_poly2(x2, x3, e2, e3);
              } else {
                e0 = VB_EXP2(x0); e1 = VB_EXP2(x1); e2 = VB_EXP2(x2); e3 = VB_EXP2(x3);
              }
              fadd2(sum0, sum1, sum0, sum1, e0, e1);
              fadd2(sum2, sum3, sum2, sum3, e2, e3);
              pk[c * 16 + (i >> 1) + 0] = pack_bf16x2(e0, e1);
              pk[c * 16 + (i >> 1) + 1] = pack_bf16x2(e2, e3);
            }
#ifdef VB_TIMELINE
            if (c == 0) { asm volatile("" ::: "memory"); if (row == 0 && h == 0) VB_STAMP(t, j, 7); }
#endif
          }
          if (blk > 0) {                     // the previous P_t (previous block or previous item) must have been consumed
            mbar_wait(&sm.bar_pv_done[t], (blk - 1) & 1u);
            tc_fence_after();
          }
          tmem_st32(p_addr, pk);            // P_t(j): keys [64 h, 64 h + 64) -> 32 columns of bf16 pairs
          l_sum += (sum0 + sum1) + (sum2 + sum3);
          if (row == 0 && h == 0) VB_STAMP(t, j, 3);
          tmem_st_wait();
          if (row == 0 && h == 0) VB_STAMP(t, j, 4);
        }
        tc_fence_before();
        mbar_arrive(h == 0 ? &bar_p_half[t] : &bar_p_ready[t]);   // PV over keys [0,64) / [64,128) may start
        if (row == 0 && h == 0) VB_STAMP(t, j, 5);
      }

      // ------------------------------------ epilogue ------------------------------------
      int item_again = item;
      asm volatile("" : "+r"(item_again));         // opaque copy: keeps the decode below from being hoisted above the loop
      const Item it = decode_item(p, item_again);
      const AttnSeg& seg = p.seg[it.seg_idx];
      const QPair& pair = it.pair;
      const AttnHead& head = it.head;
      const int batch = it.batch;
      s_xchg[t][h][row] = l_sum;
      named_bar_sync(pair_bar, 64);
      l_sum = s_xchg[t][0][row] + s_xchg[t][1][row];
      named_bar_sync(pair_bar, 64);               // both threads of the row have read: the next item may reuse xchg
      mbar_wait(&bar_o_full[t], items_t & 1u);
      tc_fence_after();
      const bool row_ok = row < pair.q_rows[t];
      const int krow = pair.q_row0[t] + row;      // row in kernel order
      const int stage = p.blend_stage;
      float w_head = 1.f;
      int64_t acc_off = 0;                        // blend mode: this head slot's rows of blend_acc
      if (stage != 0) {
        const int64_t bh = static_cast<int64_t>(batch) * p.blend_heads + head.wi;
        w_head = __ldg(p.blend_w + bh * 3 + p.blend_branch);
        acc_off = bh * p.blend_rows * kHeadDim + h * 64;
      }
      const float inv = w_head / l_sum;
      int n_dst = 0;
      int64_t dst_tok = 0;
      const int32_t* bc = nullptr;
      if (row_ok) {
        dst_tok = seg.out_map ? seg.out_map[batch * seg.out_map_stride_b + head.hk * seg.out_map_stride_h + krow] : krow;
        n_dst = 1;
        if (seg.bcast_map != nullptr && krow < seg.bcast_rows) {
          bc = seg.bcast_map + batch * seg.bcast_stride_b + head.hk * seg.bcast_stride_h +
               static_cast<int64_t>(krow) * seg.bcast_n;
          n_dst += seg.bcast_n;
        }
      }
      const int64_t head_off = batch * p.out_stride_b + head.ho * p.out_stride_h + h * 64;
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        uint32_t o[32];
        tmem_ld32(o_addr + c * 32, o);
        tmem_ld_wait();
        if (c == 1) {                               // O_t is in registers: PV(0) of the next item may overwrite it
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&sm.bar_o_free[t]);
        }
        for (int dsti = 0; dsti < n_dst; ++dsti) {
          int64_t tok = dsti == 0 ? dst_tok : static_cast<int64_t>(bc[dsti - 1]);
          // fused Ulysses "out" exchange: a video token's row goes to the rank that owns the token; a text row (tokens
          // behind the out_peer_count * out_peer_rows video tokens; HunyuanVideo) goes to EVERY rank, behind its video
          // rows — the all-gather over heads of hunyuan.py:186-187 as plain NVLink stores
          int pe = 0, pe_end = 1;
          if (p.out_peer_count > 0) {
            const int64_t video_rows = static_cast<int64_t>(p.out_peer_count) * p.out_peer_rows;
            if (tok < video_rows) {
              pe = static_cast<int>(tok / p.out_peer_rows);
              pe_end = pe + 1;
              tok -= static_cast<int64_t>(pe) * p.out_peer_rows;
            } else {
              pe_end = p.out_peer_count;
              tok = p.out_peer_rows + (tok - video_rows);
            }
          }
          for (; pe < pe_end; ++pe) {
            __nv_bfloat16* obase = p.out_peer_count > 0 ? p.out_peers[pe] : p.out;
            const int64_t off = head_off + tok * p.out_stride_s + c * 32;
            uint4* dst = reinterpret_cast<uint4*>(obase + off);
            float4* acc = reinterpret_cast<float4*>(p.blend_acc + acc_off + tok * kHeadDim + c * 32);   // blend mode only
#pragma unroll
            for (int q4i = 0; q4i < 4; ++q4i) {
              float f[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(o[q4i * 8 + i]) * inv;
              if (stage >= 2) {                      // add the fp32 partial sum of the earlier branches
                const float4 a0 = acc[2 * q4i], a1 = acc[2 * q4i + 1];
                f[0] += a0.x; f[1] += a0.y; f[2] += a0.z; f[3] += a0.w;
                f[4] += a1.x; f[5] += a1.y; f[6] += a1.z; f[7] += a1.w;
              }
              if (stage == 1 || stage == 2) {        // not the last branch: keep the sum in fp32
                acc[2 * q4i] = make_float4(f[0], f[1], f[2], f[3]);
                acc[2 * q4i + 1] = make_float4(f[4], f[5], f[6], f[7]);
              } else {
                uint4 v;
                v.x = pack_bf16x2(f[0], f[1]);
                v.y = pack_bf16x2(f[2], f[3]);
                v.z = pack_bf16x2(f[4], f[5]);
                v.w = pack_bf16x2(f[6], f[7]);
                dst[q4i] = v;
              }
            }
          }
        }
      }
      ++items_t;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  if (fn == nullptr) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess) {
      fn = reinterpret_cast<PFN_encodeTiled>(ptr);
    }
  }
  return fn;
}

// 4-D bf16 tensor map over (channel=128, token=n_rows, head, batch) with a (64, 128, 1, 1) box, SWIZZLE_128B.
int make_qkv_tensor_map(CUtensorMap* map, const void* base, int64_t n_rows, int64_t heads, int64_t batch,
                        int64_t stride_b, int64_t stride_h, int64_t stride_s) {
  PFN_encodeTiled enc = get_encode_fn();
  VB_REQUIRE(enc != nullptr, VB_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  VB_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0, VB_ERR_INVALID, "tensor base must be 16-byte aligned");
  VB_REQUIRE(stride_s % 8 == 0 && stride_h % 8 == 0 && stride_b % 8 == 0, VB_ERR_INVALID,
             "token/head/batch strides must be multiples of 8 elements (16 bytes)");
  cuuint64_t dims[4] = {static_cast<cuuint64_t>(kHeadDim), static_cast<cuuint64_t>(n_rows),
                        static_cast<cuuint64_t>(heads), static_cast<cuuint64_t>(batch)};
  // a size-1 dimension may carry a zero stride from the caller; TMA needs a positive multiple of 16 bytes
  auto fix = [](int64_t s) { return static_cast<cuuint64_t>((s > 0 ? s : 8) * 2); };
  cuuint64_t strides[3] = {fix(stride_s), fix(stride_h), fix(stride_b)};
  cuuint32_t box[4] = {64, static_cast<cuuint32_t>(kBlockN), 1, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  VB_REQUIRE(r == CUDA_SUCCESS, VB_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return VB_OK;
}

// `params.seg[i].cta_begin` must already hold the prefix sums; n_items = total work items over the segments.  The grid
// is one persistent CTA per SM (224 KB of shared memory: one CTA fits).
int launch_attn(const AttnTmaps& tmaps, const AttnParams& params_in, int n_items, cudaStream_t stream) {
  static bool configured[64] = {false};      // the attribute is per device
  static int sm_count[64] = {0};
  // Work counters: every launch takes the next of kCounters self-resetting counters of its device, so launches that
  // overlap on different streams never share one (a counter is reused kCounters launches later).
  constexpr unsigned kCounters = 256;
  static unsigned int* counters[64] = {nullptr};
  static unsigned next_counter[64] = {0};
  int dev = 0;
  VB_CUDA_OK(cudaGetDevice(&dev));
  VB_REQUIRE(dev >= 0 && dev < 64, VB_ERR_UNSUPPORTED, "device index %d out of range", dev);
  if (!configured[dev]) {
    VB_CUDA_OK(cudaFuncSetAttribute(vb_attn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    kAttnSmemBytes));
    VB_CUDA_OK(cudaDeviceGetAttribute(&sm_count[dev], cudaDevAttrMultiProcessorCount, dev));
    VB_CUDA_OK(cudaMalloc(&counters[dev], kCounters * sizeof(unsigned int)));
    VB_CUDA_OK(cudaMemset(counters[dev], 0, kCounters * sizeof(unsigned int)));
    configured[dev] = true;
  }
  if (n_items == 0) return VB_OK;
  AttnParams params = params_in;
  params.work_counter = counters[dev] + (next_counter[dev]++ % kCounters);
  const int n_ctas = std::min(n_items, sm_count[dev]);
  vb_attn_fwd_kernel<<<static_cast<unsigned>(n_ctas), kAttnThreads, kAttnSmemBytes, stream>>>(tmaps, params);
  VB_CUDA_OK(cudaGetLastError());
  return VB_OK;
}

}  // namespace vb
