// vb_common.cuh — shared host-side helpers (error plumbing) and kernel-facing parameter structs.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/vorta_b200.h"

namespace vb {

// thread-local last-error string returned by vb_last_error()
void set_error(const char* fmt, ...);
const char* get_error();

#define VB_CUDA_OK(expr)                                                                        \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess) {                                                                    \
      ::vb::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));    \
      return VB_ERR_CUDA;                                                                       \
    }                                                                                           \
  } while (0)

#define VB_REQUIRE(cond, code, ...)        \
  do {                                     \
    if (!(cond)) {                         \
      ::vb::set_error(__VA_ARGS__);        \
      return (code);                       \
    }                                      \
  } while (0)

constexpr int kHeadDim = 128;     // D of every supported model (Wan 1.3B/14B, HunyuanVideo)
constexpr int kBlockM = 128;      // query rows per MMA tile (one TMEM lane per row)
constexpr int kBlockN = 128;      // keys per MMA tile
constexpr int kMaxHeads = 64;     // heads per attention launch
constexpr int kMaxHeadTable = 128; // heads per Ulysses exchange (slot -> head table passed by value)

// One work item: up to two 128-row query tiles.  Normally both tiles attend to the SAME key/value run list (they are
// neighbouring tiles of one logical query range) and every K/V block staged in shared memory feeds both.  A "split"
// item (split != 0) pairs two single-tile leftovers of DIFFERENT ranges: tile 1 has its own run list (run_begin2 /
// run_count2, same number of 128-key blocks), the K/V ring then carries K0 V0 K1 V1 per block step, and both tile
// pipelines of the CTA stay busy where a single tile would leave one idle.
struct QPair {
  int32_t q_row0[2];   // first row of each query tile, in kernel order
  int32_t q_rows[2];   // valid rows in each tile (<= 128)
  int32_t run_begin;   // first entry in KvRun[] (tile 0, and tile 1 unless split)
  int32_t run_count;   // number of runs
  int32_t nq;          // 1 or 2
  int32_t n_blocks;    // 128-key blocks of the run list (per tile)
  int32_t split;       // 0: shared run list; 1: tile 1 uses run_begin2 / run_count2
  int32_t run_begin2, run_count2;
  int32_t pad;
};
static_assert(sizeof(QPair) == 48, "QPair layout");
// A contiguous range of keys (kernel order) every query of the pair attends to.
struct KvRun {
  int32_t start;
  int32_t len;
};
struct AttnHead {
  int32_t hk;       // head coordinate inside the Q/K/V tensor maps
  int32_t ho;       // head index in the output tensor
  int32_t wi;       // blend mode: head index into AttnParams::blend_w (top-1 mode scales by 1)
};

// One branch of a layer inside an attention launch: its own work table, Q/K/V tensor maps (AttnTmaps::m[i]) and row
// maps.  A top-1 routed layer runs its (up to) three branches as three segments of ONE launch, longest CTAs first,
// so the tail of one branch is filled by the next instead of idling the SMs between launches.
constexpr int kMaxSegments = 8;     // full, up to five kinds of query parts of full heads, coreset, sliding
struct AttnSeg {
  const QPair* pairs;
  const KvRun* runs;
  const int32_t* out_map;       // kernel row -> output token, nullptr = identity
  int64_t out_map_stride_h;     // per-head stride of out_map (0 = shared by all heads), indexed by hk
  int64_t out_map_stride_b;
  const int32_t* bcast_map;     // rows < bcast_rows also write bcast_n copies (coreset unpool)
  int64_t bcast_stride_h, bcast_stride_b;
  int32_t bcast_rows, bcast_n;
  int32_t n_pairs, n_heads;     // CTAs of the segment = n_pairs * n_heads * n_batch, pair index fastest
  int32_t head0;                // the segment's heads are AttnParams::heads[head0 .. head0 + n_heads)
  int32_t cta_begin;            // linear item index of the segment's first work item
};

struct AttnParams {
  __nv_bfloat16* out;
  int64_t out_stride_b, out_stride_h, out_stride_s;   // elements
  // Ulysses "peer" output: when out_peer_count > 0 token tok belongs to rank tok / out_peer_rows and its row is stored
  // straight into that rank's buffer over NVLink (out_stride_* then describe ONE peer buffer, token index local)
  __nv_bfloat16* out_peers[8];
  int32_t out_peer_count, out_peer_rows;
  float scale_log2;             // log2(e) / sqrt(D)
  int32_t n_items;              // work items of the launch (all segments)
  unsigned int* work_counter;   // device counter handing out items beyond the first gridDim.x; 0 before and after a launch
  int32_t n_seg;
  // Blend (Train) mode, out = sum_e w[b,h,e] * O_e (wan.py:296-300): the three branches run as three launches, stage =
  // 1, 2, 3.  Stage 1 stores w * O in fp32 into blend_acc, stage 2 adds to it, stage 3 adds and writes the bf16 output, so
  // the sum is formed in fp32 and rounded once.  blend_w: device (batch, blend_heads, 3) fp32 routing scores.
  const float* blend_w;
  float* blend_acc;             // fp32 (batch, blend_heads, blend_rows, 128): head slot wi, output token
  int32_t blend_stage;          // 0 = top-1 mode
  int32_t blend_heads, blend_branch, blend_rows;
  float* dbg;                   // optional debug dump (bring-up only), nullptr in production
  AttnSeg seg[kMaxSegments];
  AttnHead heads[kMaxHeads];
};

struct AttnTmaps {
  CUtensorMap m[kMaxSegments][3];   // q, k, v of each segment (4-D: channel, row, head, batch)
};

// Source head of each processed head slot, passed BY VALUE inside the launch parameters (<= 64 bytes): a layer's
// head lists change with the routing of every layer and used to cost a pageable host->device copy each.
struct HeadList {
  uint8_t h[kMaxHeads];
  int32_t used;                // 0 = identity (slot i reads head i)
  __host__ __device__ int head(int slot) const { return used ? h[slot] : slot; }
};

// Zeroing of rows [row0, row0 + n_rows) of the listed output heads of every batch element, the head list passed BY
// VALUE like HeadList (vb_kernels.cu)
constexpr int kMaxZeroHeads = 256;
struct ZeroRowsParams {
  __nv_bfloat16* out;
  int64_t stride_b, stride_h, stride_s;
  int32_t batch, n_heads, row0, n_rows;
  int32_t head[kMaxZeroHeads];  // output head index of each listed head
};

// Coreset selection launch parameters (vb_kernels.cu)
struct SelectParams {
  const __nv_bfloat16* x;
  int64_t stride_b, stride_h, stride_s;
  const int32_t* center_tok;   // (G)
  const int32_t* margin_tok;   // (G, g-1)
  HeadList head_list;          // source head of each processed head slot
  int32_t batch, heads, G, n_margin, n_unpooled, seq_len, text_len;
  int64_t* unpooled_argsort;   // (B, heads, G, n_u)
  int64_t* pooled_argsort;     // (B, heads, G, n_margin - n_u)
  int32_t* kept_tok;           // (B, heads, S_c + text_len)
  int32_t* dropped_tok;        // (B, heads, G, n_margin - n_u)
};
// Token tables from int64 matching tables (vb_kernels.cu)
struct TablesParams {
  const int64_t* unpooled_argsort;
  const int64_t* pooled_argsort;
  const int32_t* center_tok;
  const int32_t* margin_tok;
  int32_t batch, heads, G, n_margin, n_unpooled, seq_len, text_len;
  int32_t* kept_tok;
  int32_t* dropped_tok;
  int32_t* unpool_src;
};
// Row gather launch parameters: up to three tensors share one row map (vb_kernels.cu)
struct GatherParams {
  const __nv_bfloat16* src[3];
  __nv_bfloat16* dst[3];
  int64_t src_stride[3][3];   // [tensor][b, h, s]
  int64_t dst_stride[3];      // b, h, s (shared by the tensors)
  const int32_t* map;
  const int32_t* map0;        // optional: tensor 0 follows its own row map (same strides)
  int64_t map_stride_b, map_stride_h;
  HeadList head_list;
  int32_t n_tensors, batch, heads, n_rows;
};

}  // namespace vb
