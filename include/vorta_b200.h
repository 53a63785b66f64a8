/*
 * vorta_b200.h — C ABI of the B200-native routed sparse attention path.
 *
 * This is the drop-in boundary for the hot path of wenhao728/VORTA (reference citations are relative to the
 * reference tree).  The reference has no native code: every function below replaces a chain of PyTorch library
 * calls made by the reference's attention processors.  Only plain pointers, sizes and a cudaStream_t cross the
 * boundary; the caller owns every buffer; the only hidden state is the opaque vb_plan.
 *
 * All device tensors are bf16 unless stated.  Attention tensors are addressed with explicit element strides
 * (batch, head, token); the channel stride is 1 and head_dim is 128.  That covers both the reference's
 * (B, H, S, D) view and the (B, S, H, D) memory it is a transpose of (vorta/attention/wan.py:91-94), so no copy
 * is needed on either side of the call.
 *
 * Return value of every int function: VB_OK or a negative VB_ERR_* code; vb_last_error() gives the message of
 * the last failure on the calling thread.  The Python host maps VB_ERR_INVALID to ValueError (the reference's
 * _check_input, wan.py:181-193) and the others to RuntimeError.
 */
#ifndef VORTA_B200_H_
#define VORTA_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VB_OK 0
#define VB_ERR_INVALID (-1)     /* bad shapes / arguments (reference: ValueError) */
#define VB_ERR_CUDA (-2)        /* CUDA runtime or driver failure */
#define VB_ERR_UNSUPPORTED (-3) /* valid request this build does not implement */

/* branch ids == the reference's expert order (wan.py:352-354): 0 full, 1 coreset ("lowres"), 2 sliding tile */
#define VB_BRANCH_FULL 0
#define VB_BRANCH_CORESET 1
#define VB_BRANCH_SLIDING 2
#define VB_BRANCH_SKIP (-1)
/* Ulysses work units finer than a head (SURVEY.md section 8e): a full-attention head may be computed by two ranks, each
 * taking one half of the QUERY work items (the head's keys and values are needed by both).  A head slot with one of
 * these ids runs full attention for its half of the query rows only and writes only those output rows. */
#define VB_BRANCH_FULL_LO 3
#define VB_BRANCH_FULL_HI 4
/* general form: part k of n equal parts of the head's query work items (n = 2 .. 7); LO / HI are parts 0 / 1 of 2 */
#define VB_BRANCH_FULL_PART(k, n) (16 + 8 * (n) + (k))

#define VB_DTYPE_F32 0
#define VB_DTYPE_BF16 1

typedef void* vb_stream_t; /* cudaStream_t */
typedef struct vb_plan vb_plan;

const char* vb_last_error(void);
int vb_version(void);
/* 0 when the current device is sm_100 (B200); VB_ERR_UNSUPPORTED otherwise. The product has no other path. */
int vb_device_check(void);

/* ------------------------------------------------------------------------------------------------------
 * Plan: geometry-only state shared by all layers and steps.
 *   replaces get_group_info            (vorta/attention/coreset_select.py:15-60)
 *            create_sliding_tile_attn_mask_func + create_block_mask (vorta/attention/sliding_attn_flex.py:72-134)
 *            tile_layout / untile_layout index math (vorta/attention/tile.py:7-78)
 *            _check_input              (vorta/attention/wan.py:168-193, hunyuan.py:247-272)
 * ---------------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t latent[3];        /* (T, H, W) token grid */
  int32_t tile[3];          /* sliding-tile tile size */
  int32_t window[3];        /* sliding-tile window, in tiles; any size (clamped to the tile grid like the reference) */
  int32_t lowres_window[3]; /* coreset group window: g = product of the three, any g up to 4843 tokens (VB_ERR_UNSUPPORTED
                             * above: the selection kernel keeps a group's similarities in shared memory) */
  int32_t n_unpooled;       /* margins kept per group = int(g * (1 - reduction_rate)) - 1, computed by the host */
  int32_t text_len;         /* text tokens appended after the video tokens (HunyuanVideo); 0 for Wan */
  int32_t text_valid;       /* un-padded text tokens, <= text_len */
} vb_plan_desc;

int vb_plan_create(vb_plan** plan, const vb_plan_desc* desc);
void vb_plan_destroy(vb_plan* plan);
/* Change the un-padded text length (HunyuanVideo: per prompt, pipeline_hunyuan.py:380-392) without rebuilding. */
int vb_plan_set_text_valid(vb_plan* plan, int32_t text_valid);

enum {
  VB_PLAN_SEQ_LEN = 0,        /* S = T*H*W */
  VB_PLAN_NUM_GROUPS = 1,     /* G */
  VB_PLAN_GROUP_SIZE = 2,     /* g */
  VB_PLAN_CORESET_LEN = 3,    /* S_c = G * (1 + n_unpooled) */
  VB_PLAN_NUM_TILES = 4,
  VB_PLAN_TILE_TOKENS = 5,
  VB_PLAN_NUM_POOLED = 6,     /* dropped margins per group = g - 1 - n_unpooled */
  VB_PLAN_KEYS_PER_QUERY = 7, /* video keys each video query sees in the sliding branch */
  VB_PLAN_SLIDING_PAIRS = 8,  /* CTAs per head, sliding branch */
  VB_PLAN_SLIDING_RUNS = 9    /* entries in the sliding run table */
};
int vb_plan_query(const vb_plan* plan, int what, int64_t* value);

enum {
  VB_EXPORT_CENTER_INDICES = 0, /* int64 (G)        == LowresGroupInfo.center_indices[:, 0] */
  VB_EXPORT_MARGIN_INDICES = 1, /* int64 (G, g-1)   == LowresGroupInfo.margin_indices */
  VB_EXPORT_TILE_MAP = 2,       /* int32 (S)  tile-major position -> raster token (tile.py:26-29) */
  VB_EXPORT_TILE_WINDOW = 3,    /* int32 (num_tiles, 6) lo/hi tile coordinate of each query tile's window */
  VB_EXPORT_SLIDING_RUNS = 4,   /* int32 (runs, 2) start/len of key runs in tile-major order, one consecutive set per
                                 * window group (query tiles whose clamped windows coincide), then the text queries';
                                 * a set has at most nt[0] * nt[1] video runs (contiguous ones merged) + 1 text run */
  VB_EXPORT_SLIDING_ITEMS = 5,  /* int32 (items, 12) work items of the sliding branch in launch order: q_row0[2],
                                 * q_rows[2], run_begin, run_count, nq, n_blocks, split, run_begin2, run_count2, pad.
                                 * An item is up to two 128-row query tiles; query rows are positions of
                                 * VB_EXPORT_SLIDING_QUERY_MAP; split = 1 pairs two single-tile leftovers with different
                                 * windows, tile 1 then attends to runs [run_begin2, run_begin2 + run_count2) */
  VB_EXPORT_SLIDING_QUERY_MAP = 6 /* int32 (S + text_len) query position of the sliding branch -> raster token: window
                                 * group by window group, tiles of a group in tile order, tokens in tile-major order */
};
/* Copies a host-side table for parity tests; *bytes is in: capacity, out: size. */
int vb_plan_export(const vb_plan* plan, int what, void* dst, int64_t* bytes);

/* ------------------------------------------------------------------------------------------------------
 * Router head.  replaces Router.forward (vorta/patch/router.py:33-43) and the top-1 + threshold of
 * _get_routed_qkv (vorta/attention/wan.py:396-400).  fp32 arithmetic.  n_layers routers at once: weights are
 * addressed as w + l*w_layer_stride (elements), so one stacked buffer serves a whole denoise step.
 *   temb   (B, E)           temb_dtype
 *   w      (L, 3H, E), bias (L, 3H)   w_dtype
 *   scores (L, B, H, 3) fp32  out
 *   branch (L, H) int32 out: argmax_e scores[l, 0, h, e]; set to 0 when that score < tau (NaN tau: no threshold)
 * w_dtype VB_DTYPE_F32: fp32 arithmetic throughout (the contract of north_star).  w_dtype VB_DTYPE_BF16 (the reference's
 * inference default router_dtype): SiLU output, logits and scores are each rounded to bf16 as the reference's bf16
 * modules do, and the decision is taken on the rounded scores (ties -> lowest expert index); scores stay an fp32
 * buffer holding bf16-exact values.
 * ---------------------------------------------------------------------------------------------------- */
int vb_router_forward(const void* temb, int temb_dtype, const void* w, const void* bias, int w_dtype,
                      int64_t w_layer_stride, int64_t bias_layer_stride, int32_t n_layers, int32_t batch,
                      int32_t embed_dim, int32_t heads, float tau, float* scores, int32_t* branch,
                      vb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * Coreset selection.  replaces the similarity / argsort part of pool_sequence_by_similarity
 * (vorta/attention/coreset_select.py:91-113).  Dot products and norms accumulate in fp64.  Groups of up to 33 tokens
 * run one warp per group with a margin per lane; larger groups (up to 4843 tokens) one warp per group with the
 * similarities in shared memory.  Both return the same tables for the same group.
 *   x (B, H, S[+text], 128) bf16 with element strides; only the first S tokens are read
 *   unpooled_argsort (B, H, G, n_unpooled) int64, pooled_argsort (B, H, G, g-1-n_unpooled) int64:
 *        positions inside the group's margin list, ascending similarity (ties: lower position first)
 *   kept_tok    (B, H, S_c) int32: raster token of every pooled-sequence row ([centres | kept margins])
 *   dropped_tok (B, H, G, g-1-n_unpooled) int32: raster tokens that receive their centre's output
 * Any output pointer may be NULL.
 * ---------------------------------------------------------------------------------------------------- */
int vb_coreset_select(const vb_plan* plan, const void* x, int64_t stride_b, int64_t stride_h, int64_t stride_s,
                      int32_t batch, int32_t heads, int64_t* unpooled_argsort, int64_t* pooled_argsort,
                      int32_t* kept_tok, int32_t* dropped_tok, vb_stream_t stream);

/* Token tables from a MatchingResults pair (the index arithmetic of unpool_sequence_by_similarity,
 * coreset_select.py:159-166).  Inputs are the int64 argsort tables; outputs (any may be NULL):
 *   kept_tok (B, H, S_c + text_len), dropped_tok (B, H, G, n_pooled) as in vb_coreset_select, and
 *   unpool_src (B, H, S) int32: pooled-sequence row whose output every raster token receives. */
int vb_coreset_tables(const vb_plan* plan, const int64_t* unpooled_argsort, const int64_t* pooled_argsort,
                      int32_t batch, int32_t heads, int32_t* kept_tok, int32_t* dropped_tok, int32_t* unpool_src,
                      vb_stream_t stream);

/* Row gather: dst[b, h, i, :] = src[b, h, map[b, h, i], :] for i < n_rows (128 bf16 per row, 16-byte vectors).
 * replaces the index/gather/cat of pool_sequence_by_similarity (coreset_select.py:91-93,118-123) and
 * tile_layout (tile.py:7-41).  map strides of 0 share one map across heads / batches. */
int vb_gather_rows(const void* src, int64_t src_stride_b, int64_t src_stride_h, int64_t src_stride_s, void* dst,
                   int64_t dst_stride_b, int64_t dst_stride_h, int64_t dst_stride_s, const int32_t* map,
                   int64_t map_stride_b, int64_t map_stride_h, int32_t batch, int32_t heads, int32_t n_rows,
                   vb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * Routed attention for one self-attention layer.
 *   replaces WanAttnProcessorTripleEval / TripleTrain branches + combine (vorta/attention/wan.py:243-300,
 *   388-438) and the HunyuanVideo equivalents (hunyuan.py:136-189, 410-513, 612-661), i.e. SDPA,
 *   flex_attention with the sliding-tile BlockMask, pool / unpool, head gather / scatter and the blend.
 *
 *   q, k, v, out: (B, H, S + text_len, 128) bf16 addressed by element strides (batch, head, token)
 *   branch[H]  : VB_BRANCH_* per head (top-1 mode), ignored in blend mode
 *   weights    : NULL for top-1 mode (Eval processor); (B, H, 3) fp32 routing scores for blend mode (Train
 *                processor: every branch on every head, out = sum_e w[b,h,e] * O_e, summed in fp32 in the workspace
 *                and rounded to bf16 once; one launch per branch)
 *   flags      : VB_ATTN_* bits
 *   workspace  : device scratch of at least vb_attn_workspace_bytes(...) bytes
 * Text tokens (HunyuanVideo) sit after the video tokens; rows of padded text queries are written as zero.  The
 * un-padded text length is the plan's text_valid for every sample, or per sample (vb_attn_args::text_valid): then
 * output sample b equals a batch-1 call on sample b alone with a plan whose text_valid is text_valid[b], bit for bit,
 * and its rows [S + text_valid[b], S + text_len) are zero.  Routing is unchanged: one branch list for the batch (top-1),
 * or per-(batch, head) scores (blend).
 * ---------------------------------------------------------------------------------------------------- */
#define VB_ATTN_CORESET_KV_FROM_K 1u /* HunyuanVideo: K and V pooled with K's own matching (hunyuan.py:433-438) */

typedef struct {
  const void* q;
  const void* k;
  const void* v;
  void* out;
  int64_t q_stride[3]; /* batch, head, token (elements) */
  int64_t k_stride[3];
  int64_t v_stride[3];
  int64_t out_stride[3];
  int32_t batch;
  int32_t heads;
  const int32_t* branch; /* host pointer, heads entries */
  const float* weights;  /* host pointer, batch*heads*3 entries, or NULL */
  uint32_t flags;
  void* workspace;
  int64_t workspace_bytes;
  float* debug; /* bring-up only (read by -DVB_DEBUG_DUMP / -DVB_TIMELINE builds); NULL in production */
  /* Fused Ulysses "out" exchange over NVLink peer memory (top-1 mode only): when out_peer_count > 0, `out` is
   * ignored and the output row of token tok is stored into out_peer_ptrs[tok / out_peer_rows] at local token
   * tok % out_peer_rows, using out_stride as the strides of ONE peer buffer.  The pointers are peer-mapped device
   * addresses of every rank's receive buffer (this rank's own included).  out_peer_rows * out_peer_count must equal the
   * number of video tokens; with a text segment (HunyuanVideo) each buffer has text_len more rows behind its
   * out_peer_rows video rows, and the row of text token j is stored into row out_peer_rows + j of EVERY peer (the head
   * all-gather of hunyuan.py:186-187); rows of padded text queries are not written — the owner zeroes them. */
  void* out_peer_ptrs[8];
  int32_t out_peer_count;
  int32_t out_peer_rows;
  /* Optional (host pointer, heads entries, or NULL = identity): head index along `out`'s head stride that receives
   * the output of local head h.  Lets a rank that holds an arbitrary, cost-balanced subset of the layer's heads
   * (Ulysses, SURVEY.md section 8e) write each head where the token owner expects it.  Padded text rows are zeroed in
   * the same heads: a VB_BRANCH_SKIP slot writes nothing, and of a head split into query parts only the last part
   * (k = n - 1) writes them, so the parts of a head own disjoint rows. */
  const int32_t* out_heads;
  /* Blend mode with the routing scores left on the device: (batch, heads, 3) fp32, same meaning as `weights`; when set,
   * `weights` is ignored and no host copy of the scores is needed (the reference blends device tensors, wan.py:296-300). */
  const float* weights_device;
  /* Optional (host pointer, batch entries, or NULL = the plan's text_valid for every sample): the un-padded text length
   * of each sample, each within [0, text_len] (else VB_ERR_INVALID).  Samples with the same length share one schedule
   * and one segment of the launch; the schedules of lengths other than the plan's are built on first use and cached in
   * the plan (a bounded number of lengths, freed by vb_plan_destroy).  Prompts of different lengths can so be batched,
   * e.g. num_videos_per_prompt > 1 or several prompts in one forward. */
  const int32_t* text_valid;
} vb_attn_args;

int64_t vb_attn_workspace_bytes(const vb_plan* plan, int32_t batch, int32_t heads);
int vb_attn_fwd(vb_plan* plan, const vb_attn_args* args, vb_stream_t stream);

/* Dense softmax(Q K^T / sqrt(128)) V with independent query / key lengths: the base processor
 * (WanAttnProcessor2_0._attn, wan.py:142-144: cross attention, I2V image keys, use_original_attn).  Same kernel,
 * one key run [0, n_k).  q, out: (B, H, n_q, 128); k, v: (B, H, n_k, 128); element strides (batch, head, token). */
int vb_attn_dense(const void* q, const void* k, const void* v, void* out, const int64_t* q_stride,
                  const int64_t* k_stride, const int64_t* v_stride, const int64_t* out_stride, int32_t batch,
                  int32_t heads, int32_t n_q, int32_t n_k, vb_stream_t stream);

/* Counters for bench.py: number of kernels this library launched on the calling thread since the last reset,
 * and the algorithmic attention FLOPs (BASELINE.md section 3 formulas) they covered. */
void vb_stats_reset(void);
int64_t vb_stats_launches(void);
double vb_stats_attn_flops(void);

/* ------------------------------------------------------------------------------------------------------
 * Fused elementwise kernels of the DiT block around the path (SURVEY.md section 8f rows 1-2; "next" rows).
 * Rows are tokens, bf16, contiguous, `dim` channels (multiple of 8, <= 8192); fp32 math; one read + one write.
 * x, y, out and the bf16 weights (and headnorm's cos / sin tables) must be 16-byte aligned: VB_ERR_INVALID otherwise.
 *   vb_block_ln_modulate : out = (LayerNorm(x) [* weight + bias]) [* (1 + scale) + shift]
 *        replaces norm1/norm3 + adaLN modulate and norm2 (vorta/patch/modeling_wan.py:205-206, 226, 232-234);
 *        weight/bias fp32 (dim) or NULL (each applies on its own); scale/shift fp32 (batch, dim) or NULL;
 *        batch = row / rows_per_batch
 *   vb_block_gate_residual: out = x + y * gate  (gate fp32 (batch, dim), NULL = plain add)   (:225, :229, :238)
 *   vb_block_rmsnorm_rope : RMSNorm over the whole row * weight (bf16, dim), then the complex rotation of channel
 *        pairs of every 128-wide head by (cos, sin) fp32 (tokens_per_batch, 64); token = row % tokens_per_batch.
 *        NULL tables = norm only.  replaces norm_q/norm_k + apply_rotary_emb (vorta/attention/wan.py:85-100, 34-37)
 * ---------------------------------------------------------------------------------------------------- */
int vb_block_ln_modulate(const void* x, const float* weight, const float* bias, const float* scale, const float* shift,
                         void* out, int64_t rows, int32_t dim, int32_t rows_per_batch, float eps, vb_stream_t stream);
int vb_block_gate_residual(const void* x, const void* y, const float* gate, void* out, int64_t rows, int32_t dim,
                           int32_t rows_per_batch, vb_stream_t stream);
int vb_block_rmsnorm_rope(const void* x, const void* weight, const float* cos_tab, const float* sin_tab, void* out,
                          int64_t rows, int32_t dim, int32_t tokens_per_batch, float eps, vb_stream_t stream);

/* HunyuanVideo Q / K prologue in one pass: per-head RMSNorm (weight bf16 (128), NULL = none) over every 128-channel
 * head of x (batch, rows, heads*128) bf16 contiguous, then the rotation of channel pairs (2i, 2i+1) by
 * (cos, sin)[row][i] (fp32 (rope_rows, 64), NULL = none) for rows < rope_rows (the video tokens; text rows are not
 * rotated), written to rows [dst_row0, dst_row0 + rows) of out (batch, dst_rows, heads*128) — the joint
 * [video | text] sequence the attention reads.  out may alias x when dst_rows == rows and dst_row0 == 0.
 * replaces _step_qk_norm + _step_rotary_emb + the torch.cat of _step_encoder_to_qkv_and_concat
 * (vorta/attention/hunyuan.py:62-134; diffusers' apply_rotary_emb(use_real=True, use_real_unbind_dim=-1)). */
int vb_block_headnorm_rope(const void* x, const void* weight, const float* cos_tab, const float* sin_tab, void* out,
                           int32_t batch, int32_t rows, int32_t heads, int32_t rope_rows, int32_t dst_rows,
                           int32_t dst_row0, float eps, vb_stream_t stream);

/* Live timing of the attention kernel for the roofline line of bench.py: while enabled, every launch of the
 * tcgen05 attention kernel is bracketed by CUDA events on its own stream; vb_timing_collect waits for them and
 * returns the summed kernel time (ms), the number of launches and their algorithmic FLOPs, then clears. */
void vb_timing_enable(int on);
int vb_timing_collect(double* kernel_ms, int64_t* launches, double* flops);
/* The same, split by caller: index VB_TIMING_ROUTED = launches made by vb_attn_fwd (the routed self-attention of a
 * layer, all branches), VB_TIMING_DENSE = launches made by vb_attn_dense (cross attention, I2V image keys,
 * use_original_attn).  Each array has VB_TIMING_KINDS entries. */
#define VB_TIMING_ROUTED 0
#define VB_TIMING_DENSE 1
#define VB_TIMING_KINDS 2
int vb_timing_collect_kinds(double* kernel_ms, int64_t* launches, double* flops);

/* ------------------------------------------------------------------------------------------------------
 * Ulysses sequence parallelism helpers (vorta/ulysses/utils.py:15-93).  The exchange itself is an NCCL
 * all-to-all issued by the host through torch.distributed; these kernels produce / consume its buffers.
 *   pack  : x (S_loc, H, 128) token-major -> send (P, S_loc, H/P, 128), chunk p = heads [p*H/P, (p+1)*H/P)
 *   unpack: recv (P, S_loc, H/P, 128)     -> y (S_loc, H, 128)
 * The receive buffer of the "in" direction, (P*S_loc, H/P, 128), and the send buffer of the "out" direction are
 * consumed / produced by vb_attn_fwd directly through its strides, so each direction needs one pass only.
 *
 * head_at (host pointer, H entries, or NULL): slot p*H/P + i of the exchanged layout holds head head_at[p*H/P + i].
 * NULL is the reference's contiguous chunking (ulysses/utils.py:60-66).  Because every rank knows the whole step's
 * routing before the first block runs, the host can pass a permutation that balances the per-rank attention cost
 * (full : coreset : sliding heads differ ~ 6 : 1.6 : 1); it must be a permutation of [0, H), H <= 128, identical on
 * every rank and for the pack and unpack sides of one layer.
 * ---------------------------------------------------------------------------------------------------- */
int vb_ulysses_pack_heads(const void* x, void* send, int32_t s_loc, int32_t heads, int32_t world, int32_t n_tensors,
                          int64_t x_tensor_stride, int64_t send_tensor_stride, const int32_t* head_at,
                          vb_stream_t stream);
/* q, k, v: (S_loc, H, 128), each with its own element strides stride_s[3] (token) / stride_h[3] (head) ->
 * send (3, P, S_loc, H/P, 128) in one pass (the reference makes two transposed copies per tensor,
 * ulysses/utils.py:68-74,89). */
int vb_ulysses_pack_qkv(const void* q, const void* k, const void* v, const int64_t* stride_s, const int64_t* stride_h,
                        void* send, int32_t s_loc, int32_t heads, int32_t world, const int32_t* head_at,
                        vb_stream_t stream);
int vb_ulysses_unpack_heads(const void* recv, void* y, int32_t s_loc, int32_t heads, int32_t world,
                            const int32_t* head_at, vb_stream_t stream);
/* Fused Ulysses "in" exchange over NVLink peer memory, replacing pack + all-to-all (ulysses/utils.py:60-81): entry e
 * stores head entry_head[e] of this rank's S_loc tokens of q, k, v straight into slot entry_slot[e] of peer
 * entry_peer[e]'s receive buffer peer_qkv[entry_peer[e]], laid out (3, rows_total, slots, 128) with this rank's tokens
 * at rows [rank*S_loc, (rank+1)*S_loc).  Ranks may hold different numbers of heads, and a head may be sent to two peers
 * (VB_BRANCH_FULL_LO / _HI units).  n_entries <= 128; host pointers. */
int vb_ulysses_scatter_qkv_slots(const void* q, const void* k, const void* v, const int64_t* stride_s,
                                 const int64_t* stride_h, void* const* peer_qkv, int64_t rows_total, int32_t s_loc,
                                 int32_t slots, int32_t world, int32_t rank, const int32_t* entry_peer,
                                 const int32_t* entry_slot, const int32_t* entry_head, int32_t n_entries,
                                 vb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* VORTA_B200_H_ */
