// vb_api.cu — the C ABI (include/vorta_b200.h): plan construction (closed-form schedules, no mask tensors),
// per-layer orchestration of the three branches, and thin wrappers over the kernels.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <array>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <vector>

#include <nvtx3/nvToolsExt.h>     // header-only NVTX v3: ranges cost a few ns unless a profiler is attached

#include "vb_common.cuh"

namespace vb {

// NVTX range over one host-side phase of the path (visible in nsys / ncu --nvtx; SURVEY.md section 5)
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

// ---- error plumbing -----------------------------------------------------------------------------
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* get_error() { return g_err; }

static thread_local int64_t g_launches = 0;
static thread_local double g_flops = 0.0;
// optional live timing of the attention kernel (bench.py roofline): event pairs on the launching stream
static thread_local bool g_timing = false;
struct TimedLaunch {
  cudaEvent_t ev0, ev1;
  int kind;        // VB_TIMING_ROUTED (vb_attn_fwd) or VB_TIMING_DENSE (vb_attn_dense)
  double flops;
};
static thread_local std::vector<TimedLaunch> g_events;

// ---- kernels implemented in the other translation units -----------------------------------------
int launch_coreset_select(const SelectParams& p, cudaStream_t stream);
int launch_gather_rows(const GatherParams& p, cudaStream_t stream);
int launch_coreset_tables(const TablesParams& p, cudaStream_t stream);
int launch_zero_rows(const ZeroRowsParams& p, cudaStream_t stream);
int launch_router(const void* temb, int temb_dtype, const void* w, const void* bias, int w_dtype,
                  int64_t w_layer_stride, int64_t bias_layer_stride, int n_layers, int batch, int embed_dim,
                  int heads, float tau, float* scores, int32_t* branch, cudaStream_t stream);
int launch_ulysses_permute(const void* src, void* dst, int s_loc, int heads, int world, int n_tensors,
                           int64_t src_tensor_stride, int64_t dst_tensor_stride, int pack, const int32_t* head_at,
                           cudaStream_t stream);
int launch_ulysses_pack_qkv(const void* q, const void* k, const void* v, const int64_t* stride_s,
                            const int64_t* stride_h, void* send, int s_loc, int heads, int world,
                            const int32_t* head_at, cudaStream_t stream);
int launch_ln_modulate(const void* x, const float* w, const float* b, const float* scale, const float* shift, void* out,
                       int64_t rows, int dim, int rows_per_batch, float eps, cudaStream_t stream);
int launch_gate_residual(const void* x, const void* y, const float* gate, void* out, int64_t rows, int dim,
                         int rows_per_batch, cudaStream_t stream);
int launch_rmsnorm_rope(const void* x, const void* weight, const float* cs, const float* sn, void* out, int64_t rows,
                        int dim, int tokens_per_batch, float eps, cudaStream_t stream);
int launch_headnorm_rope(const void* x, const void* weight, const float* cs, const float* sn, void* out, int batch,
                         int rows, int heads, int rope_rows, int dst_rows, int dst_row0, float eps,
                         cudaStream_t stream);
int launch_ulysses_scatter_slots(const void* q, const void* k, const void* v, const int64_t* stride_s,
                                 const int64_t* stride_h, void* const* peer_qkv, int64_t rows_total, int s_loc, int slots,
                                 int world, int rank, const int32_t* entry_peer, const int32_t* entry_slot,
                                 const int32_t* entry_head, int n_entries, cudaStream_t stream);
int make_qkv_tensor_map(CUtensorMap* map, const void* base, int64_t n_rows, int64_t heads, int64_t batch,
                        int64_t stride_b, int64_t stride_h, int64_t stride_s);
int launch_attn(const AttnTmaps& tmaps, const AttnParams& params, int n_ctas, cudaStream_t stream);


// ---- schedule tables ----------------------------------------------------------------------------
struct Schedule {
  std::vector<QPair> pairs;
  std::vector<KvRun> runs;
  QPair* d_pairs = nullptr;
  KvRun* d_runs = nullptr;
  double flops_per_head = 0.0;   // 4 * D * sum_q keys(q)

  void add_query_range(int row0, int n_rows, int run_begin, int run_count, int64_t keys) {
    // split [row0, row0+n_rows) into 128-row tiles, two per work item
    int n_blocks = 0;
    for (int r = 0; r < run_count; ++r) n_blocks += (runs[run_begin + r].len + kBlockN - 1) / kBlockN;
    for (int off = 0; off < n_rows; off += 2 * kBlockM) {
      QPair qp;
      memset(&qp, 0, sizeof(qp));
      qp.run_begin = run_begin;
      qp.run_count = run_count;
      qp.n_blocks = n_blocks;
      qp.q_row0[0] = row0 + off;
      qp.q_rows[0] = std::min(kBlockM, n_rows - off);
      qp.nq = 1;
      if (off + kBlockM < n_rows) {
        qp.q_row0[1] = row0 + off + kBlockM;
        qp.q_rows[1] = std::min(kBlockM, n_rows - off - kBlockM);
        qp.nq = 2;
      }
      pairs.push_back(qp);
    }
    flops_per_head += 4.0 * kHeadDim * static_cast<double>(n_rows) * static_cast<double>(keys);
  }
  // Single-tile items leave one of the CTA's two tile pipelines idle.  When EVERY item of the branch is a single tile
  // (sliding tiles of <= 128 tokens, e.g. the 120-token tiles of Wan-1.3B), pair two of them that walk the same number
  // of key blocks into ONE split item: tile 1 keeps its own run list (measured 724 -> 768 TFLOP/s, profiles/r2b_*).
  // A split item stages every K/V block for one tile only, i.e. twice the ring traffic per MMA; mixed with ordinary
  // two-tile items (the odd last slot of a window group) that cost more than the idle pipeline it fills
  // (1140 -> 986 TFLOP/s), so those leftovers stay single.  With window groups (vb_plan::groups) all-single schedules
  // only arise when every group is one tile of <= 128 tokens.  Then order the items longest first (stable): the
  // persistent kernel hands them out greedily.
  void finalize() {
    bool all_single = !pairs.empty();
    for (const QPair& qp : pairs) all_single = all_single && qp.nq == 1;
    if (all_single) {
      std::vector<QPair> out;
      std::vector<int> open_by_blocks;        // index in `out` of an unpaired single-tile item, per block count
      for (const QPair& qp : pairs) {
        if (qp.nq != 1) {
          out.push_back(qp);
          continue;
        }
        int partner = -1;
        for (size_t i = 0; i < open_by_blocks.size(); ++i)
          if (out[open_by_blocks[i]].n_blocks == qp.n_blocks) {
            partner = static_cast<int>(i);
            break;
          }
        if (partner < 0) {
          open_by_blocks.push_back(static_cast<int>(out.size()));
          out.push_back(qp);
        } else {
          QPair& a = out[open_by_blocks[partner]];
          a.q_row0[1] = qp.q_row0[0];
          a.q_rows[1] = qp.q_rows[0];
          a.nq = 2;
          a.split = (qp.run_begin == a.run_begin && qp.run_count == a.run_count) ? 0 : 1;
          a.run_begin2 = qp.run_begin;
          a.run_count2 = qp.run_count;
          open_by_blocks.erase(open_by_blocks.begin() + partner);
        }
      }
      pairs.swap(out);
    }
    std::stable_sort(pairs.begin(), pairs.end(), [](const QPair& a, const QPair& b) {
      return a.n_blocks * a.nq > b.n_blocks * b.nq;
    });
  }
  int upload() {
    release();
    if (!pairs.empty()) {
      VB_CUDA_OK(cudaMalloc(&d_pairs, pairs.size() * sizeof(QPair)));
      VB_CUDA_OK(cudaMemcpy(d_pairs, pairs.data(), pairs.size() * sizeof(QPair), cudaMemcpyHostToDevice));
    }
    if (!runs.empty()) {
      VB_CUDA_OK(cudaMalloc(&d_runs, runs.size() * sizeof(KvRun)));
      VB_CUDA_OK(cudaMemcpy(d_runs, runs.data(), runs.size() * sizeof(KvRun), cudaMemcpyHostToDevice));
    }
    return VB_OK;
  }
  void release() {
    if (d_pairs) cudaFree(d_pairs);
    if (d_runs) cudaFree(d_runs);
    d_pairs = nullptr;
    d_runs = nullptr;
  }
  void clear() {
    pairs.clear();
    runs.clear();
    flops_per_head = 0.0;
  }
};

// The schedules that depend on the un-padded text length: full, coreset and sliding (queries in window-group order).
struct TextSchedules {
  int32_t text_valid = 0;
  Schedule full, coreset, sliding;
  int64_t keys_per_query = 0;   // video keys of a video query of the first window group (sliding)
  uint64_t last_use = 0;
  void release() {
    full.release();
    coreset.release();
    sliding.release();
  }
};
constexpr size_t kMaxCachedTextLengths = 16;

}  // namespace vb

using namespace vb;

struct vb_plan {
  vb_plan_desc d;
  int S = 0, G = 0, g = 0, n_u = 0, n_p = 0, S_c = 0;
  int nt[3] = {0, 0, 0}, n_tiles = 0, tile_tokens = 0;
  bool has_device = false;
  // host tables
  std::vector<int64_t> center, margin;        // (G), (G, g-1)
  std::vector<int32_t> tile_map;              // (S + text_len): tile-major position -> raster token
  std::vector<int32_t> tile_window;           // (n_tiles, 6)
  // Query tiles whose (clamped) windows coincide — the two outermost tiles along every axis — see exactly the same keys.
  // The sliding branch lays its QUERY rows out window group by window group (keys stay tile-major), so a group of s tiles
  // is cut into ceil(s * tau / 128) query slots instead of s * ceil(tau / 128): Wan-14B's 432-token tiles fill 606
  // slots instead of 700, and Wan-1.3B's 120-token tiles pair up inside ordinary two-tile items that share one K/V stream.
  struct WindowGroup {
    int lo[3], hi[3];
    int row0, n_tiles;                        // first row in query order, tiles in the group
  };
  std::vector<WindowGroup> groups;
  std::vector<int32_t> query_map;             // (S + text_len): sliding-branch query position -> raster token
  TextSchedules text;                         // for d.text_valid
  // Per-sample text lengths (vb_attn_args::text_valid): the schedules of other lengths, built on first use and kept
  // for later calls, at most kMaxCachedTextLengths of them between calls (least recently used dropped first)
  std::vector<std::unique_ptr<TextSchedules>> other_text;
  uint64_t text_clock = 0;
  std::mutex text_mutex;                      // guards other_text for calls that pass per-sample lengths
  // device tables
  int32_t* d_center_tok = nullptr;
  int32_t* d_margin_tok = nullptr;
  int32_t* d_tile_map = nullptr;
  int32_t* d_query_map = nullptr;
};

static void window_range(int q, int n, int w, int& lo, int& hi) {
  // reference: sliding_attn_flex.py:118-127; torch.clamp(min > max) returns max
  const int half = w / 2;
  const int cmin = half, cmax = (n - 1) - half;
  int c = q;
  if (cmin > cmax) c = cmax;
  else c = std::min(std::max(q, cmin), cmax);
  lo = std::max(0, c - half);
  hi = std::min(n - 1, c + half);
}

// The schedules of text length tv (the plan's text_valid, or one sample's length) into ts.
static int build_text_dependent(const vb_plan* pl, int tv, TextSchedules& ts) {
  const int S = pl->S;
  ts.text_valid = tv;
  // ---- full: every query sees [0, S + text_valid) (wan.py:142-144; hunyuan.py:169-176)
  ts.full.clear();
  ts.full.runs.push_back({0, S + tv});
  ts.full.add_query_range(0, S + tv, 0, 1, S + tv);
  // ---- coreset: same over the pooled sequence [centres | kept margins | text] (hunyuan.py:440-448)
  ts.coreset.clear();
  ts.coreset.runs.push_back({0, pl->S_c + tv});
  ts.coreset.add_query_range(0, pl->S_c + tv, 0, 1, pl->S_c + tv);
  // ---- sliding tile (sliding_attn_flex.py:93-127): keys in tile-major order; one query range per window group
  ts.sliding.clear();
  const int tau = pl->tile_tokens;
  Schedule& sc = ts.sliding;
  for (const vb_plan::WindowGroup& g : pl->groups) {
    const int run_begin = static_cast<int>(sc.runs.size());
    int64_t keys = 0;
    for (int x = g.lo[0]; x <= g.hi[0]; ++x)
      for (int y = g.lo[1]; y <= g.hi[1]; ++y) {
        KvRun r;
        r.start = ((x * pl->nt[1] + y) * pl->nt[2] + g.lo[2]) * tau;
        r.len = (g.hi[2] - g.lo[2] + 1) * tau;
        keys += r.len;
        if (static_cast<int>(sc.runs.size()) > run_begin && sc.runs.back().start + sc.runs.back().len == r.start) {
          sc.runs.back().len += r.len;   // contiguous in tile-major order: merge
        } else {
          sc.runs.push_back(r);
        }
      }
    if (tv > 0) {   // video queries see the valid text keys (:112)
      sc.runs.push_back({S, tv});
      keys += tv;
    }
    const int run_count = static_cast<int>(sc.runs.size()) - run_begin;   // any number: walked from global memory
    sc.add_query_range(g.row0, g.n_tiles * tau, run_begin, run_count, keys);
    if (g.row0 == 0) ts.keys_per_query = keys - tv;
  }
  if (tv > 0) {   // valid text queries see every non-pad key (:108) as two runs, video and text: one run [0, S + tv)
                  // would cut the keys into different 128-key blocks and so change these rows' output bits
    const int run_begin = static_cast<int>(sc.runs.size());
    sc.runs.push_back({0, S});
    sc.runs.push_back({S, tv});
    sc.add_query_range(S, tv, run_begin, 2, S + tv);
  }
  ts.full.finalize();
  ts.coreset.finalize();
  ts.sliding.finalize();
  if (pl->has_device) {
    int rc;
    if ((rc = ts.full.upload()) != VB_OK) return rc;
    if ((rc = ts.coreset.upload()) != VB_OK) return rc;
    if ((rc = ts.sliding.upload()) != VB_OK) return rc;
  }
  return VB_OK;
}

// The schedules of every length in `lengths` (distinct, each within [0, text_len]) into out[i]: the plan's own for its
// text_valid, a cached set otherwise, built on first use.  When new sets would take the cache beyond
// kMaxCachedTextLengths, the least recently used sets that this call does not need are dropped first, after a device
// synchronize (earlier launches may still read their tables).  Caller holds pl->text_mutex.
static int text_schedules(vb_plan* pl, const std::vector<int32_t>& lengths, std::vector<const TextSchedules*>& out) {
  out.assign(lengths.size(), nullptr);
  const uint64_t now = ++pl->text_clock;
  size_t missing = 0;
  for (size_t i = 0; i < lengths.size(); ++i) {
    if (lengths[i] == pl->d.text_valid) {
      out[i] = &pl->text;
      continue;
    }
    for (const auto& e : pl->other_text)
      if (e->text_valid == lengths[i]) {
        e->last_use = now;
        out[i] = e.get();
      }
    if (out[i] == nullptr) ++missing;
  }
  if (missing > 0 && pl->other_text.size() + missing > kMaxCachedTextLengths) {
    if (pl->has_device) VB_CUDA_OK(cudaDeviceSynchronize());
    while (pl->other_text.size() + missing > kMaxCachedTextLengths) {
      auto victim = pl->other_text.end();
      for (auto it = pl->other_text.begin(); it != pl->other_text.end(); ++it)
        if ((*it)->last_use != now && (victim == pl->other_text.end() || (*it)->last_use < (*victim)->last_use))
          victim = it;
      if (victim == pl->other_text.end()) break;        // every cached set serves this call
      (*victim)->release();
      pl->other_text.erase(victim);
    }
  }
  for (size_t i = 0; i < lengths.size(); ++i) {
    if (out[i] != nullptr) continue;
    std::unique_ptr<TextSchedules> ts(new TextSchedules());
    int rc = build_text_dependent(pl, lengths[i], *ts);
    if (rc != VB_OK) {
      ts->release();
      return rc;
    }
    ts->last_use = now;
    out[i] = ts.get();
    pl->other_text.push_back(std::move(ts));
  }
  return VB_OK;
}

extern "C" {

const char* vb_last_error(void) { return get_error(); }
int vb_version(void) { return 101; }

int vb_device_check(void) {
  int dev = 0, major = 0, minor = 0, count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
    cudaGetLastError();
    set_error("no CUDA device: vorta_b200 has no CPU path");
    return VB_ERR_UNSUPPORTED;
  }
  VB_CUDA_OK(cudaGetDevice(&dev));
  VB_CUDA_OK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  VB_CUDA_OK(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  VB_REQUIRE(major == 10, VB_ERR_UNSUPPORTED, "device is sm_%d%d; this library is built for sm_100a only", major,
             minor);
  return VB_OK;
}

int vb_plan_create(vb_plan** out, const vb_plan_desc* desc) {
  VB_REQUIRE(out != nullptr && desc != nullptr, VB_ERR_INVALID, "null argument");
  const vb_plan_desc& d = *desc;
  for (int i = 0; i < 3; ++i) {
    VB_REQUIRE(d.latent[i] > 0 && d.tile[i] > 0 && d.window[i] > 0 && d.lowres_window[i] > 0, VB_ERR_INVALID,
               "latent / tile / window sizes must be positive");
    // reference: wan.py:186-189
    VB_REQUIRE(d.latent[i] % d.tile[i] == 0, VB_ERR_INVALID,
               "Tile size (%d, %d, %d) (dim=%d) does not divide latent shape (%d, %d, %d) (dim=%d).", d.tile[0],
               d.tile[1], d.tile[2], d.tile[i], d.latent[0], d.latent[1], d.latent[2], d.latent[i]);
  }
  vb_plan* pl = new vb_plan();
  pl->d = d;
  pl->S = d.latent[0] * d.latent[1] * d.latent[2];
  const int fg = d.latent[0] / d.lowres_window[0], hg = d.latent[1] / d.lowres_window[1],
            wg = d.latent[2] / d.lowres_window[2];
  pl->G = fg * hg * wg;
  pl->g = d.lowres_window[0] * d.lowres_window[1] * d.lowres_window[2];
  pl->n_u = d.n_unpooled;
  pl->n_p = pl->g - 1 - pl->n_u;
  pl->S_c = pl->G * (1 + pl->n_u);
  auto fail = [&](int code) {
    delete pl;
    return code;
  };
  // reference: wan.py:191-193 (S == G * g)
  if (pl->S != pl->G * pl->g) {
    set_error("Input sequence length %d does not match low-res info %dx%d.", pl->S, pl->G, pl->g);
    return fail(VB_ERR_INVALID);
  }
  if (pl->n_u < 0 || pl->n_p < 0) {
    set_error("n_unpooled %d out of range for group size %d", pl->n_u, pl->g);
    return fail(VB_ERR_INVALID);
  }
  if (pl->g > kSelectMaxGroup) {
    set_error("coreset group of %d tokens exceeds the selection kernel's maximum of %d tokens", pl->g, kSelectMaxGroup);
    return fail(VB_ERR_UNSUPPORTED);
  }
  if (d.text_len < 0 || d.text_valid < 0 || d.text_valid > d.text_len) {
    set_error("text_valid %d must be within [0, text_len %d]", d.text_valid, d.text_len);
    return fail(VB_ERR_INVALID);
  }
  for (int i = 0; i < 3; ++i) pl->nt[i] = d.latent[i] / d.tile[i];
  pl->n_tiles = pl->nt[0] * pl->nt[1] * pl->nt[2];
  pl->tile_tokens = d.tile[0] * d.tile[1] * d.tile[2];

  // ---- coreset groups (coreset_select.py:31-54): raster group order, raster member order
  const int fw = d.lowres_window[0], hw = d.lowres_window[1], ww = d.lowres_window[2];
  const int center_slot = (fw / 2) * hw * ww + (hw / 2) * ww + ww / 2;
  pl->center.resize(pl->G);
  pl->margin.resize(static_cast<size_t>(pl->G) * (pl->g - 1));
  std::vector<int32_t> center32(pl->G), margin32(pl->margin.size());
  for (int gf = 0; gf < fg; ++gf)
    for (int gh = 0; gh < hg; ++gh)
      for (int gw = 0; gw < wg; ++gw) {
        const int grp = (gf * hg + gh) * wg + gw;
        int slot = 0, mi = 0;
        for (int f = 0; f < fw; ++f)
          for (int h = 0; h < hw; ++h)
            for (int w = 0; w < ww; ++w, ++slot) {
              const int tok = ((gf * fw + f) * d.latent[1] + (gh * hw + h)) * d.latent[2] + (gw * ww + w);
              if (slot == center_slot) {
                pl->center[grp] = tok;
                center32[grp] = tok;
              } else {
                pl->margin[static_cast<size_t>(grp) * (pl->g - 1) + mi] = tok;
                margin32[static_cast<size_t>(grp) * (pl->g - 1) + mi] = tok;
                ++mi;
              }
            }
      }

  // ---- tile-major map (tile.py:26-29): position (tile_id * tau + intra) -> raster token; text rows keep theirs
  pl->tile_map.resize(pl->S + d.text_len);
  {
    int pos = 0;
    for (int a = 0; a < pl->nt[0]; ++a)
      for (int b = 0; b < pl->nt[1]; ++b)
        for (int c = 0; c < pl->nt[2]; ++c)
          for (int x = 0; x < d.tile[0]; ++x)
            for (int y = 0; y < d.tile[1]; ++y)
              for (int z = 0; z < d.tile[2]; ++z)
                pl->tile_map[pos++] =
                    ((a * d.tile[0] + x) * d.latent[1] + (b * d.tile[1] + y)) * d.latent[2] + (c * d.tile[2] + z);
    for (int i = 0; i < d.text_len; ++i) pl->tile_map[pl->S + i] = pl->S + i;
  }

  // ---- windows per tile (sliding_attn_flex.py:118-127), window groups in order of first appearance, and the
  //      sliding branch's query order: group by group, tiles of a group in tile order, tokens in tile-major order
  pl->tile_window.assign(static_cast<size_t>(pl->n_tiles) * 6, 0);
  {
    std::vector<std::vector<int>> members;
    std::map<std::array<int, 6>, int> index_of;             // window -> group
    for (int a = 0; a < pl->nt[0]; ++a)
      for (int b = 0; b < pl->nt[1]; ++b)
        for (int c = 0; c < pl->nt[2]; ++c) {
          const int tile_id = (a * pl->nt[1] + b) * pl->nt[2] + c;
          int32_t* w = &pl->tile_window[static_cast<size_t>(tile_id) * 6];
          int lo, hi;
          window_range(a, pl->nt[0], d.window[0], lo, hi); w[0] = lo; w[3] = hi;
          window_range(b, pl->nt[1], d.window[1], lo, hi); w[1] = lo; w[4] = hi;
          window_range(c, pl->nt[2], d.window[2], lo, hi); w[2] = lo; w[5] = hi;
          const std::array<int, 6> key = {w[0], w[1], w[2], w[3], w[4], w[5]};
          auto hit = index_of.find(key);
          int found;
          if (hit != index_of.end()) {
            found = hit->second;
          } else {
            vb_plan::WindowGroup g;
            for (int i = 0; i < 3; ++i) { g.lo[i] = w[i]; g.hi[i] = w[3 + i]; }
            g.row0 = 0; g.n_tiles = 0;
            found = static_cast<int>(pl->groups.size());
            pl->groups.push_back(g);
            members.emplace_back();
            index_of.emplace(key, found);
          }
          members[found].push_back(tile_id);
        }
    pl->query_map.resize(pl->S + d.text_len);
    int pos = 0;
    const int tau = pl->tile_tokens;
    for (size_t g = 0; g < pl->groups.size(); ++g) {
      pl->groups[g].row0 = pos;
      pl->groups[g].n_tiles = static_cast<int>(members[g].size());
      for (int tile_id : members[g])
        for (int i = 0; i < tau; ++i) pl->query_map[pos++] = pl->tile_map[static_cast<size_t>(tile_id) * tau + i];
    }
    for (int i = 0; i < d.text_len; ++i) pl->query_map[pl->S + i] = pl->S + i;
  }

  // device copies only when a device exists: geometry queries / exports also work on a CPU-only host
  int count = 0;
  if (cudaGetDeviceCount(&count) == cudaSuccess && count > 0) {
    pl->has_device = true;
    auto up = [&](int32_t** dptr, const std::vector<int32_t>& v) -> int {
      if (v.empty()) return VB_OK;
      VB_CUDA_OK(cudaMalloc(dptr, v.size() * sizeof(int32_t)));
      VB_CUDA_OK(cudaMemcpy(*dptr, v.data(), v.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
      return VB_OK;
    };
    int rc;
    if ((rc = up(&pl->d_center_tok, center32)) != VB_OK || (rc = up(&pl->d_margin_tok, margin32)) != VB_OK ||
        (rc = up(&pl->d_tile_map, pl->tile_map)) != VB_OK || (rc = up(&pl->d_query_map, pl->query_map)) != VB_OK) {
      vb_plan_destroy(pl);
      return rc;
    }
  } else {
    cudaGetLastError();
  }
  int rc = build_text_dependent(pl, d.text_valid, pl->text);
  if (rc != VB_OK) {
    vb_plan_destroy(pl);
    return rc;
  }
  *out = pl;
  return VB_OK;
}

void vb_plan_destroy(vb_plan* pl) {
  if (pl == nullptr) return;
  pl->text.release();
  for (auto& ts : pl->other_text) ts->release();
  if (pl->d_query_map) cudaFree(pl->d_query_map);
  if (pl->d_center_tok) cudaFree(pl->d_center_tok);
  if (pl->d_margin_tok) cudaFree(pl->d_margin_tok);
  if (pl->d_tile_map) cudaFree(pl->d_tile_map);
  delete pl;
}

int vb_plan_set_text_valid(vb_plan* pl, int32_t text_valid) {
  VB_REQUIRE(pl != nullptr, VB_ERR_INVALID, "null plan");
  VB_REQUIRE(text_valid >= 0 && text_valid <= pl->d.text_len, VB_ERR_INVALID,
             "text_valid %d must be within [0, text_len %d]", text_valid, pl->d.text_len);
  if (text_valid == pl->d.text_valid) return VB_OK;
  if (pl->has_device) VB_CUDA_OK(cudaDeviceSynchronize());   // tables may still be in use by earlier launches
  pl->d.text_valid = text_valid;
  pl->text.release();
  return build_text_dependent(pl, text_valid, pl->text);
}

int vb_plan_query(const vb_plan* pl, int what, int64_t* value) {
  VB_REQUIRE(pl != nullptr && value != nullptr, VB_ERR_INVALID, "null argument");
  switch (what) {
    case VB_PLAN_SEQ_LEN: *value = pl->S; break;
    case VB_PLAN_NUM_GROUPS: *value = pl->G; break;
    case VB_PLAN_GROUP_SIZE: *value = pl->g; break;
    case VB_PLAN_CORESET_LEN: *value = pl->S_c; break;
    case VB_PLAN_NUM_TILES: *value = pl->n_tiles; break;
    case VB_PLAN_TILE_TOKENS: *value = pl->tile_tokens; break;
    case VB_PLAN_NUM_POOLED: *value = pl->n_p; break;
    case VB_PLAN_KEYS_PER_QUERY: *value = pl->text.keys_per_query; break;
    case VB_PLAN_SLIDING_PAIRS: *value = static_cast<int64_t>(pl->text.sliding.pairs.size()); break;
    case VB_PLAN_SLIDING_RUNS: *value = static_cast<int64_t>(pl->text.sliding.runs.size()); break;
    default: VB_REQUIRE(false, VB_ERR_INVALID, "unknown plan query %d", what);
  }
  return VB_OK;
}

int vb_plan_export(const vb_plan* pl, int what, void* dst, int64_t* bytes) {
  VB_REQUIRE(pl != nullptr && bytes != nullptr, VB_ERR_INVALID, "null argument");
  const void* src = nullptr;
  int64_t n = 0;
  switch (what) {
    case VB_EXPORT_CENTER_INDICES: src = pl->center.data(); n = pl->center.size() * sizeof(int64_t); break;
    case VB_EXPORT_MARGIN_INDICES: src = pl->margin.data(); n = pl->margin.size() * sizeof(int64_t); break;
    case VB_EXPORT_TILE_MAP: src = pl->tile_map.data(); n = pl->tile_map.size() * sizeof(int32_t); break;
    case VB_EXPORT_TILE_WINDOW: src = pl->tile_window.data(); n = pl->tile_window.size() * sizeof(int32_t); break;
    case VB_EXPORT_SLIDING_RUNS: src = pl->text.sliding.runs.data(); n = pl->text.sliding.runs.size() * sizeof(KvRun); break;
    case VB_EXPORT_SLIDING_ITEMS:
      src = pl->text.sliding.pairs.data();
      n = pl->text.sliding.pairs.size() * sizeof(QPair);
      break;
    case VB_EXPORT_SLIDING_QUERY_MAP: src = pl->query_map.data(); n = pl->query_map.size() * sizeof(int32_t); break;
    default: VB_REQUIRE(false, VB_ERR_INVALID, "unknown plan export %d", what);
  }
  if (dst != nullptr) {
    VB_REQUIRE(*bytes >= n, VB_ERR_INVALID, "export buffer too small: %lld < %lld", (long long)*bytes, (long long)n);
    memcpy(dst, src, n);
  }
  *bytes = n;
  return VB_OK;
}

int vb_router_forward(const void* temb, int temb_dtype, const void* w, const void* bias, int w_dtype,
                      int64_t w_layer_stride, int64_t bias_layer_stride, int32_t n_layers, int32_t batch,
                      int32_t embed_dim, int32_t heads, float tau, float* scores, int32_t* branch,
                      vb_stream_t stream) {
  VB_REQUIRE(temb && w && bias && scores, VB_ERR_INVALID, "null argument");
  int rc = launch_router(temb, temb_dtype, w, bias, w_dtype, w_layer_stride, bias_layer_stride, n_layers, batch,
                         embed_dim, heads, tau, scores, branch, static_cast<cudaStream_t>(stream));
  if (rc == VB_OK) ++g_launches;
  return rc;
}

// Coreset selection over x, (b, h, s) element strides, for `heads` head slots of every batch element: slot i reads head
// i, and no output table is set yet.
static SelectParams select_params(const vb_plan* pl, const void* x, const int64_t* stride, int batch, int heads) {
  SelectParams p;
  memset(&p, 0, sizeof(p));
  p.x = static_cast<const __nv_bfloat16*>(x);
  p.stride_b = stride[0]; p.stride_h = stride[1]; p.stride_s = stride[2];
  p.center_tok = pl->d_center_tok; p.margin_tok = pl->d_margin_tok;
  p.batch = batch; p.heads = heads; p.G = pl->G; p.n_margin = pl->g - 1; p.n_unpooled = pl->n_u;
  p.seq_len = pl->S; p.text_len = pl->d.text_len;
  return p;
}

int vb_coreset_select(const vb_plan* pl, const void* x, int64_t stride_b, int64_t stride_h, int64_t stride_s,
                      int32_t batch, int32_t heads, int64_t* unpooled_argsort, int64_t* pooled_argsort,
                      int32_t* kept_tok, int32_t* dropped_tok, vb_stream_t stream) {
  VB_REQUIRE(pl && x, VB_ERR_INVALID, "null argument");
  VB_REQUIRE(pl->has_device, VB_ERR_UNSUPPORTED, "no CUDA device: vorta_b200 has no CPU path");
  VB_REQUIRE(stride_s % 8 == 0 && stride_h % 8 == 0 && stride_b % 8 == 0, VB_ERR_INVALID,
             "strides must be multiples of 8 elements");
  const int64_t stride[3] = {stride_b, stride_h, stride_s};
  SelectParams p = select_params(pl, x, stride, batch, heads);
  p.unpooled_argsort = unpooled_argsort; p.pooled_argsort = pooled_argsort;
  p.kept_tok = kept_tok; p.dropped_tok = dropped_tok;
  int rc = launch_coreset_select(p, static_cast<cudaStream_t>(stream));
  if (rc == VB_OK) ++g_launches;
  return rc;
}

int vb_coreset_tables(const vb_plan* pl, const int64_t* unpooled_argsort, const int64_t* pooled_argsort,
                      int32_t batch, int32_t heads, int32_t* kept_tok, int32_t* dropped_tok, int32_t* unpool_src,
                      vb_stream_t stream) {
  VB_REQUIRE(pl && unpooled_argsort && pooled_argsort, VB_ERR_INVALID, "null argument");
  VB_REQUIRE(pl->has_device, VB_ERR_UNSUPPORTED, "no CUDA device: vorta_b200 has no CPU path");
  TablesParams p;
  p.unpooled_argsort = unpooled_argsort; p.pooled_argsort = pooled_argsort;
  p.center_tok = pl->d_center_tok; p.margin_tok = pl->d_margin_tok;
  p.batch = batch; p.heads = heads; p.G = pl->G; p.n_margin = pl->g - 1; p.n_unpooled = pl->n_u;
  p.seq_len = pl->S; p.text_len = pl->d.text_len;
  p.kept_tok = kept_tok; p.dropped_tok = dropped_tok; p.unpool_src = unpool_src;
  int rc = launch_coreset_tables(p, static_cast<cudaStream_t>(stream));
  if (rc == VB_OK) ++g_launches;
  return rc;
}

int vb_gather_rows(const void* src, int64_t src_stride_b, int64_t src_stride_h, int64_t src_stride_s, void* dst,
                   int64_t dst_stride_b, int64_t dst_stride_h, int64_t dst_stride_s, const int32_t* map,
                   int64_t map_stride_b, int64_t map_stride_h, int32_t batch, int32_t heads, int32_t n_rows,
                   vb_stream_t stream) {
  VB_REQUIRE(src && dst, VB_ERR_INVALID, "null argument");
  GatherParams p;
  memset(&p, 0, sizeof(p));
  p.src[0] = static_cast<const __nv_bfloat16*>(src);
  p.dst[0] = static_cast<__nv_bfloat16*>(dst);
  p.src_stride[0][0] = src_stride_b; p.src_stride[0][1] = src_stride_h; p.src_stride[0][2] = src_stride_s;
  p.dst_stride[0] = dst_stride_b; p.dst_stride[1] = dst_stride_h; p.dst_stride[2] = dst_stride_s;
  p.map = map; p.map_stride_b = map_stride_b; p.map_stride_h = map_stride_h;
  p.head_list.used = 0; p.n_tensors = 1; p.batch = batch; p.heads = heads; p.n_rows = n_rows;
  int rc = launch_gather_rows(p, static_cast<cudaStream_t>(stream));
  if (rc == VB_OK) ++g_launches;
  return rc;
}

// ---- attention orchestration --------------------------------------------------------------------
static inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

int64_t vb_attn_workspace_bytes(const vb_plan* pl, int32_t batch, int32_t heads) {
  if (pl == nullptr) return 0;
  const int64_t rows_s = pl->S + pl->d.text_len;            // sliding: tile-major copy of q, k, v
  const int64_t rows_c = pl->S_c + pl->d.text_len;          // coreset: pooled q, k, v
  const int64_t bh = static_cast<int64_t>(batch) * heads;
  int64_t bytes = 0;
  bytes += 3 * align_up(bh * rows_s * kHeadDim * 2, 1024);
  bytes += 3 * align_up(bh * rows_c * kHeadDim * 2, 1024);
  bytes += 2 * align_up(bh * rows_c * 4, 1024);                              // kept_tok for Q and K matchings
  bytes += 2 * align_up(bh * static_cast<int64_t>(pl->G) * std::max(pl->n_p, 1) * 4, 1024);   // dropped_tok
  bytes += align_up(bh * rows_s * kHeadDim * 4, 1024) + align_up(bh * 3 * 4, 1024);             // blend: fp32 sums, scores
  return bytes + 4096;
}

namespace {
struct Carver {
  uint8_t* base;
  int64_t off, cap;
  void* take(int64_t bytes) {
    off = align_up(off, 1024);
    void* p = base + off;
    off += bytes;
    return off <= cap ? p : nullptr;
  }
};

// One branch of a layer, or one query part of the full branch, with the head slots it covers: one AttnSeg of a launch.
struct Segment {
  const __nv_bfloat16 *q = nullptr, *k = nullptr, *v = nullptr;
  int64_t qs[3] = {}, ks[3] = {}, vs[3] = {};   // b, h, s strides
  int64_t n_rows_q = 0, n_rows_kv = 0, n_heads_tensor = 0;
  const Schedule* sched = nullptr;
  int pair_begin = 0, n_pairs = 0;              // the segment's work items: sched->pairs[pair_begin, + n_pairs)
  const int32_t* out_map = nullptr;
  int64_t out_map_stride_b = 0, out_map_stride_h = 0;
  const int32_t* bcast_map = nullptr;
  int64_t bcast_stride_b = 0, bcast_stride_h = 0;
  int32_t bcast_rows = 0, bcast_n = 0;
  std::vector<AttnHead> heads;
  std::vector<int32_t> batches;                 // batch elements of the segment (<= kMaxSegBatch); empty = all of them
  int branch = 0;                               // 0 full (and its query parts), 1 coreset, 2 sliding
  double flops_per_head = 0.0;                  // of the segment's work items
};

// Where the attention output goes: `ptr`, or the peer buffers of the fused Ulysses exchange (vb_attn_args::out_peer_*).
struct Output {
  __nv_bfloat16* ptr;
  int64_t stride[3];                            // b, h, s
  __nv_bfloat16* peers[8];
  int32_t peer_count, peer_rows;
};

// Blend mode: the routing scores, the fp32 sums, and which of the three accumulation stages a launch is.
struct BlendState {
  const float* w;
  float* acc;
  int stage, branch, heads, rows;
};
}  // namespace

// A segment over all of `sched` for q, k, v with (b, h, s) element strides; no head slots yet.
static Segment segment_of(const void* q, const void* k, const void* v, const int64_t* qs, const int64_t* ks,
                          const int64_t* vs, int64_t n_rows_q, int64_t n_rows_kv, int64_t n_heads_tensor,
                          const Schedule& sched) {
  Segment sg;
  sg.q = static_cast<const __nv_bfloat16*>(q);
  sg.k = static_cast<const __nv_bfloat16*>(k);
  sg.v = static_cast<const __nv_bfloat16*>(v);
  for (int i = 0; i < 3; ++i) { sg.qs[i] = qs[i]; sg.ks[i] = ks[i]; sg.vs[i] = vs[i]; }
  sg.n_rows_q = n_rows_q; sg.n_rows_kv = n_rows_kv; sg.n_heads_tensor = n_heads_tensor;
  sg.sched = &sched;
  sg.n_pairs = static_cast<int>(sched.pairs.size());
  sg.flops_per_head = sched.flops_per_head;
  return sg;
}

// A segment over q, k, v gathered into contiguous (batch, nh, rows, 128) workspace tensors, n_rows of them attended.
static Segment workspace_segment(__nv_bfloat16* const qkv[3], int nh, int64_t rows, int64_t n_rows,
                                 const Schedule& sched) {
  const int64_t st[3] = {nh * rows * kHeadDim, rows * kHeadDim, kHeadDim};
  return segment_of(qkv[0], qkv[1], qkv[2], st, st, st, n_rows, n_rows, nh, sched);
}

// Tensors first .. first + n - 1 of the layer's (q, k, v) as the sources of a gather into dst[first ..].
static void gather_from_args(GatherParams& gp, const vb_attn_args& a, int first, int n, __nv_bfloat16* const dst[3]) {
  const void* src[3] = {a.q, a.k, a.v};
  const int64_t* stride[3] = {a.q_stride, a.k_stride, a.v_stride};
  gp.n_tensors = n;
  for (int t = 0; t < n; ++t) {
    gp.src[t] = static_cast<const __nv_bfloat16*>(src[first + t]);
    gp.dst[t] = dst[first + t];
    for (int i = 0; i < 3; ++i) gp.src_stride[t][i] = stride[first + t][i];
  }
}

// Launches the head slots of n_seg segments, in the given order (longest CTAs first), as grids of at most kMaxHeads
// heads and kMaxSegments segments: a grid takes segments until either is full, so a segment with more heads spans
// several launches, and so do more segments than one grid holds.  Segments of the same heads over different batch
// elements (one per text-length group) share their head slots.  The segments write disjoint outputs: different heads,
// or the same heads of different batch elements (blend mode accumulates branch after branch, one call per branch).
static int launch_segments(const Segment* segs, int n_seg, int batch, const Output& out, float* dbg,
                           const BlendState* blend, int kind, cudaStream_t stream) {
  AttnTmaps tm;
  AttnParams p;
  int rc, n_used, head0;
  int64_t n_ctas;
  double flops;
  auto start_grid = [&]() {
    memset(&tm, 0, sizeof(tm));
    memset(&p, 0, sizeof(p));
    n_used = head0 = 0;
    n_ctas = 0;
    flops = 0.0;
  };
  auto launch_grid = [&]() -> int {
    if (n_used == 0) return VB_OK;
    VB_REQUIRE(n_ctas < (1ll << 31), VB_ERR_UNSUPPORTED, "attention grid too large");
    p.n_seg = n_used;
    p.n_items = static_cast<int32_t>(n_ctas);
    p.out = out.ptr;
    p.out_stride_b = out.stride[0]; p.out_stride_h = out.stride[1]; p.out_stride_s = out.stride[2];
    p.out_peer_count = out.peer_count;
    p.out_peer_rows = out.peer_rows;
    for (int i = 0; i < 8; ++i) p.out_peers[i] = out.peers[i];
    p.scale_log2 = 1.4426950408889634f / sqrtf(static_cast<float>(kHeadDim));
    if (blend != nullptr) {
      p.blend_w = blend->w; p.blend_acc = blend->acc; p.blend_stage = blend->stage;
      p.blend_heads = blend->heads; p.blend_branch = blend->branch; p.blend_rows = blend->rows;
    }
    p.dbg = dbg;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    if (g_timing) {
      VB_CUDA_OK(cudaEventCreate(&ev0));
      VB_CUDA_OK(cudaEventCreate(&ev1));
      VB_CUDA_OK(cudaEventRecord(ev0, stream));
    }
    const int r = launch_attn(tm, p, static_cast<int>(n_ctas), stream);
    if (r != VB_OK) return r;
    if (g_timing) {
      VB_CUDA_OK(cudaEventRecord(ev1, stream));
      g_events.push_back({ev0, ev1, kind, flops});
    }
    ++g_launches;
    g_flops += flops;
    start_grid();
    return VB_OK;
  };
  // head0 of n slots of this grid that already hold exactly hs[0, n), or -1
  auto placed_heads = [&](const AttnHead* hs, int n) -> int {
    for (int j = 0; j < n_used; ++j)
      if (p.seg[j].n_heads == n && memcmp(&p.heads[p.seg[j].head0], hs, n * sizeof(AttnHead)) == 0)
        return p.seg[j].head0;
    return -1;
  };
  start_grid();
  for (int i = 0; i < n_seg; ++i) {
    const Segment& sg = segs[i];
    if (sg.n_pairs == 0) continue;
    VB_REQUIRE(sg.batches.size() <= static_cast<size_t>(kMaxSegBatch), VB_ERR_UNSUPPORTED,
               "a segment lists at most %d batch elements", kMaxSegBatch);
    const int n_batch = sg.batches.empty() ? batch : static_cast<int>(sg.batches.size());
    for (size_t h = 0; h < sg.heads.size();) {
      if (n_used == kMaxSegments && (rc = launch_grid()) != VB_OK) return rc;
      int n = static_cast<int>(std::min(sg.heads.size() - h, static_cast<size_t>(kMaxHeads)));
      int first = placed_heads(&sg.heads[h], n);
      if (first < 0) {
        if (head0 == kMaxHeads && (rc = launch_grid()) != VB_OK) return rc;
        n = static_cast<int>(std::min(sg.heads.size() - h, static_cast<size_t>(kMaxHeads - head0)));
        first = head0;
        for (int j = 0; j < n; ++j) p.heads[head0 + j] = sg.heads[h + j];
        head0 += n;
      }
      CUtensorMap* m = tm.m[n_used];
      if ((rc = make_qkv_tensor_map(&m[0], sg.q, sg.n_rows_q, sg.n_heads_tensor, batch, sg.qs[0], sg.qs[1], sg.qs[2])))
        return rc;
      if ((rc = make_qkv_tensor_map(&m[1], sg.k, sg.n_rows_kv, sg.n_heads_tensor, batch, sg.ks[0], sg.ks[1], sg.ks[2])))
        return rc;
      if ((rc = make_qkv_tensor_map(&m[2], sg.v, sg.n_rows_kv, sg.n_heads_tensor, batch, sg.vs[0], sg.vs[1], sg.vs[2])))
        return rc;
      AttnSeg& s = p.seg[n_used];
      s.pairs = sg.sched->d_pairs + sg.pair_begin;
      s.runs = sg.sched->d_runs;
      s.out_map = sg.out_map; s.out_map_stride_b = sg.out_map_stride_b; s.out_map_stride_h = sg.out_map_stride_h;
      s.bcast_map = sg.bcast_map; s.bcast_stride_b = sg.bcast_stride_b; s.bcast_stride_h = sg.bcast_stride_h;
      s.bcast_rows = sg.bcast_rows; s.bcast_n = sg.bcast_n;
      s.n_pairs = sg.n_pairs;
      s.n_heads = n;
      s.n_batch = n_batch;
      s.batch_listed = sg.batches.empty() ? 0 : 1;
      for (size_t j = 0; j < sg.batches.size(); ++j) s.batch_of[j] = static_cast<uint16_t>(sg.batches[j]);
      s.head0 = first;
      s.cta_begin = static_cast<int32_t>(n_ctas);
      h += n;
      n_ctas += static_cast<int64_t>(s.n_pairs) * s.n_heads * n_batch;
      flops += sg.flops_per_head * s.n_heads * n_batch;
      ++n_used;
    }
  }
  return launch_grid();
}

// Samples of one text length: that length's schedules and the batch elements that run them (empty = all of them).
namespace {
struct LengthGroup {
  const TextSchedules* ts;
  std::vector<int32_t> batches;
};
}  // namespace

int vb_attn_fwd(vb_plan* pl, const vb_attn_args* args, vb_stream_t stream_) {
  VB_REQUIRE(pl != nullptr && args != nullptr, VB_ERR_INVALID, "null argument");
  VB_REQUIRE(pl->has_device, VB_ERR_UNSUPPORTED, "no CUDA device: vorta_b200 has no CPU path");
  const vb_attn_args& a = *args;
  VB_REQUIRE(a.q && a.k && a.v && (a.out || a.out_peer_count > 0), VB_ERR_INVALID, "null tensor");
  VB_REQUIRE(a.out_peer_count >= 0 && a.out_peer_count <= 8, VB_ERR_INVALID, "out_peer_count must be within [0, 8]");
  VB_REQUIRE(a.out_peer_count == 0 ||
                 (a.weights == nullptr && a.out_peer_rows > 0 &&
                  static_cast<int64_t>(a.out_peer_rows) * a.out_peer_count == pl->S),
             VB_ERR_UNSUPPORTED, "peer output needs top-1 routing and out_peer_rows * out_peer_count == video tokens");
  VB_REQUIRE(a.batch > 0 && a.heads > 0, VB_ERR_INVALID, "batch and heads must be positive");
  VB_REQUIRE(a.weights != nullptr || a.weights_device != nullptr || a.branch != nullptr, VB_ERR_INVALID,
             "need branch ids or blend weights");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const bool blend = a.weights != nullptr || a.weights_device != nullptr;
  NvtxRange nvtx_layer(blend ? "vb_attn_fwd (blend)" : "vb_attn_fwd (top-1)");
  const int S = pl->S, TL = pl->d.text_len;
  const int N = S + TL;
  int rc;

  // un-padded text length of every sample (NULL: the plan's text_valid), and the samples grouped by length, longest
  // first.  One length is one group over all samples, which runs the plan's own schedules when it is the plan's length.
  std::vector<int32_t> tv_of(a.batch, pl->d.text_valid);
  if (a.text_valid != nullptr) {
    for (int b = 0; b < a.batch; ++b) {
      VB_REQUIRE(a.text_valid[b] >= 0 && a.text_valid[b] <= TL, VB_ERR_INVALID,
                 "text_valid[%d] = %d must be within [0, text_len %d]", b, a.text_valid[b], TL);
      tv_of[b] = a.text_valid[b];
    }
  }
  std::vector<int32_t> lengths(tv_of);
  std::sort(lengths.begin(), lengths.end(), std::greater<int32_t>());
  lengths.erase(std::unique(lengths.begin(), lengths.end()), lengths.end());
  std::vector<const TextSchedules*> sched_of(1, &pl->text);
  std::unique_lock<std::mutex> cache_lock;        // held until the launches that read cached tables are enqueued
  if (lengths.size() > 1 || lengths[0] != pl->d.text_valid) {
    cache_lock = std::unique_lock<std::mutex>(pl->text_mutex);
    if ((rc = text_schedules(pl, lengths, sched_of)) != VB_OK) return rc;
  }
  std::vector<LengthGroup> groups;
  if (lengths.size() == 1) {
    groups.push_back({sched_of[0], {}});
  } else {
    for (size_t i = 0; i < lengths.size(); ++i)
      for (int b = 0; b < a.batch; ++b) {
        if (tv_of[b] != lengths[i]) continue;
        if (groups.empty() || groups.back().ts != sched_of[i] || groups.back().batches.size() == kMaxSegBatch)
          groups.push_back({sched_of[i], {}});
        groups.back().batches.push_back(b);
      }
  }

  // heads of each branch, ascending head order (wan.py:409 torch.nonzero)
  std::vector<int32_t> by_branch[3];      // 0 full, 1 coreset, 2 sliding
  // full attention over part k of n of the query work items (VB_BRANCH_FULL_PART; LO / HI = 0 / 1 of 2): heads per (n, k)
  std::vector<std::pair<int, std::vector<int32_t>>> parts;
  for (int h = 0; h < a.heads; ++h) {
    if (blend) {
      for (int e = 0; e < 3; ++e) by_branch[e].push_back(h);
    } else {
      int e = a.branch[h];
      if (e == VB_BRANCH_SKIP) continue;
      if (e == VB_BRANCH_FULL_LO) e = VB_BRANCH_FULL_PART(0, 2);
      if (e == VB_BRANCH_FULL_HI) e = VB_BRANCH_FULL_PART(1, 2);
      if (e >= 16) {
        const int n = (e - 16) >> 3, k = (e - 16) & 7;
        VB_REQUIRE(n >= 2 && n <= 7 && k < n, VB_ERR_INVALID, "branch id %d of head %d is not a valid query part", e, h);
        size_t i = 0;
        while (i < parts.size() && parts[i].first != e) ++i;
        if (i == parts.size()) parts.push_back({e, {}});
        parts[i].second.push_back(h);
        continue;
      }
      VB_REQUIRE(e >= 0 && e < 3, VB_ERR_INVALID, "branch id %d of head %d out of range", e, h);
      by_branch[e].push_back(h);
    }
  }
  VB_REQUIRE(parts.size() + 3 <= static_cast<size_t>(kMaxSegments), VB_ERR_UNSUPPORTED,
             "at most %d different query parts per launch", kMaxSegments - 3);
  const int64_t need = vb_attn_workspace_bytes(pl, a.batch, a.heads);
  const bool needs_ws = blend || !by_branch[1].empty() || !by_branch[2].empty();
  VB_REQUIRE(!needs_ws || (a.workspace != nullptr && a.workspace_bytes >= need), VB_ERR_INVALID,
             "workspace too small: %lld < %lld bytes", (long long)a.workspace_bytes, (long long)need);
  Carver ws{static_cast<uint8_t*>(a.workspace), 0, a.workspace_bytes};
  // blend mode: fp32 partial sums per (batch, head slot, output token), whatever the output's strides and out_heads, and
  // the routing scores on the device
  BlendState blend_state;
  memset(&blend_state, 0, sizeof(blend_state));
  if (blend) {
    VB_REQUIRE(a.out != nullptr && a.out_peer_count == 0, VB_ERR_UNSUPPORTED, "blend mode writes a local output");
    blend_state.acc = static_cast<float*>(ws.take(static_cast<int64_t>(a.batch) * a.heads * N * kHeadDim * 4));
    float* w_dev = static_cast<float*>(ws.take(static_cast<int64_t>(a.batch) * a.heads * 3 * 4));
    VB_REQUIRE(blend_state.acc != nullptr && w_dev != nullptr, VB_ERR_INVALID, "workspace exhausted");
    if (a.weights_device != nullptr) {
      blend_state.w = a.weights_device;
    } else {
      VB_CUDA_OK(cudaMemcpyAsync(w_dev, a.weights, static_cast<size_t>(a.batch) * a.heads * 3 * 4, cudaMemcpyHostToDevice,
                                 stream));
      blend_state.w = w_dev;
    }
    blend_state.heads = a.heads;
    blend_state.rows = N;
  }

  // head slots of a segment over heads hs; hk is the head in the segment's q / k / v: the layer's head, or the slot of a
  // workspace copy that holds only hs
  auto head_entries = [&](const std::vector<int32_t>& hs, bool slot_is_index) {
    std::vector<AttnHead> v(hs.size());
    for (size_t i = 0; i < hs.size(); ++i) {
      v[i].hk = slot_is_index ? static_cast<int32_t>(i) : hs[i];
      v[i].ho = a.out_heads ? a.out_heads[hs[i]] : hs[i];
      v[i].wi = hs[i];
    }
    return v;
  };
  auto head_list_of = [&](const std::vector<int32_t>& hs, HeadList* out) -> int {
    VB_REQUIRE(hs.size() <= static_cast<size_t>(kMaxHeads) && a.heads <= 256, VB_ERR_UNSUPPORTED,
               "more than %d heads of one branch in a layer", kMaxHeads);
    memset(out, 0, sizeof(*out));
    out->used = 1;
    for (size_t i = 0; i < hs.size(); ++i) out->h[i] = static_cast<uint8_t>(hs[i]);
    return VB_OK;
  };
  // top-1 mode: every head is in exactly one segment, so the segments write disjoint outputs and run as ONE launch after
  // all selection / gather passes; kept in branch order full, query parts, coreset, sliding, which is longest-CTA-first
  // (full: S/128 key blocks per CTA, coreset: ~S/256, sliding: <= 27 tiles)
  const bool merge = !blend && a.heads <= kMaxHeads;
  VB_REQUIRE(!blend || parts.empty(), VB_ERR_INVALID, "query-part ids need top-1 mode");
  std::vector<Segment> segs;

  // ---------------- branch 0: full attention, straight from the caller's tensors ----------------
  // One segment per length group, of each of the full heads and the query parts
  auto full_of = [&](const LengthGroup& g) {
    const int tv = g.ts->text_valid;
    Segment sg = segment_of(a.q, a.k, a.v, a.q_stride, a.k_stride, a.v_stride, S + tv, S + tv, a.heads, g.ts->full);
    sg.batches = g.batches;
    return sg;
  };
  if (!by_branch[0].empty()) {
    for (const LengthGroup& g : groups) {
      segs.push_back(full_of(g));
      segs.back().heads = head_entries(by_branch[0], false);
    }
  }
  // query parts: work items [k N / n, (k + 1) N / n) of the same schedule (other ranks run the other parts); a part's
  // share of the head's FLOPs goes by query rows
  for (const auto& part : parts) {
    const int n = (part.first - 16) >> 3, k = (part.first - 16) & 7;
    for (const LengthGroup& g : groups) {
      const std::vector<QPair>& items = g.ts->full.pairs;
      auto rows_of = [&](int begin, int end) {
        int64_t rows = 0;
        for (int i = begin; i < end; ++i) rows += items[i].q_rows[0] + (items[i].nq == 2 ? items[i].q_rows[1] : 0);
        return rows;
      };
      const int64_t n_items = static_cast<int64_t>(items.size());
      const int64_t rows_all = rows_of(0, static_cast<int>(n_items));
      const int begin = static_cast<int>(n_items * k / n), end = static_cast<int>(n_items * (k + 1) / n);
      if (end <= begin) continue;
      VB_REQUIRE(merge, VB_ERR_UNSUPPORTED, "query-half work units need the merged top-1 launch");
      segs.push_back(full_of(g));
      Segment& sg = segs.back();
      sg.heads = head_entries(part.second, false);
      sg.pair_begin = begin;
      sg.n_pairs = end - begin;
      sg.flops_per_head = g.ts->full.flops_per_head * (static_cast<double>(rows_of(begin, end)) /
                                                       static_cast<double>(std::max<int64_t>(rows_all, 1)));
    }
  }

  // ---------------- branch 1: coreset ----------------
  if (!by_branch[1].empty()) {
    NvtxRange nvtx("vb: coreset select + pool");
    const std::vector<int32_t>& hs = by_branch[1];
    const int nh = static_cast<int>(hs.size());
    const int64_t rows = pl->S_c + TL;
    const int64_t bh = static_cast<int64_t>(a.batch) * nh;
    __nv_bfloat16* pooled[3];
    for (__nv_bfloat16*& t : pooled) t = static_cast<__nv_bfloat16*>(ws.take(bh * rows * kHeadDim * 2));
    int32_t* kept_q = static_cast<int32_t*>(ws.take(bh * rows * 4));
    int32_t* drop_q = static_cast<int32_t*>(ws.take(bh * pl->G * std::max(pl->n_p, 1) * 4));
    int32_t* kept_k = kept_q;
    const bool kv_from_k = (a.flags & VB_ATTN_CORESET_KV_FROM_K) != 0;
    if (kv_from_k) kept_k = static_cast<int32_t*>(ws.take(bh * rows * 4));
    HeadList heads_c;
    if ((rc = head_list_of(hs, &heads_c)) != VB_OK) return rc;
    VB_REQUIRE(pooled[0] && pooled[1] && pooled[2] && kept_q && drop_q && kept_k, VB_ERR_INVALID, "workspace exhausted");

    SelectParams sp = select_params(pl, a.q, a.q_stride, a.batch, nh);
    sp.head_list = heads_c; sp.kept_tok = kept_q; sp.dropped_tok = drop_q;
    if ((rc = launch_coreset_select(sp, stream)) != VB_OK) return rc;
    ++g_launches;
    if (kv_from_k) {
      sp = select_params(pl, a.k, a.k_stride, a.batch, nh);
      sp.head_list = heads_c; sp.kept_tok = kept_k;
      if ((rc = launch_coreset_select(sp, stream)) != VB_OK) return rc;
      ++g_launches;
    }
    // pooled sequences [centres | kept margins | text]
    GatherParams gp;
    memset(&gp, 0, sizeof(gp));
    gp.dst_stride[0] = nh * rows * kHeadDim; gp.dst_stride[1] = rows * kHeadDim; gp.dst_stride[2] = kHeadDim;
    gp.map = kept_q; gp.map_stride_b = nh * rows; gp.map_stride_h = rows;
    gp.head_list = heads_c; gp.batch = a.batch; gp.heads = nh; gp.n_rows = static_cast<int32_t>(rows);
    if (!kv_from_k) {
      gather_from_args(gp, a, 0, 3, pooled);
      if ((rc = launch_gather_rows(gp, stream)) != VB_OK) return rc;
      ++g_launches;
    } else {
      gather_from_args(gp, a, 0, 1, pooled);
      if ((rc = launch_gather_rows(gp, stream)) != VB_OK) return rc;
      gp.map = kept_k;
      gather_from_args(gp, a, 1, 2, pooled);
      if ((rc = launch_gather_rows(gp, stream)) != VB_OK) return rc;
      g_launches += 2;
    }
    // the pooled sequences hold every sample's text rows; a length group attends to the first S_c + tv of them
    for (const LengthGroup& g : groups) {
      Segment sg = workspace_segment(pooled, nh, rows, pl->S_c + g.ts->text_valid, g.ts->coreset);
      sg.heads = head_entries(hs, true);
      sg.batches = g.batches;
      sg.branch = 1;
      sg.out_map = kept_q; sg.out_map_stride_b = nh * rows; sg.out_map_stride_h = rows;
      if (pl->n_p > 0) {   // dropped margins receive their centre's output (coreset_select.py:157)
        sg.bcast_map = drop_q; sg.bcast_stride_b = static_cast<int64_t>(nh) * pl->G * pl->n_p;
        sg.bcast_stride_h = static_cast<int64_t>(pl->G) * pl->n_p; sg.bcast_rows = pl->G; sg.bcast_n = pl->n_p;
      }
      segs.push_back(std::move(sg));
    }
  }

  // ---------------- branch 2: sliding tile ----------------
  if (!by_branch[2].empty()) {
    const std::vector<int32_t>& hs = by_branch[2];
    const int nh = static_cast<int>(hs.size());
    // layout pass: K and V in tile-major order, Q in window-group order (vb_plan::groups); the epilogue scatters the
    // output rows back to raster order through the same query map
    NvtxRange nvtx("vb: sliding tile-major layout");
    const int64_t rows = N;
    const int64_t bh = static_cast<int64_t>(a.batch) * nh;
    __nv_bfloat16* tiled[3];
    for (__nv_bfloat16*& t : tiled) t = static_cast<__nv_bfloat16*>(ws.take(bh * rows * kHeadDim * 2));
    HeadList heads_s;
    if ((rc = head_list_of(hs, &heads_s)) != VB_OK) return rc;
    VB_REQUIRE(tiled[0] && tiled[1] && tiled[2], VB_ERR_INVALID, "workspace exhausted");
    GatherParams gp;
    memset(&gp, 0, sizeof(gp));
    gp.map = pl->d_tile_map; gp.map0 = pl->d_query_map; gp.map_stride_b = 0; gp.map_stride_h = 0;
    gather_from_args(gp, a, 0, 3, tiled);
    gp.dst_stride[0] = nh * rows * kHeadDim; gp.dst_stride[1] = rows * kHeadDim; gp.dst_stride[2] = kHeadDim;
    gp.head_list = heads_s; gp.batch = a.batch; gp.heads = nh; gp.n_rows = static_cast<int32_t>(rows);
    if ((rc = launch_gather_rows(gp, stream)) != VB_OK) return rc;
    ++g_launches;
    for (const LengthGroup& g : groups) {
      Segment sg = workspace_segment(tiled, nh, rows, S + g.ts->text_valid, g.ts->sliding);
      sg.heads = head_entries(hs, true);
      sg.batches = g.batches;
      sg.branch = 2;
      sg.out_map = pl->d_query_map;
      segs.push_back(std::move(sg));
    }
  }

  Output out;
  memset(&out, 0, sizeof(out));
  out.ptr = static_cast<__nv_bfloat16*>(a.out);
  for (int i = 0; i < 3; ++i) out.stride[i] = a.out_stride[i];
  for (int i = 0; i < a.out_peer_count; ++i) out.peers[i] = static_cast<__nv_bfloat16*>(a.out_peer_ptrs[i]);
  out.peer_count = a.out_peer_count;
  out.peer_rows = a.out_peer_rows;
  if (merge) {
    NvtxRange nvtx("vb: attention launch (full + coreset + sliding segments)");
    rc = launch_segments(segs.data(), static_cast<int>(segs.size()), a.batch, out, a.debug, nullptr, VB_TIMING_ROUTED,
                         stream);
    if (rc != VB_OK) return rc;
  } else {
    // one branch at a time.  Blend: branch e is stage e + 1 of the fp32 accumulation; ONE launch covers every batch
    // element (the scores are read per (batch, head) from the device table), a segment per length group, so each
    // (batch, head) is accumulated once per stage
    for (size_t i = 0; i < segs.size();) {
      size_t j = i;
      while (j < segs.size() && segs[j].branch == segs[i].branch) ++j;
      blend_state.stage = segs[i].branch + 1;
      blend_state.branch = segs[i].branch;
      rc = launch_segments(&segs[i], static_cast<int>(j - i), a.batch, out, a.debug, blend ? &blend_state : nullptr,
                           VB_TIMING_ROUTED, stream);
      if (rc != VB_OK) return rc;
      i = j;
    }
  }

  // ---------------- padded text queries produce zeros (hunyuan.py:176; flex fully-masked rows) ----------------
  // They belong to the output heads the slots write (out_heads): a SKIP slot owns none, and of a head split into query
  // parts only the last part owns them, since its work items end where the padded rows begin.
  // Each sample's own padded rows [S + tv[b], S + text_len), all samples in one launch.
  const int min_tv = lengths.back();
  if (TL > min_tv && a.out_peer_count == 0) {      // (peer mode: every rank zeroes its own receive buffer)
    std::vector<int32_t> zero_heads;
    for (int h = 0; h < a.heads; ++h) {
      if (!blend) {
        int e = a.branch[h];
        if (e == VB_BRANCH_FULL_LO) e = VB_BRANCH_FULL_PART(0, 2);
        if (e == VB_BRANCH_FULL_HI) e = VB_BRANCH_FULL_PART(1, 2);
        if (e == VB_BRANCH_SKIP || (e >= 16 && ((e - 16) & 7) != ((e - 16) >> 3) - 1)) continue;
      }
      zero_heads.push_back(a.out_heads ? a.out_heads[h] : h);
    }
    ZeroRowsParams zp;
    memset(&zp, 0, sizeof(zp));
    zp.stride_b = a.out_stride[0]; zp.stride_h = a.out_stride[1]; zp.stride_s = a.out_stride[2];
    zp.row_end = N; zp.n_rows = TL - min_tv;
    // one launch for up to kMaxZeroBatch batch elements and kMaxZeroHeads heads
    for (int b0 = 0; b0 < a.batch; b0 += kMaxZeroBatch) {
      zp.out = static_cast<__nv_bfloat16*>(a.out) + static_cast<int64_t>(b0) * a.out_stride[0];
      zp.batch = std::min(kMaxZeroBatch, a.batch - b0);
      for (int i = 0; i < zp.batch; ++i) zp.row0[i] = S + tv_of[b0 + i];
      for (size_t h0 = 0; h0 < zero_heads.size(); h0 += kMaxZeroHeads) {
        zp.n_heads = static_cast<int32_t>(std::min(zero_heads.size() - h0, static_cast<size_t>(kMaxZeroHeads)));
        for (int i = 0; i < zp.n_heads; ++i) zp.head[i] = zero_heads[h0 + i];
        if ((rc = launch_zero_rows(zp, stream)) != VB_OK) return rc;
        ++g_launches;
      }
    }
  }
  return VB_OK;
}

// Dense attention with independent query / key lengths; schedules are cached per (n_q, n_k).
int vb_attn_dense(const void* q, const void* k, const void* v, void* out, const int64_t* q_stride,
                  const int64_t* k_stride, const int64_t* v_stride, const int64_t* out_stride, int32_t batch,
                  int32_t heads, int32_t n_q, int32_t n_k, vb_stream_t stream_) {
  VB_REQUIRE(q && k && v && out && q_stride && k_stride && v_stride && out_stride, VB_ERR_INVALID, "null argument");
  VB_REQUIRE(batch > 0 && heads > 0 && n_q > 0 && n_k > 0, VB_ERR_INVALID, "sizes must be positive");
  struct DenseKey {
    int dev, n_q, n_k;
  };
  static thread_local std::vector<std::pair<DenseKey, Schedule*>> cache;      // device tables: one entry per device
  int dev = 0;
  VB_CUDA_OK(cudaGetDevice(&dev));
  Schedule* sched = nullptr;
  for (auto& e : cache)
    if (e.first.dev == dev && e.first.n_q == n_q && e.first.n_k == n_k) sched = e.second;
  if (sched == nullptr) {
    sched = new Schedule();
    sched->runs.push_back({0, n_k});
    sched->add_query_range(0, n_q, 0, 1, n_k);
    sched->finalize();
    int rc = sched->upload();
    if (rc != VB_OK) {
      delete sched;
      return rc;
    }
    cache.push_back({DenseKey{dev, n_q, n_k}, sched});
  }
  Output o;
  memset(&o, 0, sizeof(o));
  o.ptr = static_cast<__nv_bfloat16*>(out);
  for (int i = 0; i < 3; ++i) o.stride[i] = out_stride[i];
  Segment sg = segment_of(q, k, v, q_stride, k_stride, v_stride, n_q, n_k, heads, *sched);
  for (int h = 0; h < heads; ++h) sg.heads.push_back(AttnHead{h, h, 0});
  NvtxRange nvtx("vb_attn_dense");
  return launch_segments(&sg, 1, batch, o, nullptr, nullptr, VB_TIMING_DENSE, static_cast<cudaStream_t>(stream_));
}

int vb_block_ln_modulate(const void* x, const float* weight, const float* bias, const float* scale, const float* shift,
                         void* out, int64_t rows, int32_t dim, int32_t rows_per_batch, float eps, vb_stream_t stream) {
  VB_REQUIRE(x && out, VB_ERR_INVALID, "null argument");
  VB_REQUIRE((scale == nullptr) == (shift == nullptr), VB_ERR_INVALID, "scale and shift come together");
  int rc = launch_ln_modulate(x, weight, bias, scale, shift, out, rows, dim, rows_per_batch, eps,
                              static_cast<cudaStream_t>(stream));
  if (rc == VB_OK) ++g_launches;
  return rc;
}
int vb_block_gate_residual(const void* x, const void* y, const float* gate, void* out, int64_t rows, int32_t dim,
                           int32_t rows_per_batch, vb_stream_t stream) {
  VB_REQUIRE(x && y && out, VB_ERR_INVALID, "null argument");
  int rc = launch_gate_residual(x, y, gate, out, rows, dim, rows_per_batch, static_cast<cudaStream_t>(stream));
  if (rc == VB_OK) ++g_launches;
  return rc;
}
int vb_block_rmsnorm_rope(const void* x, const void* weight, const float* cos_tab, const float* sin_tab, void* out,
                          int64_t rows, int32_t dim, int32_t tokens_per_batch, float eps, vb_stream_t stream) {
  VB_REQUIRE(x && weight && out, VB_ERR_INVALID, "null argument");
  VB_REQUIRE((cos_tab == nullptr) == (sin_tab == nullptr), VB_ERR_INVALID, "cos and sin tables come together");
  int rc = launch_rmsnorm_rope(x, weight, cos_tab, sin_tab, out, rows, dim, tokens_per_batch, eps,
                               static_cast<cudaStream_t>(stream));
  if (rc == VB_OK) ++g_launches;
  return rc;
}

int vb_block_headnorm_rope(const void* x, const void* weight, const float* cos_tab, const float* sin_tab, void* out,
                           int32_t batch, int32_t rows, int32_t heads, int32_t rope_rows, int32_t dst_rows,
                           int32_t dst_row0, float eps, vb_stream_t stream) {
  VB_REQUIRE(x && out, VB_ERR_INVALID, "null argument");
  int rc = launch_headnorm_rope(x, weight, cos_tab, sin_tab, out, batch, rows, heads, rope_rows, dst_rows, dst_row0, eps,
                                static_cast<cudaStream_t>(stream));
  if (rc == VB_OK) ++g_launches;
  return rc;
}

void vb_timing_enable(int on) { g_timing = on != 0; }

int vb_timing_collect_kinds(double* kernel_ms, int64_t* launches, double* flops) {
  for (int k = 0; k < VB_TIMING_KINDS; ++k) {
    if (kernel_ms) kernel_ms[k] = 0.0;
    if (launches) launches[k] = 0;
    if (flops) flops[k] = 0.0;
  }
  for (auto& e : g_events) {
    VB_CUDA_OK(cudaEventSynchronize(e.ev1));
    float ms = 0.f;
    VB_CUDA_OK(cudaEventElapsedTime(&ms, e.ev0, e.ev1));
    const int k = e.kind >= 0 && e.kind < VB_TIMING_KINDS ? e.kind : 0;
    if (kernel_ms) kernel_ms[k] += ms;
    if (launches) launches[k] += 1;
    if (flops) flops[k] += e.flops;
    cudaEventDestroy(e.ev0);
    cudaEventDestroy(e.ev1);
  }
  g_events.clear();
  return VB_OK;
}

int vb_timing_collect(double* kernel_ms, int64_t* launches, double* flops) {
  double ms[VB_TIMING_KINDS], fl[VB_TIMING_KINDS];
  int64_t n[VB_TIMING_KINDS];
  const int rc = vb_timing_collect_kinds(ms, n, fl);
  if (rc != VB_OK) return rc;
  if (kernel_ms) *kernel_ms = 0.0;
  if (launches) *launches = 0;
  if (flops) *flops = 0.0;
  for (int k = 0; k < VB_TIMING_KINDS; ++k) {
    if (kernel_ms) *kernel_ms += ms[k];
    if (launches) *launches += n[k];
    if (flops) *flops += fl[k];
  }
  return VB_OK;
}

void vb_stats_reset(void) {
  g_launches = 0;
  g_flops = 0.0;
}
int64_t vb_stats_launches(void) { return g_launches; }
double vb_stats_attn_flops(void) { return g_flops; }

int vb_ulysses_pack_heads(const void* x, void* send, int32_t s_loc, int32_t heads, int32_t world, int32_t n_tensors,
                          int64_t x_tensor_stride, int64_t send_tensor_stride, const int32_t* head_at,
                          vb_stream_t stream) {
  VB_REQUIRE(x && send, VB_ERR_INVALID, "null argument");
  int rc = launch_ulysses_permute(x, send, s_loc, heads, world, n_tensors, x_tensor_stride, send_tensor_stride, 1,
                                  head_at, static_cast<cudaStream_t>(stream));
  if (rc == VB_OK) ++g_launches;
  return rc;
}
int vb_ulysses_pack_qkv(const void* q, const void* k, const void* v, const int64_t* stride_s, const int64_t* stride_h,
                        void* send, int32_t s_loc, int32_t heads, int32_t world, const int32_t* head_at,
                        vb_stream_t stream) {
  VB_REQUIRE(q && k && v && send && stride_s && stride_h, VB_ERR_INVALID, "null argument");
  int rc = launch_ulysses_pack_qkv(q, k, v, stride_s, stride_h, send, s_loc, heads, world, head_at,
                                   static_cast<cudaStream_t>(stream));
  if (rc == VB_OK) ++g_launches;
  return rc;
}
int vb_ulysses_scatter_qkv_slots(const void* q, const void* k, const void* v, const int64_t* stride_s,
                                 const int64_t* stride_h, void* const* peer_qkv, int64_t rows_total, int32_t s_loc,
                                 int32_t slots, int32_t world, int32_t rank, const int32_t* entry_peer,
                                 const int32_t* entry_slot, const int32_t* entry_head, int32_t n_entries,
                                 vb_stream_t stream) {
  VB_REQUIRE(q && k && v && stride_s && stride_h && peer_qkv && entry_peer && entry_slot && entry_head, VB_ERR_INVALID,
             "null argument");
  int rc = launch_ulysses_scatter_slots(q, k, v, stride_s, stride_h, peer_qkv, rows_total, s_loc, slots, world, rank,
                                        entry_peer, entry_slot, entry_head, n_entries, static_cast<cudaStream_t>(stream));
  if (rc == VB_OK) ++g_launches;
  return rc;
}
int vb_ulysses_unpack_heads(const void* recv, void* y, int32_t s_loc, int32_t heads, int32_t world,
                            const int32_t* head_at, vb_stream_t stream) {
  VB_REQUIRE(recv && y, VB_ERR_INVALID, "null argument");
  int rc = launch_ulysses_permute(recv, y, s_loc, heads, world, 1, 0, 0, 0, head_at,
                                  static_cast<cudaStream_t>(stream));
  if (rc == VB_OK) ++g_launches;
  return rc;
}

}  // extern "C"
