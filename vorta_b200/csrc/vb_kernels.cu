// vb_kernels.cu — the HBM-bound kernels of the path: coreset similarity selection, row gather (pooling and
// tile-major layout), router head, zero-fill of padded text rows and the Ulysses pack / unpack passes.
// These are byte / index kernels: 16-byte vector accesses, one warp per small work unit, grids in multiples of
// the SM count.  No tensor cores here on purpose.
#include <string.h>

#include <algorithm>

#include "vb_common.cuh"

namespace vb {

__device__ __forceinline__ uint4 ld_stream(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void bf16x8_to_double(const uint4& v, double (&d)[8]) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    d[2 * i + 0] = static_cast<double>(__uint_as_float(w[i] << 16));
    d[2 * i + 1] = static_cast<double>(__uint_as_float(w[i] & 0xffff0000u));
  }
}

// ------------------------------------------------------------------------------------------------
// Coreset selection (reference: vorta/attention/coreset_select.py:91-113)
//   one warp per (batch, head, group).  The ranking contract is the fp64 one: <c, m>, |m|^2 and |c|^2 accumulated in
//   fp64, cosine similarities of the g-1 margins ranked by counting (ascending, ties -> lower margin position first).
//   fp64 on this part costs one F2F conversion per element (16 / clk / SM) and caps the kernel at ~1/5 of HBM speed
//   (round-1 measurement), so the similarities are first computed in fp32 — products of two bf16 values are exact
//   in fp32, only the 127 additions round — with a rigorous error bound; the group is recomputed in fp64 only when
//   two similarities are closer than that bound can separate (or a norm leaves the range where the bound holds).
//   Both paths therefore produce the ranking of the fp64 computation.
//
//   fast path : 8 lanes per 256-byte token row (32 B per lane), 4 rows per warp step, every row of the group
//               requested before the first is used (4.6 KB in flight per warp at 17 margins, 24 warps per SM).
//   bound     : |cos32 - cos| <= 127 u (1 + |cos|) + O(u) < 1.6e-5 with u = 2^-24 when |c|^2, |m|^2 are normal fp32
//               numbers >= 1e-30; two similarities further apart than kSimGap = 4e-5 cannot swap.
// ------------------------------------------------------------------------------------------------
constexpr int kSelectWarps = 8;
constexpr float kSimGap = 4e-5f;

__device__ __forceinline__ void bf16x8_to_float(const uint4& v, float (&f)[8]) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f[2 * i + 0] = __uint_as_float(w[i] << 16);
    f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}

// fp64 similarities of one group into sim[0 .. n_margin): a half-warp (16 lanes x 16 B) streams one row
__device__ __noinline__ void select_sims_fp64(const __nv_bfloat16* base, int64_t stride_s, int ctok, const int32_t* mtok,
                                              int n_margin, double* sim) {
  const int lane = threadIdx.x & 31;
  const int half = lane >> 4, hl = lane & 15;
  double c[8];
  bf16x8_to_double(ld_stream(reinterpret_cast<const uint4*>(base + ctok * stride_s) + hl), c);
  double cn = 0.0;
#pragma unroll
  for (int i = 0; i < 8; ++i) cn = fma(c[i], c[i], cn);
#pragma unroll
  for (int o = 8; o >= 1; o >>= 1) cn += __shfl_xor_sync(0xffffffffu, cn, o);
  const double c_norm = fmax(sqrt(cn), 1e-12);   // F.normalize eps
  for (int m0 = 0; m0 < n_margin; m0 += 2) {
    const int m = m0 + half;
    double dot = 0.0, mn = 0.0;
    if (m < n_margin) {
      double v[8];
      bf16x8_to_double(ld_stream(reinterpret_cast<const uint4*>(base + mtok[m] * stride_s) + hl), v);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        dot = fma(c[i], v[i], dot);
        mn = fma(v[i], v[i], mn);
      }
    }
#pragma unroll
    for (int o = 8; o >= 1; o >>= 1) {
      dot += __shfl_xor_sync(0xffffffffu, dot, o);
      mn += __shfl_xor_sync(0xffffffffu, mn, o);
    }
    if (hl == 0 && m < n_margin) sim[m] = dot / (c_norm * fmax(sqrt(mn), 1e-12));
  }
}

// NSTEPS = ceil(n_margin / 4) is a template parameter so that a lane holds exactly the rows it needs.  8 lanes share a
// 256-byte token row (32 B per lane), 4 rows per warp step: 2 * NSTEPS 16-byte loads in flight per lane and ~80 registers,
// so that three CTAs (24 warps, each with a whole group of rows requested) fit an SM.  (Round 1: 4 lanes per row, 128
// registers, two CTAs per SM: 2.1 TB/s = 0.32 of the copy bandwidth, latency-bound.)
#ifndef VB_SELECT_CTAS
#define VB_SELECT_CTAS 3
#endif
template <int NSTEPS>
__global__ void __launch_bounds__(kSelectWarps * 32, VB_SELECT_CTAS) vb_coreset_select_kernel(const SelectParams p) {
  __shared__ double s_sim[kSelectWarps][32];
  __shared__ float s_simf[kSelectWarps][32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int lig = lane & 7, rg = lane >> 3;      // lane inside a row's 8-lane group, row slot 0..3 of a step
  const int64_t total = static_cast<int64_t>(p.batch) * p.heads * p.G;
  const int n_p = p.n_margin - p.n_unpooled;
  const int row_len = p.G * (1 + p.n_unpooled) + p.text_len;   // kept_tok row length

  // units are ordered head-fastest: neighbouring warps read the same tokens of neighbouring heads, which sit next to
  // each other in the (B, S, H, 128) memory the projections produce (one DRAM page instead of H pages 10 KB apart)
  for (int64_t unit = static_cast<int64_t>(blockIdx.x) * kSelectWarps + warp; unit < total;
       unit += static_cast<int64_t>(gridDim.x) * kSelectWarps) {
    const int hs = static_cast<int>(unit % p.heads);
    const int grp = static_cast<int>((unit / p.heads) % p.G);
    const int b = static_cast<int>(unit / (static_cast<int64_t>(p.G) * p.heads));
    const int h_src = p.head_list.head(hs);
    const __nv_bfloat16* base = p.x + b * p.stride_b + h_src * p.stride_h;
    const int ctok = p.center_tok[grp];
    const int32_t* mtok = p.margin_tok + static_cast<int64_t>(grp) * p.n_margin;
    const int my_tok = lane < p.n_margin ? mtok[lane] : 0;       // lane i holds the token of margin i

    // ---- fast path: request every row of the group, then fp32 dot products / norms ----
    uint4 raw[NSTEPS][2];
#pragma unroll
    for (int s = 0; s < NSTEPS; ++s) {
      const int m = s * 4 + rg;
      const int tok = __shfl_sync(0xffffffffu, my_tok, m & 31);
      if (m < p.n_margin) {
        const uint4* row = reinterpret_cast<const uint4*>(base + tok * p.stride_s);
        raw[s][0] = ld_stream(row + lig);            // the 8 lanes of a row cover 128 B per load instruction
        raw[s][1] = ld_stream(row + 8 + lig);
      }
    }
    float c[2][8];
    float cn = 0.f;
    {
      const uint4* crow = reinterpret_cast<const uint4*>(base + ctok * p.stride_s);
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        bf16x8_to_float(__ldg(crow + j * 8 + lig), c[j]);      // the 4 row groups read the same bytes: L1
#pragma unroll
        for (int i = 0; i < 8; ++i) cn = fmaf(c[j][i], c[j][i], cn);
      }
      cn += __shfl_xor_sync(0xffffffffu, cn, 1);
      cn += __shfl_xor_sync(0xffffffffu, cn, 2);
      cn += __shfl_xor_sync(0xffffffffu, cn, 4);
    }
    const bool c_ok = cn >= 1e-30f && cn < INFINITY;
    const float c_norm = sqrtf(cn);
#pragma unroll
    for (int s = 0; s < NSTEPS; ++s) {
      const int m = s * 4 + rg;
      float dot = 0.f, mn = 0.f;
      if (m < p.n_margin) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          float v[8];
          bf16x8_to_float(raw[s][j], v);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            dot = fmaf(c[j][i], v[i], dot);
            mn = fmaf(v[i], v[i], mn);
          }
        }
      }
#pragma unroll
      for (int o = 1; o <= 4; o <<= 1) {
        dot += __shfl_xor_sync(0xffffffffu, dot, o);
        mn += __shfl_xor_sync(0xffffffffu, mn, o);
      }
      if (lig == 0 && m < p.n_margin) {
        const bool ok = c_ok && mn >= 1e-30f && mn < INFINITY;
        const float cosv = ok ? dot / (c_norm * sqrtf(mn)) : NAN;
        s_simf[warp][m] = cosv;
        s_sim[warp][m] = static_cast<double>(cosv);
      }
    }
    __syncwarp();

    // ---- can fp32 separate every pair?  (NaN marks a row outside the bound's range) ----
    bool unsure = false;
    if (lane < p.n_margin) {
      const float mine = s_simf[warp][lane];
      for (int j = 0; j < p.n_margin; ++j) {
        const float d = fabsf(s_simf[warp][j] - mine);
        unsure |= j != lane && !(d >= kSimGap);      // also true when either value is NaN
      }
    }
    if (__any_sync(0xffffffffu, unsure)) {
      __syncwarp();
      select_sims_fp64(base, p.stride_s, ctok, mtok, p.n_margin, s_sim[warp]);
    }
    __syncwarp();

    if (lane < p.n_margin) {
      const double mine = s_sim[warp][lane];
      int rank = 0;
      for (int j = 0; j < p.n_margin; ++j) {
        const double o = s_sim[warp][j];
        rank += (o < mine) || (o == mine && j < lane);
      }
      const int64_t bh = static_cast<int64_t>(b) * p.heads + hs;
      const int tok = my_tok;
      if (rank < p.n_unpooled) {
        if (p.unpooled_argsort) p.unpooled_argsort[(bh * p.G + grp) * p.n_unpooled + rank] = lane;
        if (p.kept_tok) p.kept_tok[bh * row_len + p.G + static_cast<int64_t>(grp) * p.n_unpooled + rank] = tok;
      } else {
        if (p.pooled_argsort) p.pooled_argsort[(bh * p.G + grp) * n_p + (rank - p.n_unpooled)] = lane;
        if (p.dropped_tok) p.dropped_tok[(bh * p.G + grp) * n_p + (rank - p.n_unpooled)] = tok;
      }
      if (lane == 0 && p.kept_tok) p.kept_tok[bh * row_len + grp] = ctok;
    }
    // text rows keep their position behind the pooled video rows
    if (p.kept_tok && grp == 0) {
      const int64_t bh = static_cast<int64_t>(b) * p.heads + hs;
      for (int i = lane; i < p.text_len; i += 32)
        p.kept_tok[bh * row_len + p.G * (1 + p.n_unpooled) + i] = p.seq_len + i;
    }
    __syncwarp();
  }
}

// Groups of more than 33 tokens (lowres windows such as (2,4,6), (4,4,4), (2,6,6)): still one warp per group and the
// same contract — fp32 filter with the same bound (it does not depend on g), fp64 recheck, ranking by counting with the
// same tie-break — but the similarities live in dynamic shared memory and the rows are streamed in chunks of
// 4 * kLargeSteps margins, so any group size up to kSelectMaxGroup runs the same code.
//   shared memory per warp: n_margin doubles (fp64 sims) + n_margin floats (fp32 sims) = 12 B per margin.  The
//   margin-by-rank table needs n_margin int32 as well; it lives in whichever of the two arrays the decision no longer
//   reads (fp32 decision: the double array; fp64 decision: the float array), so 12 B per margin is all.
//   fp32 decision without an n^2 gap test: rank the fp32 sims by counting, then every pair is at least kSimGap apart
//   iff every pair of rank neighbours is — one linear pass over the margin-by-rank table.
constexpr int kLargeWarps = kSelectLargeWarps;
constexpr int kLargeSteps = 4;                  // 16 margin rows (4 KB) in flight per warp
static_assert(kLargeWarps * (kSelectMaxGroup - 1) * 12 <= kSelectSmemCap, "selection smem exceeds 227 KB");

__global__ void __launch_bounds__(kLargeWarps * 32, 4) vb_coreset_select_large_kernel(const SelectParams p) {
  extern __shared__ __align__(16) unsigned char s_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int lig = lane & 7, rg = lane >> 3;
  const int n = p.n_margin;
  double* s_sim = reinterpret_cast<double*>(s_raw) + static_cast<int64_t>(warp) * n;
  float* s_simf = reinterpret_cast<float*>(reinterpret_cast<double*>(s_raw) + static_cast<int64_t>(kLargeWarps) * n) +
                  static_cast<int64_t>(warp) * n;
  const int64_t total = static_cast<int64_t>(p.batch) * p.heads * p.G;
  const int n_p = n - p.n_unpooled;
  const int row_len = p.G * (1 + p.n_unpooled) + p.text_len;

  for (int64_t unit = static_cast<int64_t>(blockIdx.x) * kLargeWarps + warp; unit < total;
       unit += static_cast<int64_t>(gridDim.x) * kLargeWarps) {
    const int hs = static_cast<int>(unit % p.heads);
    const int grp = static_cast<int>((unit / p.heads) % p.G);
    const int b = static_cast<int>(unit / (static_cast<int64_t>(p.G) * p.heads));
    const int h_src = p.head_list.head(hs);
    const __nv_bfloat16* base = p.x + b * p.stride_b + h_src * p.stride_h;
    const int ctok = p.center_tok[grp];
    const int32_t* mtok = p.margin_tok + static_cast<int64_t>(grp) * n;

    float c[2][8];
    float cn = 0.f;
    {
      const uint4* crow = reinterpret_cast<const uint4*>(base + ctok * p.stride_s);
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        bf16x8_to_float(__ldg(crow + j * 8 + lig), c[j]);
#pragma unroll
        for (int i = 0; i < 8; ++i) cn = fmaf(c[j][i], c[j][i], cn);
      }
      cn += __shfl_xor_sync(0xffffffffu, cn, 1);
      cn += __shfl_xor_sync(0xffffffffu, cn, 2);
      cn += __shfl_xor_sync(0xffffffffu, cn, 4);
    }
    const bool c_ok = cn >= 1e-30f && cn < INFINITY;
    const float c_norm = sqrtf(cn);

    // ---- fast path: fp32 similarities, 4 rows per warp step, kLargeSteps steps requested before the first is used
    for (int m0 = 0; m0 < n; m0 += 4 * kLargeSteps) {
      uint4 raw[kLargeSteps][2];
#pragma unroll
      for (int s = 0; s < kLargeSteps; ++s) {
        const int m = m0 + s * 4 + rg;
        if (m < n) {
          const uint4* row = reinterpret_cast<const uint4*>(base + __ldg(mtok + m) * p.stride_s);
          raw[s][0] = ld_stream(row + lig);
          raw[s][1] = ld_stream(row + 8 + lig);
        }
      }
#pragma unroll
      for (int s = 0; s < kLargeSteps; ++s) {
        const int m = m0 + s * 4 + rg;
        float dot = 0.f, mn = 0.f;
        if (m < n) {
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            float v[8];
            bf16x8_to_float(raw[s][j], v);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              dot = fmaf(c[j][i], v[i], dot);
              mn = fmaf(v[i], v[i], mn);
            }
          }
        }
#pragma unroll
        for (int o = 1; o <= 4; o <<= 1) {
          dot += __shfl_xor_sync(0xffffffffu, dot, o);
          mn += __shfl_xor_sync(0xffffffffu, mn, o);
        }
        if (lig == 0 && m < n) {
          const bool ok = c_ok && mn >= 1e-30f && mn < INFINITY;
          s_simf[m] = ok ? dot / (c_norm * sqrtf(mn)) : NAN;
        }
      }
    }
    __syncwarp();

    // ---- fp32 decision: no NaN, and rank neighbours at least kSimGap apart.  by_rank[r] = margin of rank r.
    bool unsure = false;
    for (int m = lane; m < n; m += 32) unsure |= isnan(s_simf[m]);
    unsure = __any_sync(0xffffffffu, unsure);
    int32_t* by_rank = reinterpret_cast<int32_t*>(s_sim);
    if (!unsure) {
      for (int m = lane; m < n; m += 32) {
        const float mine = s_simf[m];
        int rank = 0;
        for (int j = 0; j < n; ++j) {
          const float o = s_simf[j];
          rank += (o < mine) || (o == mine && j < m);
        }
        by_rank[rank] = m;
      }
      __syncwarp();
      for (int r = lane + 1; r < n; r += 32) unsure |= !(s_simf[by_rank[r]] - s_simf[by_rank[r - 1]] >= kSimGap);
      unsure = __any_sync(0xffffffffu, unsure);
    }
    if (unsure) {   // fp64 similarities over the double array, ranked into the float array
      __syncwarp();
      select_sims_fp64(base, p.stride_s, ctok, mtok, n, s_sim);
      __syncwarp();
      by_rank = reinterpret_cast<int32_t*>(s_simf);
      for (int m = lane; m < n; m += 32) {
        const double mine = s_sim[m];
        int rank = 0;
        for (int j = 0; j < n; ++j) {
          const double o = s_sim[j];
          rank += (o < mine) || (o == mine && j < m);
        }
        by_rank[rank] = m;
      }
    }
    __syncwarp();

    const int64_t bh = static_cast<int64_t>(b) * p.heads + hs;
    for (int r = lane; r < n; r += 32) {
      const int m = by_rank[r];
      const int tok = __ldg(mtok + m);
      if (r < p.n_unpooled) {
        if (p.unpooled_argsort) p.unpooled_argsort[(bh * p.G + grp) * p.n_unpooled + r] = m;
        if (p.kept_tok) p.kept_tok[bh * row_len + p.G + static_cast<int64_t>(grp) * p.n_unpooled + r] = tok;
      } else {
        if (p.pooled_argsort) p.pooled_argsort[(bh * p.G + grp) * n_p + (r - p.n_unpooled)] = m;
        if (p.dropped_tok) p.dropped_tok[(bh * p.G + grp) * n_p + (r - p.n_unpooled)] = tok;
      }
    }
    if (lane == 0 && p.kept_tok) p.kept_tok[bh * row_len + grp] = ctok;
    if (p.kept_tok && grp == 0)
      for (int i = lane; i < p.text_len; i += 32) p.kept_tok[bh * row_len + p.G * (1 + p.n_unpooled) + i] = p.seq_len + i;
    __syncwarp();   // the next unit overwrites this warp's shared arrays
  }
}

// Groups of up to 33 tokens (32 margins) run the warp kernel above, larger ones the shared-memory kernel; both produce
// the tables of the fp64 ranking, so which kernel ran a group does not show in its output.
int launch_coreset_select(const SelectParams& p, cudaStream_t stream) {
  const int64_t total = static_cast<int64_t>(p.batch) * p.heads * p.G;
  if (total == 0) return VB_OK;
  VB_REQUIRE(p.n_margin >= 1 && p.n_margin + 1 <= kSelectMaxGroup, VB_ERR_UNSUPPORTED,
             "coreset group of %d tokens exceeds the selection kernel's maximum of %d tokens", p.n_margin + 1,
             kSelectMaxGroup);
  if (p.n_margin > 32) {
    const int smem = kLargeWarps * p.n_margin * 12;
    if (smem > 48 * 1024)   // beyond the default limit (groups above 1025 tokens): opt in, on the current device
      VB_CUDA_OK(cudaFuncSetAttribute(vb_coreset_select_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const int64_t blocks_needed = (total + kLargeWarps - 1) / kLargeWarps;
    const int grid = static_cast<int>(blocks_needed < 148 * 16 ? blocks_needed : 148 * 16);
    vb_coreset_select_large_kernel<<<grid, kLargeWarps * 32, smem, stream>>>(p);
    VB_CUDA_OK(cudaGetLastError());
    return VB_OK;
  }
  const int64_t blocks_needed = (total + kSelectWarps - 1) / kSelectWarps;
  const int grid = static_cast<int>(blocks_needed < 148 * 12 ? blocks_needed : 148 * 12);
  const int steps = (p.n_margin + 3) >> 2;        // 4 margin rows per warp step
  if (steps <= 2) vb_coreset_select_kernel<2><<<grid, kSelectWarps * 32, 0, stream>>>(p);
  else if (steps <= 3) vb_coreset_select_kernel<3><<<grid, kSelectWarps * 32, 0, stream>>>(p);
  else if (steps <= 5) vb_coreset_select_kernel<5><<<grid, kSelectWarps * 32, 0, stream>>>(p);
  else vb_coreset_select_kernel<8><<<grid, kSelectWarps * 32, 0, stream>>>(p);
  VB_CUDA_OK(cudaGetLastError());
  return VB_OK;
}

// ------------------------------------------------------------------------------------------------
// Matching tables -> token tables (reference: coreset_select.py:157-166), one thread per (b, h, group, margin)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) vb_coreset_tables_kernel(const TablesParams p) {
  const int n_p = p.n_margin - p.n_unpooled;
  const int S_c = p.G * (1 + p.n_unpooled);
  const int row_len = S_c + p.text_len;
  const int64_t total = static_cast<int64_t>(p.batch) * p.heads * p.G * (p.n_margin + 1);
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int j = static_cast<int>(i % (p.n_margin + 1));      // 0 = centre, 1.. = sorted margin rank j-1
    const int64_t u = i / (p.n_margin + 1);
    const int grp = static_cast<int>(u % p.G);
    const int64_t bh = u / p.G;
    if (j == 0) {
      const int tok = p.center_tok[grp];
      if (p.kept_tok) p.kept_tok[bh * row_len + grp] = tok;
      if (p.unpool_src) p.unpool_src[bh * p.seq_len + tok] = grp;
      if (p.kept_tok && grp == 0)
        for (int t = 0; t < p.text_len; ++t) p.kept_tok[bh * row_len + S_c + t] = p.seq_len + t;
      continue;
    }
    const int rank = j - 1;
    if (rank < p.n_unpooled) {
      const int pos = static_cast<int>(p.unpooled_argsort[(bh * p.G + grp) * p.n_unpooled + rank]);
      const int tok = p.margin_tok[static_cast<int64_t>(grp) * p.n_margin + pos];
      const int row = p.G + grp * p.n_unpooled + rank;
      if (p.kept_tok) p.kept_tok[bh * row_len + row] = tok;
      if (p.unpool_src) p.unpool_src[bh * p.seq_len + tok] = row;
    } else {
      const int r = rank - p.n_unpooled;
      const int pos = static_cast<int>(p.pooled_argsort[(bh * p.G + grp) * n_p + r]);
      const int tok = p.margin_tok[static_cast<int64_t>(grp) * p.n_margin + pos];
      if (p.dropped_tok) p.dropped_tok[(bh * p.G + grp) * n_p + r] = tok;
      if (p.unpool_src) p.unpool_src[bh * p.seq_len + tok] = grp;   // dropped margins copy their centre
    }
  }
}

int launch_coreset_tables(const TablesParams& p, cudaStream_t stream) {
  const int64_t total = static_cast<int64_t>(p.batch) * p.heads * p.G * (p.n_margin + 1);
  if (total == 0) return VB_OK;
  const int grid = static_cast<int>((total + 255) / 256 < 148 * 8 ? (total + 255) / 256 : 148 * 8);
  vb_coreset_tables_kernel<<<grid, 256, 0, stream>>>(p);
  VB_CUDA_OK(cudaGetLastError());
  return VB_OK;
}

// ------------------------------------------------------------------------------------------------
// Row gather: dst[t][b, hs, i, :] = src[t][b, head_list[hs], map[b, hs, i], :], up to 3 tensors per launch
// (reference: coreset_select.py:91-93,118-123 pooling; tile.py:7-41 tile-major layout)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) vb_gather_rows_kernel(const GatherParams p) {
  // half-warp per row: 16 lanes x 16 B = one 256-byte row; 4 rows in flight per half-warp for latency hiding
  const int lane16 = threadIdx.x & 15;
  const int64_t hw = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 4;
  const int64_t n_hw = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 4;
  const int64_t rows_per_tensor = static_cast<int64_t>(p.batch) * p.heads * p.n_rows;
  const int64_t total = rows_per_tensor * p.n_tensors;
  for (int64_t r0 = hw * 4; r0 < total; r0 += n_hw * 4) {
    uint4 val[4];
    uint4* dptr[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t r = r0 + u;
      dptr[u] = nullptr;
      if (r < total) {
        const int t = static_cast<int>(r / rows_per_tensor);
        int64_t rr = r % rows_per_tensor;
        const int i = static_cast<int>(rr % p.n_rows);
        rr /= p.n_rows;
        const int hs = static_cast<int>(rr % p.heads);
        const int b = static_cast<int>(rr / p.heads);
        const int h_src = p.head_list.head(hs);
        const int32_t* map = (t == 0 && p.map0 != nullptr) ? p.map0 : p.map;
        const int src_row = map ? map[b * p.map_stride_b + hs * p.map_stride_h + i] : i;
        const __nv_bfloat16* s = p.src[t] + b * p.src_stride[t][0] + h_src * p.src_stride[t][1] +
                                 static_cast<int64_t>(src_row) * p.src_stride[t][2];
        val[u] = ld_stream(reinterpret_cast<const uint4*>(s) + lane16);
        dptr[u] = reinterpret_cast<uint4*>(p.dst[t] + b * p.dst_stride[0] + hs * p.dst_stride[1] +
                                           static_cast<int64_t>(i) * p.dst_stride[2]) + lane16;
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (dptr[u]) *dptr[u] = val[u];
  }
}

int launch_gather_rows(const GatherParams& p, cudaStream_t stream) {
  const int64_t total = static_cast<int64_t>(p.batch) * p.heads * p.n_rows * p.n_tensors;
  if (total == 0) return VB_OK;
  const int64_t blocks_needed = (total / 4 * 16 + 255) / 256 + 1;
  const int grid = static_cast<int>(blocks_needed < 148 * 16 ? blocks_needed : 148 * 16);
  vb_gather_rows_kernel<<<grid, 256, 0, stream>>>(p);
  VB_CUDA_OK(cudaGetLastError());
  return VB_OK;
}

// ------------------------------------------------------------------------------------------------
// Zero rows [row0[b], row_end) of every (batch b, listed output head): padded text queries produce 0 (hunyuan.py:176);
// each sample has its own number of padded rows, the grid covers the largest
// ------------------------------------------------------------------------------------------------
__global__ void vb_zero_rows_kernel(const ZeroRowsParams p) {
  const int64_t total = static_cast<int64_t>(p.batch) * p.n_heads * p.n_rows * 16;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i & 15);
    int64_t r = i >> 4;
    const int row = p.row_end - p.n_rows + static_cast<int>(r % p.n_rows);
    r /= p.n_rows;
    const int h = p.head[r % p.n_heads];
    const int b = static_cast<int>(r / p.n_heads);
    if (row < p.row0[b]) continue;        // a valid text row of this sample
    reinterpret_cast<uint4*>(p.out + b * p.stride_b + h * p.stride_h + static_cast<int64_t>(row) * p.stride_s)[c] =
        make_uint4(0, 0, 0, 0);
  }
}
int launch_zero_rows(const ZeroRowsParams& p, cudaStream_t stream) {
  const int64_t total = static_cast<int64_t>(p.batch) * p.n_heads * p.n_rows * 16;
  if (total == 0) return VB_OK;
  const int grid = static_cast<int>((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184);
  vb_zero_rows_kernel<<<grid, 256, 0, stream>>>(p);
  VB_CUDA_OK(cudaGetLastError());
  return VB_OK;
}

// ------------------------------------------------------------------------------------------------
// Router (reference: vorta/patch/router.py:33-43 and wan.py:396-400), fp32, all layers of a step in one launch.
//   grid (n_layers, batch); the block stages silu(temb[b]) in shared memory, warps own output rows.
// ------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ float to_f32(T v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

// bf16 routers (the reference's inference default, scripts/wan/inference.py:132 router_dtype=torch.bfloat16): torch
// rounds after every module — SiLU output, Linear output (fp32 accumulate, one rounding), Softmax output — and the
// top-1 / threshold compare then sees bf16 scores.  With bf16 weights the kernel rounds at the same three points, so
// heads whose fp32 scores are closer than a bf16 ulp tie (-> lowest expert index) exactly like they do there.
template <typename T>
struct RoundLike {
  static __device__ __forceinline__ float r(float v) { return v; }
};
template <>
struct RoundLike<__nv_bfloat16> {
  static __device__ __forceinline__ float r(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
};

template <typename TE, typename TW>
__global__ void __launch_bounds__(256)
vb_router_kernel(const TE* temb, const TW* w, const TW* bias, int64_t w_layer_stride, int64_t bias_layer_stride,
                 int embed_dim, int heads, float tau, float* scores, int32_t* branch) {
  extern __shared__ float s_buf[];   // embed_dim silu values, then 3*heads logits
  float* s_act = s_buf;
  float* s_logit = s_buf + embed_dim;
  const int layer = blockIdx.x, b = blockIdx.y, batch = gridDim.y;
  const int n_out = heads * 3;
  for (int i = threadIdx.x; i < embed_dim; i += blockDim.x) {
    const float x = to_f32(temb[static_cast<int64_t>(b) * embed_dim + i]);
    s_act[i] = RoundLike<TW>::r(x / (1.f + expf(-x)));   // SiLU
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n_warps = blockDim.x >> 5;
  const TW* wl = w + layer * w_layer_stride;
  for (int o = warp; o < n_out; o += n_warps) {
    const TW* row = wl + static_cast<int64_t>(o) * embed_dim;
    float acc = 0.f;
    for (int i = lane; i < embed_dim; i += 32) acc = fmaf(to_f32(row[i]), s_act[i], acc);
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) s_logit[o] = RoundLike<TW>::r(acc + to_f32(bias[layer * bias_layer_stride + o]));
  }
  __syncthreads();
  for (int h = threadIdx.x; h < heads; h += blockDim.x) {
    const float l0 = s_logit[3 * h], l1 = s_logit[3 * h + 1], l2 = s_logit[3 * h + 2];
    const float mx = fmaxf(l0, fmaxf(l1, l2));
    const float e0 = expf(l0 - mx), e1 = expf(l1 - mx), e2 = expf(l2 - mx);
    const float inv = 1.f / (e0 + e1 + e2);
    const float p0 = RoundLike<TW>::r(e0 * inv), p1 = RoundLike<TW>::r(e1 * inv), p2 = RoundLike<TW>::r(e2 * inv);
    float* sc = scores + ((static_cast<int64_t>(layer) * batch + b) * heads + h) * 3;
    sc[0] = p0; sc[1] = p1; sc[2] = p2;
    if (b == 0 && branch != nullptr) {   // the first sample decides for the whole batch (wan.py:398)
      int best = 0;
      float bs = p0;
      if (p1 > bs) { best = 1; bs = p1; }
      if (p2 > bs) { best = 2; bs = p2; }
      if (bs < RoundLike<TW>::r(tau)) best = 0;            // NaN tau compares false: no threshold
      branch[layer * heads + h] = best;
    }
  }
}

int launch_router(const void* temb, int temb_dtype, const void* w, const void* bias, int w_dtype,
                  int64_t w_layer_stride, int64_t bias_layer_stride, int n_layers, int batch, int embed_dim,
                  int heads, float tau, float* scores, int32_t* branch, cudaStream_t stream) {
  if (n_layers == 0 || batch == 0) return VB_OK;
  dim3 grid(n_layers, batch);
  const size_t smem = (static_cast<size_t>(embed_dim) + 3 * heads) * sizeof(float);
  VB_REQUIRE(smem <= 48 * 1024, VB_ERR_UNSUPPORTED, "router: embedding dim %d too large", embed_dim);
#define VB_ROUTER_LAUNCH(TE, TW)                                                                            \
  vb_router_kernel<TE, TW><<<grid, 256, smem, stream>>>(static_cast<const TE*>(temb), static_cast<const TW*>(w), \
                                                        static_cast<const TW*>(bias), w_layer_stride,       \
                                                        bias_layer_stride, embed_dim, heads, tau, scores, branch)
  if (temb_dtype == VB_DTYPE_F32 && w_dtype == VB_DTYPE_F32) VB_ROUTER_LAUNCH(float, float);
  else if (temb_dtype == VB_DTYPE_BF16 && w_dtype == VB_DTYPE_BF16) VB_ROUTER_LAUNCH(__nv_bfloat16, __nv_bfloat16);
  else if (temb_dtype == VB_DTYPE_F32 && w_dtype == VB_DTYPE_BF16) VB_ROUTER_LAUNCH(float, __nv_bfloat16);
  else if (temb_dtype == VB_DTYPE_BF16 && w_dtype == VB_DTYPE_F32) VB_ROUTER_LAUNCH(__nv_bfloat16, float);
  else VB_REQUIRE(false, VB_ERR_INVALID, "router: unknown dtype codes %d / %d", temb_dtype, w_dtype);
#undef VB_ROUTER_LAUNCH
  VB_CUDA_OK(cudaGetLastError());
  return VB_OK;
}

// ------------------------------------------------------------------------------------------------
// Ulysses head pack / unpack (reference: vorta/ulysses/utils.py:60-74 and :84-89 transposes)
//   pack  : x (S_loc, H, 128) -> send (P, S_loc, H/P, 128)
//   unpack: recv (P, S_loc, H/P, 128) -> y (S_loc, H, 128)
// Both are a permutation of 256-byte head rows; one half-warp per row, 16-byte vectors.
// Slot (p, i) of the exchanged layout holds head `at[p * H/P + i]`: the identity for the reference's contiguous head
// chunks, or the cost-balanced assignment the host derives from the step's routing (SURVEY.md section 8e).
// ------------------------------------------------------------------------------------------------
struct HeadTable {
  uint8_t at[kMaxHeadTable];
};

static int fill_head_table(HeadTable& t, const int32_t* head_at, int heads) {
  VB_REQUIRE(heads <= kMaxHeadTable, VB_ERR_UNSUPPORTED, "at most %d heads per exchange, got %d", kMaxHeadTable, heads);
  uint8_t seen[kMaxHeadTable] = {0};
  for (int i = 0; i < heads; ++i) {
    const int h = head_at ? head_at[i] : i;
    VB_REQUIRE(h >= 0 && h < heads && !seen[h], VB_ERR_INVALID, "head_at is not a permutation of [0, %d) at slot %d",
               heads, i);
    seen[h] = 1;
    t.at[i] = static_cast<uint8_t>(h);
  }
  return VB_OK;
}

__global__ void __launch_bounds__(256)
vb_ulysses_permute_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, const HeadTable tab, int s_loc,
                          int heads, int world, int n_tensors, int64_t src_tensor_stride, int64_t dst_tensor_stride,
                          int pack) {
  const int hp = heads / world;
  const int64_t rows = static_cast<int64_t>(s_loc) * heads;
  const int64_t total = rows * n_tensors * 16;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i & 15);
    int64_t r = i >> 4;
    const int t = static_cast<int>(r / rows);
    r %= rows;
    // r indexes (token, slot); the head in that slot comes from the table
    const int slot = static_cast<int>(r % heads);
    const int64_t s = r / heads;
    const int h = tab.at[slot];
    const int64_t tm = (s * heads + h) * 16 + c;                                         // (S_loc, H, 128)
    const int64_t pm = ((static_cast<int64_t>(slot / hp) * s_loc + s) * hp + (slot % hp)) * 16 + c;  // (P, S_loc, H/P, 128)
    if (pack) dst[t * (dst_tensor_stride >> 3) + pm] = src[t * (src_tensor_stride >> 3) + tm];
    else dst[t * (dst_tensor_stride >> 3) + tm] = src[t * (src_tensor_stride >> 3) + pm];
  }
}

// q, k, v (S_loc, H, 128) with (token, head) strides -> send (3, P, S_loc, H/P, 128) in ONE pass; each tensor's
// (P, S_loc, H/P, 128) block is the send buffer of one equal-split all-to-all.
struct PackQkvParams {
  const uint4* src[3];
  int64_t stride_s[3], stride_h[3];   // elements
};

__global__ void __launch_bounds__(256)
vb_ulysses_pack_qkv_kernel(const PackQkvParams p, const HeadTable tab, uint4* __restrict__ send, int s_loc, int heads,
                           int world) {
  const int hp = heads / world;
  const int64_t rows = static_cast<int64_t>(s_loc) * heads;
  const int64_t total = rows * 3 * 16;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i & 15);
    int64_t r = i >> 4;
    const int t = static_cast<int>(r / rows);
    r %= rows;
    const int slot = static_cast<int>(r % heads);
    const int64_t s = r / heads;
    const int h = tab.at[slot];
    const int64_t dst = ((((static_cast<int64_t>(t) * world + slot / hp) * s_loc + s) * hp) + (slot % hp)) * 16 + c;
    send[dst] = p.src[t][(s * p.stride_s[t] + h * p.stride_h[t]) / 8 + c];
  }
}

int launch_ulysses_pack_qkv(const void* q, const void* k, const void* v, const int64_t* stride_s,
                            const int64_t* stride_h, void* send, int s_loc, int heads, int world,
                            const int32_t* head_at, cudaStream_t stream) {
  VB_REQUIRE(world > 0 && heads % world == 0, VB_ERR_INVALID, "heads %d not divisible by world %d", heads, world);
  PackQkvParams p;
  p.src[0] = static_cast<const uint4*>(q);
  p.src[1] = static_cast<const uint4*>(k);
  p.src[2] = static_cast<const uint4*>(v);
  for (int i = 0; i < 3; ++i) {
    VB_REQUIRE(stride_s[i] % 8 == 0 && stride_h[i] % 8 == 0, VB_ERR_INVALID,
               "strides must be multiples of 8 elements");
    p.stride_s[i] = stride_s[i];
    p.stride_h[i] = stride_h[i];
  }
  HeadTable tab;
  if (int rc = fill_head_table(tab, head_at, heads)) return rc;
  const int64_t total = static_cast<int64_t>(s_loc) * heads * 3 * 16;
  if (total == 0) return VB_OK;
  const int grid = static_cast<int>((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  vb_ulysses_pack_qkv_kernel<<<grid, 256, 0, stream>>>(p, tab, static_cast<uint4*>(send), s_loc, heads, world);
  VB_CUDA_OK(cudaGetLastError());
  return VB_OK;
}

struct ScatterQkvParams {
  const uint4* src[3];
  int64_t stride_s[3], stride_h[3];
  uint4* peer[8];
};
struct SlotTable {
  uint8_t peer[kMaxHeadTable], slot[kMaxHeadTable], head[kMaxHeadTable];
};
// The Ulysses "in" exchange as plain NVLink stores (16-byte vectors, 256-byte rows), no staging copy and no collective
// call: entry e = (peer, slot, head) stores head `head` of every local token of q, k, v into slot `slot` of peer
// `peer`'s receive buffer.  Order (tensor, entry, token) so that consecutive threads walk one peer's rows of one head.
__global__ void __launch_bounds__(256)
vb_ulysses_scatter_slots_kernel(const ScatterQkvParams p, const SlotTable tab, int n_entries, int64_t rows_total,
                                int s_loc, int slots, int rank) {
  const int64_t per_tensor = static_cast<int64_t>(n_entries) * s_loc;
  const int64_t total = per_tensor * 3 * 16;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i & 15);
    int64_t r = i >> 4;
    const int t = static_cast<int>(r / per_tensor);
    r -= t * per_tensor;
    const int e = static_cast<int>(r % n_entries);      // entry fastest: neighbouring threads read neighbouring heads of a token
    const int64_t sidx = r / n_entries;
    const uint4 val = p.src[t][(sidx * p.stride_s[t] + tab.head[e] * p.stride_h[t]) / 8 + c];
    const int64_t dst = ((static_cast<int64_t>(t) * rows_total + static_cast<int64_t>(rank) * s_loc + sidx) * slots +
                         tab.slot[e]) * 16 + c;
    p.peer[tab.peer[e]][dst] = val;
  }
}

int launch_ulysses_scatter_slots(const void* q, const void* k, const void* v, const int64_t* stride_s,
                                 const int64_t* stride_h, void* const* peer_qkv, int64_t rows_total, int s_loc, int slots,
                                 int world, int rank, const int32_t* entry_peer, const int32_t* entry_slot,
                                 const int32_t* entry_head, int n_entries, cudaStream_t stream) {
  VB_REQUIRE(world > 0 && world <= 8 && slots > 0 && slots <= 255, VB_ERR_INVALID, "world %d / slots %d not supported",
             world, slots);
  VB_REQUIRE(n_entries >= 0 && n_entries <= kMaxHeadTable, VB_ERR_UNSUPPORTED, "at most %d placement entries, got %d",
             kMaxHeadTable, n_entries);
  ScatterQkvParams p;
  p.src[0] = static_cast<const uint4*>(q);
  p.src[1] = static_cast<const uint4*>(k);
  p.src[2] = static_cast<const uint4*>(v);
  for (int i = 0; i < 3; ++i) {
    VB_REQUIRE(stride_s[i] % 8 == 0 && stride_h[i] % 8 == 0, VB_ERR_INVALID, "strides must be multiples of 8 elements");
    p.stride_s[i] = stride_s[i];
    p.stride_h[i] = stride_h[i];
  }
  for (int i = 0; i < 8; ++i) p.peer[i] = i < world ? static_cast<uint4*>(peer_qkv[i]) : nullptr;
  SlotTable tab;
  memset(&tab, 0, sizeof(tab));
  for (int e = 0; e < n_entries; ++e) {
    VB_REQUIRE(entry_peer[e] >= 0 && entry_peer[e] < world && entry_slot[e] >= 0 && entry_slot[e] < slots &&
                   entry_head[e] >= 0 && entry_head[e] < 256,
               VB_ERR_INVALID, "placement entry %d out of range (peer %d, slot %d, head %d)", e, entry_peer[e],
               entry_slot[e], entry_head[e]);
    tab.peer[e] = static_cast<uint8_t>(entry_peer[e]);
    tab.slot[e] = static_cast<uint8_t>(entry_slot[e]);
    tab.head[e] = static_cast<uint8_t>(entry_head[e]);
  }
  const int64_t total = static_cast<int64_t>(n_entries) * s_loc * 3 * 16;
  if (total == 0) return VB_OK;
  const int grid = static_cast<int>((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  vb_ulysses_scatter_slots_kernel<<<grid, 256, 0, stream>>>(p, tab, n_entries, rows_total, s_loc, slots, rank);
  VB_CUDA_OK(cudaGetLastError());
  return VB_OK;
}

int launch_ulysses_permute(const void* src, void* dst, int s_loc, int heads, int world, int n_tensors,
                           int64_t src_tensor_stride, int64_t dst_tensor_stride, int pack, const int32_t* head_at,
                           cudaStream_t stream) {
  VB_REQUIRE(world > 0 && heads % world == 0, VB_ERR_INVALID, "heads %d not divisible by world %d", heads, world);
  VB_REQUIRE(src_tensor_stride % 8 == 0 && dst_tensor_stride % 8 == 0, VB_ERR_INVALID,
             "tensor strides must be multiples of 8 elements");
  HeadTable tab;
  if (int rc = fill_head_table(tab, head_at, heads)) return rc;
  const int64_t total = static_cast<int64_t>(s_loc) * heads * n_tensors * 16;
  if (total == 0) return VB_OK;
  const int grid = static_cast<int>((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  vb_ulysses_permute_kernel<<<grid, 256, 0, stream>>>(static_cast<const uint4*>(src), static_cast<uint4*>(dst), tab,
                                                      s_loc, heads, world, n_tensors, src_tensor_stride,
                                                      dst_tensor_stride, pack);
  VB_CUDA_OK(cudaGetLastError());
  return VB_OK;
}

}  // namespace vb
