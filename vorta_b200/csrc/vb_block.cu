// vb_block.cu — fused elementwise kernels of the DiT block AROUND the attention path (SURVEY.md section 8f rows 1-2):
//   LayerNorm (+ affine) (+ adaLN modulate)          modeling_wan.py:205-206, 226, 232-234
//   gated residual  out = x + y * gate                modeling_wan.py:225, 238
//   RMSNorm-across-heads + RoPE on Q / K              wan.py:85-100 (reference: RMSNorm in bf16, RoPE in complex128)
// All HBM-bound: 16-byte vectors, fp32 math, a single read and a single write per element.  The row kernels give one
// WARP a token row (row widths that are multiples of 256 channels, i.e. every DiT here): the whole row is requested
// up front (dim/256 independent 16-byte loads per lane), statistics are warp shuffles only, and nothing waits on a
// CTA barrier; a CTA-per-row variant covers other widths.  (Round-1 ncu: the CTA-per-row LayerNorm reached 1.3 TB/s of
// algorithmic traffic — too few bytes in flight per SM and two CTA barriers per 3 KB row.)
#include "vb_common.cuh"

namespace vb {

constexpr int kRowThreads = 256;
constexpr int kMaxVec = 4;   // 16-byte vectors per thread -> rows up to 256 * 4 * 8 = 8192 channels

__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f[2 * i + 0] = __uint_as_float(w[i] << 16);
    f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  return make_uint4(pack2(f[0], f[1]), pack2(f[2], f[3]), pack2(f[4], f[5]), pack2(f[6], f[7]));
}
// block-wide sum of two values (blockDim.x == kRowThreads)
__device__ __forceinline__ void block_sum2(float& a, float& b) {
  __shared__ float red[2][kRowThreads / 32];
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { red[0][w] = a; red[1][w] = b; }
  __syncthreads();
  a = l < kRowThreads / 32 ? red[0][l] : 0.f;
  b = l < kRowThreads / 32 ? red[1][l] : 0.f;
#pragma unroll
  for (int o = 4; o >= 1; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
  a = __shfl_sync(0xffffffffu, a, 0);
  b = __shfl_sync(0xffffffffu, b, 0);
  __syncthreads();
}

// out = (LN(x) [* w + b]) [* (1 + scale) + shift]; scale / shift are fp32 per (batch, channel)
__global__ void __launch_bounds__(kRowThreads)
vb_ln_modulate_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b,
                      const float* __restrict__ scale, const float* __restrict__ shift, __nv_bfloat16* __restrict__ out,
                      int dim, int rows_per_batch, float eps) {
  const int64_t row = blockIdx.x;
  const int nvec = dim >> 3;
  const uint4* xr = reinterpret_cast<const uint4*>(x + row * dim);
  float v[kMaxVec][8];
  float s1 = 0.f, s2 = 0.f, dummy = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxVec; ++i) {
    const int idx = threadIdx.x + i * kRowThreads;
    if (idx < nvec) {
      unpack8(xr[idx], v[i]);
#pragma unroll
      for (int e = 0; e < 8; ++e) s1 += v[i][e];
    }
  }
  block_sum2(s1, dummy);
  const float mean = s1 / dim;
  // variance in a second pass over the registers: sum(x^2)/n - mean^2 cancels catastrophically when |mean| >> std
#pragma unroll
  for (int i = 0; i < kMaxVec; ++i) {
    const int idx = threadIdx.x + i * kRowThreads;
    if (idx < nvec) {
#pragma unroll
      for (int e = 0; e < 8; ++e) { const float d = v[i][e] - mean; s2 = fmaf(d, d, s2); }
    }
  }
  block_sum2(s2, dummy);
  const float rstd = rsqrtf(s2 / dim + eps);
  const int64_t batch = row / rows_per_batch;
  const float* sc = scale ? scale + batch * dim : nullptr;
  const float* sh = shift ? shift + batch * dim : nullptr;
  uint4* orow = reinterpret_cast<uint4*>(out + row * dim);
#pragma unroll
  for (int i = 0; i < kMaxVec; ++i) {
    const int idx = threadIdx.x + i * kRowThreads;
    if (idx < nvec) {
      float y[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int c = idx * 8 + e;
        float t = (v[i][e] - mean) * rstd;
        if (w) t = t * w[c] + (b ? b[c] : 0.f);
        else if (b) t += b[c];
        if (sc) t = t * (1.f + sc[c]) + sh[c];
        y[e] = t;
      }
      orow[idx] = pack8(y);
    }
  }
}

// ---- warp-per-row variants: NV = dim / 256 vectors per row; rows wider than 1536 / 3072 channels are shared by 2 / 4
// warps so that a thread never holds more than 6 vectors (~80 registers, no spills).  Vector idx = i * 32 * WPR + tid.
constexpr int kRowCtaThreads = 256;
__host__ __device__ constexpr int row_warps(int nv) { return nv > 12 ? 4 : nv > 6 ? 2 : 1; }   // <= 6 vectors per thread

__device__ __forceinline__ float warp_sum(float a) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  return a;
}
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// sum over the WPR warps that share a row; `slot` selects one of two exchange buffers so that back-to-back
// reductions need no extra barrier
template <int WPR>
__device__ __forceinline__ float row_sum(float a, float (*xchg)[kRowCtaThreads / 32], int slot) {
  a = warp_sum(a);
  if (WPR == 1) return a;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) xchg[slot][warp] = a;
  asm volatile("bar.sync %0, %1;" ::"r"(1 + warp / WPR), "r"(32 * WPR) : "memory");
  float r = 0.f;
#pragma unroll
  for (int i = 0; i < WPR; ++i) r += xchg[slot][(warp / WPR) * WPR + i];
  return r;
}

template <int NV>
__global__ void __launch_bounds__(kRowCtaThreads)
vb_ln_modulate_warp_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w,
                           const float* __restrict__ b, const float* __restrict__ scale,
                           const float* __restrict__ shift, __nv_bfloat16* __restrict__ out, int64_t rows,
                           int rows_per_batch, float eps) {
  constexpr int dim = NV * 256;
  constexpr int WPR = row_warps(NV);
  constexpr int NVT = NV / WPR;
  constexpr int kRowsPerCta = kRowCtaThreads / (32 * WPR);
  __shared__ float xchg[2][kRowCtaThreads / 32];
  const int tid = threadIdx.x & (32 * WPR - 1);                    // thread inside the row's warp group
  // rows beyond the end are clamped (recomputed by the last group) so that every thread reaches the named barriers
  const int64_t row_raw = static_cast<int64_t>(blockIdx.x) * kRowsPerCta + threadIdx.x / (32 * WPR);
  const bool live = row_raw < rows;
  const int64_t row = live ? row_raw : rows - 1;
  const uint4* xr = reinterpret_cast<const uint4*>(x + row * dim);
  uint4 raw[NVT];
#pragma unroll
  for (int i = 0; i < NVT; ++i) raw[i] = xr[i * 32 * WPR + tid];
  float s1 = 0.f;
#pragma unroll
  for (int i = 0; i < NVT; ++i) {
    float f[8];
    unpack8(raw[i], f);
#pragma unroll
    for (int e = 0; e < 8; ++e) s1 += f[e];
  }
  const float mean = row_sum<WPR>(s1, xchg, 0) * (1.f / dim);
  float s2 = 0.f;
#pragma unroll
  for (int i = 0; i < NVT; ++i) {
    float f[8];
    unpack8(raw[i], f);
#pragma unroll
    for (int e = 0; e < 8; ++e) { const float d = f[e] - mean; s2 = fmaf(d, d, s2); }
  }
  const float rstd = rsqrtf(row_sum<WPR>(s2, xchg, 1) * (1.f / dim) + eps);
  if (!live) return;
  const int64_t batch = row / rows_per_batch;
  const float* sc = scale ? scale + batch * dim : nullptr;
  const float* sh = shift ? shift + batch * dim : nullptr;
  uint4* orow = reinterpret_cast<uint4*>(out + row * dim);
#pragma unroll
  for (int i = 0; i < NVT; ++i) {
    const int c0 = (i * 32 * WPR + tid) * 8;
    float f[8];
    unpack8(raw[i], f);
#pragma unroll
    for (int e = 0; e < 8; ++e) f[e] = (f[e] - mean) * rstd;
    if (w) {
      const float4 w0 = ldg4(w + c0), w1 = ldg4(w + c0 + 4);
      const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
      float bv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (b) {
        const float4 b0 = ldg4(b + c0), b1 = ldg4(b + c0 + 4);
        bv[0] = b0.x; bv[1] = b0.y; bv[2] = b0.z; bv[3] = b0.w; bv[4] = b1.x; bv[5] = b1.y; bv[6] = b1.z; bv[7] = b1.w;
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) f[e] = f[e] * wv[e] + bv[e];
    } else if (b) {
      const float4 b0 = ldg4(b + c0), b1 = ldg4(b + c0 + 4);
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int e = 0; e < 8; ++e) f[e] += bv[e];
    }
    if (sc) {
      const float4 a0 = ldg4(sc + c0), a1 = ldg4(sc + c0 + 4), h0 = ldg4(sh + c0), h1 = ldg4(sh + c0 + 4);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float hv[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
#pragma unroll
      for (int e = 0; e < 8; ++e) f[e] = f[e] * (1.f + av[e]) + hv[e];
    }
    orow[i * 32 * WPR + tid] = pack8(f);
  }
}

template <int NV>
__global__ void __launch_bounds__(kRowCtaThreads)
vb_rmsnorm_rope_warp_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ weight,
                            const float* __restrict__ cs, const float* __restrict__ sn,
                            __nv_bfloat16* __restrict__ out, int64_t rows, int tokens_per_batch, float eps) {
  constexpr int dim = NV * 256;
  constexpr int WPR = row_warps(NV);
  constexpr int NVT = NV / WPR;
  constexpr int kRowsPerCta = kRowCtaThreads / (32 * WPR);
  __shared__ float xchg[2][kRowCtaThreads / 32];
  const int tid = threadIdx.x & (32 * WPR - 1);
  const int64_t row_raw = static_cast<int64_t>(blockIdx.x) * kRowsPerCta + threadIdx.x / (32 * WPR);
  const bool live = row_raw < rows;
  const int64_t row = live ? row_raw : rows - 1;
  const uint4* xr = reinterpret_cast<const uint4*>(x + row * dim);
  const uint4* wr = reinterpret_cast<const uint4*>(weight);
  uint4 raw[NVT];
#pragma unroll
  for (int i = 0; i < NVT; ++i) raw[i] = xr[i * 32 * WPR + tid];
  // 8 channels = 4 pairs; a thread's pairs inside the 128-wide head are the same for every i (16 threads = one head)
  float4 c4 = make_float4(1.f, 1.f, 1.f, 1.f), s4 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (cs) {
    const int64_t tok = row % tokens_per_batch;
    const int pair0 = (tid & 15) * 4;
    c4 = ldg4(cs + tok * (kHeadDim / 2) + pair0);
    s4 = ldg4(sn + tok * (kHeadDim / 2) + pair0);
  }
  float s2 = 0.f;
#pragma unroll
  for (int i = 0; i < NVT; ++i) {
    float f[8];
    unpack8(raw[i], f);
#pragma unroll
    for (int e = 0; e < 8; ++e) s2 = fmaf(f[e], f[e], s2);
  }
  const float rinv = rsqrtf(row_sum<WPR>(s2, xchg, 0) * (1.f / dim) + eps);
  if (!live) return;
  uint4* orow = reinterpret_cast<uint4*>(out + row * dim);
  const float cv[4] = {c4.x, c4.y, c4.z, c4.w}, sv[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
  for (int i = 0; i < NVT; ++i) {
    float f[8], wv[8], y[8];
    unpack8(raw[i], f);
    unpack8(__ldg(wr + i * 32 * WPR + tid), wv);
#pragma unroll
    for (int e = 0; e < 8; ++e) y[e] = f[e] * rinv * wv[e];
    if (cs) {
#pragma unroll
      for (int pz = 0; pz < 4; ++pz) {
        const float re = y[2 * pz], im = y[2 * pz + 1];
        y[2 * pz] = re * cv[pz] - im * sv[pz];
        y[2 * pz + 1] = re * sv[pz] + im * cv[pz];
      }
    }
    orow[i * 32 * WPR + tid] = pack8(y);
  }
}

// out = x + y * gate (gate fp32 per (batch, channel); nullptr = plain residual add)
__global__ void __launch_bounds__(256)
vb_gate_residual_kernel(const uint4* __restrict__ x, const uint4* __restrict__ y, const float* __restrict__ gate,
                        uint4* __restrict__ out, int64_t n_vec, int dim, int64_t vec_per_batch) {
  const int dvec = dim >> 3;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_vec;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float a[8], c[8];
    unpack8(x[i], a);
    unpack8(y[i], c);
    if (gate) {
      const float* g = gate + (i / vec_per_batch) * dim + (i % dvec) * 8;
#pragma unroll
      for (int e = 0; e < 8; ++e) a[e] = fmaf(c[e], g[e], a[e]);
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) a[e] += c[e];
    }
    out[i] = pack8(a);
  }
}

// RMSNorm over the whole row (all heads) * weight, then RoPE on channel pairs of every 128-wide head.
// cos / sin: fp32 (tokens, 64) for the rank's token shard; token = row % tokens_per_batch
__global__ void __launch_bounds__(kRowThreads)
vb_rmsnorm_rope_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ weight,
                       const float* __restrict__ cs, const float* __restrict__ sn, __nv_bfloat16* __restrict__ out,
                       int dim, int tokens_per_batch, float eps) {
  const int64_t row = blockIdx.x;
  const int nvec = dim >> 3;
  const uint4* xr = reinterpret_cast<const uint4*>(x + row * dim);
  const uint4* wr = reinterpret_cast<const uint4*>(weight);
  float v[kMaxVec][8];
  float s2 = 0.f, dummy = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxVec; ++i) {
    const int idx = threadIdx.x + i * kRowThreads;
    if (idx < nvec) {
      unpack8(xr[idx], v[i]);
#pragma unroll
      for (int e = 0; e < 8; ++e) s2 += v[i][e] * v[i][e];
    }
  }
  block_sum2(s2, dummy);
  const float rinv = rsqrtf(s2 / dim + eps);
  const int64_t tok = row % tokens_per_batch;
  const float* c_row = cs ? cs + tok * (kHeadDim / 2) : nullptr;
  const float* s_row = sn ? sn + tok * (kHeadDim / 2) : nullptr;
  uint4* orow = reinterpret_cast<uint4*>(out + row * dim);
#pragma unroll
  for (int i = 0; i < kMaxVec; ++i) {
    const int idx = threadIdx.x + i * kRowThreads;
    if (idx < nvec) {
      float wv[8], y[8];
      unpack8(wr[idx], wv);
#pragma unroll
      for (int e = 0; e < 8; ++e) y[e] = v[i][e] * rinv * wv[e];
      if (c_row) {
        const int pair0 = ((idx * 8) & (kHeadDim - 1)) >> 1;     // first channel pair of this vector inside its head
#pragma unroll
        for (int pz = 0; pz < 4; ++pz) {
          const float c = c_row[pair0 + pz], s = s_row[pair0 + pz];
          const float re = y[2 * pz], im = y[2 * pz + 1];
          y[2 * pz] = re * c - im * s;
          y[2 * pz + 1] = re * s + im * c;
        }
      }
      orow[idx] = pack8(y);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// HunyuanVideo Q / K prologue (reference: vorta/attention/hunyuan.py:62-134): per-HEAD RMSNorm (norm_q / norm_k /
// norm_added_q / norm_added_k are RMSNorm(128)) + real-valued RoPE on the video tokens only + placement of the row in
// the joint [video | text] sequence, in ONE pass.  The reference runs this as a normalisation over a transposed
// view, an unbind / stack / float-multiply RoPE and three torch.cat over the whole joint tensor (~10 HBM passes).
//   unit = (row, head): a half-warp, 16 lanes x 16 bytes; 4 units in flight per half-warp
//   src row r of batch b  ->  dst row dst_row0 + r of batch b  (dst has dst_rows rows per batch; in place allowed)
//   rows r < rope_rows rotate channel pairs (2i, 2i+1) by (cos, sin)[r][i] (fp32 tables of 64 entries per token)
// ------------------------------------------------------------------------------------------------
struct HeadNormParams {
  const __nv_bfloat16* x;
  const __nv_bfloat16* weight;     // (128) or nullptr = no normalisation
  const float* cs;                 // (rope_rows, 64) or nullptr
  const float* sn;
  __nv_bfloat16* out;
  int64_t units;                   // batch * rows * heads
  int rows, heads, rope_rows, dst_rows, dst_row0;
  float eps;
};

__global__ void __launch_bounds__(256) vb_headnorm_rope_kernel(const HeadNormParams p) {
  constexpr int kInFlight = 4;
  const int lane16 = threadIdx.x & 15;
  const int64_t hw = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 4;
  const int64_t n_hw = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 4;
  float wv[8];
  if (p.weight) unpack8(__ldg(reinterpret_cast<const uint4*>(p.weight) + lane16), wv);
  // the loop bound is the same for both half-warps of a warp (the shuffles below are full-warp)
  const int64_t n_steps = (p.units + n_hw * kInFlight - 1) / (n_hw * kInFlight);
  for (int64_t step = 0; step < n_steps; ++step) {
    const int64_t u0 = (step * n_hw + hw) * kInFlight;
    uint4 raw[kInFlight];
#pragma unroll
    for (int i = 0; i < kInFlight; ++i) {
      const int64_t u = u0 + i;
      raw[i] = u < p.units ? (reinterpret_cast<const uint4*>(p.x) + u * 16)[lane16] : make_uint4(0, 0, 0, 0);   // plain load: x may alias out
    }
#pragma unroll
    for (int i = 0; i < kInFlight; ++i) {
      const int64_t u = u0 + i;
      float f[8];
      unpack8(raw[i], f);
      float s2 = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) s2 = fmaf(f[e], f[e], s2);
#pragma unroll
      for (int o = 8; o >= 1; o >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
      if (u >= p.units) continue;
      const int head = static_cast<int>(u % p.heads);
      const int64_t rb = u / p.heads;
      const int r = static_cast<int>(rb % p.rows);
      const int64_t b = rb / p.rows;
      if (p.weight) {
        const float rinv = rsqrtf(s2 * (1.f / kHeadDim) + p.eps);
#pragma unroll
        for (int e = 0; e < 8; ++e) f[e] = f[e] * rinv * wv[e];
      }
      if (p.cs != nullptr && r < p.rope_rows) {
        const float4 c4 = ldg4(p.cs + static_cast<int64_t>(r) * (kHeadDim / 2) + lane16 * 4);
        const float4 s4 = ldg4(p.sn + static_cast<int64_t>(r) * (kHeadDim / 2) + lane16 * 4);
        const float cv[4] = {c4.x, c4.y, c4.z, c4.w}, sv[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
        for (int pz = 0; pz < 4; ++pz) {
          const float re = f[2 * pz], im = f[2 * pz + 1];
          f[2 * pz] = re * cv[pz] - im * sv[pz];
          f[2 * pz + 1] = re * sv[pz] + im * cv[pz];
        }
      }
      const int64_t drow = b * p.dst_rows + p.dst_row0 + r;
      reinterpret_cast<uint4*>(p.out)[(drow * p.heads + head) * 16 + lane16] = pack8(f);
    }
  }
}

// the kernels read and write x / y / out (and the bf16 weights, and headnorm's tables) with 16-byte vectors
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int launch_headnorm_rope(const void* x, const void* weight, const float* cs, const float* sn, void* out, int batch,
                         int rows, int heads, int rope_rows, int dst_rows, int dst_row0, float eps,
                         cudaStream_t stream) {
  VB_REQUIRE(batch >= 0 && rows >= 0 && heads > 0 && dst_row0 >= 0 && dst_row0 + rows <= dst_rows, VB_ERR_INVALID,
             "headnorm_rope: rows [%d, %d) do not fit a destination of %d rows", dst_row0, dst_row0 + rows, dst_rows);
  VB_REQUIRE((cs == nullptr) == (sn == nullptr) && rope_rows <= rows, VB_ERR_INVALID,
             "headnorm_rope: cos / sin tables come together and cover at most the source rows");
  VB_REQUIRE(aligned16(x) && aligned16(out) && aligned16(weight) && aligned16(cs) && aligned16(sn), VB_ERR_INVALID,
             "headnorm_rope: x, out, weight and the cos / sin tables must be 16-byte aligned");
  HeadNormParams p;
  p.x = static_cast<const __nv_bfloat16*>(x);
  p.weight = static_cast<const __nv_bfloat16*>(weight);
  p.cs = cs; p.sn = sn;
  p.out = static_cast<__nv_bfloat16*>(out);
  p.units = static_cast<int64_t>(batch) * rows * heads;
  p.rows = rows; p.heads = heads; p.rope_rows = cs ? rope_rows : 0; p.dst_rows = dst_rows; p.dst_row0 = dst_row0;
  p.eps = eps;
  if (p.units == 0) return VB_OK;
  const int64_t blocks_needed = (p.units / 4 * 16 + 255) / 256 + 1;
  const int grid = static_cast<int>(blocks_needed < 148 * 8 ? blocks_needed : 148 * 8);
  vb_headnorm_rope_kernel<<<grid, 256, 0, stream>>>(p);
  VB_CUDA_OK(cudaGetLastError());
  return VB_OK;
}

static unsigned row_grid(int64_t rows, int nv) {
  const int rows_per_cta = kRowCtaThreads / (32 * row_warps(nv));
  return static_cast<unsigned>((rows + rows_per_cta - 1) / rows_per_cta);
}

int launch_ln_modulate(const void* x, const float* w, const float* b, const float* scale, const float* shift, void* out,
                       int64_t rows, int dim, int rows_per_batch, float eps, cudaStream_t stream) {
  VB_REQUIRE(dim % 8 == 0 && dim <= kRowThreads * kMaxVec * 8, VB_ERR_UNSUPPORTED, "row width %d not supported", dim);
  VB_REQUIRE(aligned16(x) && aligned16(out), VB_ERR_INVALID, "ln_modulate: x and out must be 16-byte aligned");
  if (rows == 0) return VB_OK;
  const __nv_bfloat16* xb = static_cast<const __nv_bfloat16*>(x);
  __nv_bfloat16* ob = static_cast<__nv_bfloat16*>(out);
  // the CTA-per-row kernel reads the fp32 parameters with scalar loads, so misaligned parameters take it
  const bool aligned = ((reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(scale) |
                         reinterpret_cast<uintptr_t>(shift)) & 15) == 0;
#define VB_LN_CASE(NV)                                                                                              \
  case NV * 256:                                                                                                    \
    vb_ln_modulate_warp_kernel<NV><<<row_grid(rows, NV), kRowCtaThreads, 0, stream>>>(xb, w, b, scale, shift, ob,  \
                                                                                       rows, rows_per_batch, eps); \
    break;
  switch (aligned ? dim : 0) {
    VB_LN_CASE(4) VB_LN_CASE(6) VB_LN_CASE(8) VB_LN_CASE(12) VB_LN_CASE(16) VB_LN_CASE(20) VB_LN_CASE(24)
    default:
      vb_ln_modulate_kernel<<<static_cast<unsigned>(rows), kRowThreads, 0, stream>>>(xb, w, b, scale, shift, ob, dim,
                                                                                      rows_per_batch, eps);
  }
#undef VB_LN_CASE
  VB_CUDA_OK(cudaGetLastError());
  return VB_OK;
}
int launch_gate_residual(const void* x, const void* y, const float* gate, void* out, int64_t rows, int dim,
                         int rows_per_batch, cudaStream_t stream) {
  VB_REQUIRE(dim % 8 == 0, VB_ERR_UNSUPPORTED, "row width %d not supported", dim);
  VB_REQUIRE(aligned16(x) && aligned16(y) && aligned16(out), VB_ERR_INVALID,
             "gate_residual: x, y and out must be 16-byte aligned");
  const int64_t n_vec = rows * (dim >> 3);
  if (n_vec == 0) return VB_OK;
  const int64_t blocks = (n_vec + 255) / 256;
  const int grid = static_cast<int>(blocks < 148 * 32 ? blocks : 148 * 32);
  vb_gate_residual_kernel<<<grid, 256, 0, stream>>>(static_cast<const uint4*>(x), static_cast<const uint4*>(y), gate,
                                                    static_cast<uint4*>(out), n_vec, dim,
                                                    static_cast<int64_t>(rows_per_batch) * (dim >> 3));
  VB_CUDA_OK(cudaGetLastError());
  return VB_OK;
}
int launch_rmsnorm_rope(const void* x, const void* weight, const float* cs, const float* sn, void* out, int64_t rows,
                        int dim, int tokens_per_batch, float eps, cudaStream_t stream) {
  VB_REQUIRE(dim % kHeadDim == 0 && dim <= kRowThreads * kMaxVec * 8, VB_ERR_UNSUPPORTED,
             "row width %d not supported", dim);
  VB_REQUIRE(aligned16(x) && aligned16(out) && aligned16(weight), VB_ERR_INVALID,
             "rmsnorm_rope: x, out and weight must be 16-byte aligned");
  if (rows == 0) return VB_OK;
  const __nv_bfloat16* xb = static_cast<const __nv_bfloat16*>(x);
  const __nv_bfloat16* wb = static_cast<const __nv_bfloat16*>(weight);
  __nv_bfloat16* ob = static_cast<__nv_bfloat16*>(out);
  // the CTA-per-row kernel reads the tables with scalar loads, so misaligned tables take it
  const bool aligned = aligned16(cs) && aligned16(sn);
#define VB_RMS_CASE(NV)                                                                                             \
  case NV * 256:                                                                                                    \
    vb_rmsnorm_rope_warp_kernel<NV><<<row_grid(rows, NV), kRowCtaThreads, 0, stream>>>(xb, wb, cs, sn, ob, rows,   \
                                                                                        tokens_per_batch, eps);    \
    break;
  switch (aligned ? dim : 0) {
    VB_RMS_CASE(4) VB_RMS_CASE(6) VB_RMS_CASE(8) VB_RMS_CASE(12) VB_RMS_CASE(16) VB_RMS_CASE(20) VB_RMS_CASE(24)
    default:
      vb_rmsnorm_rope_kernel<<<static_cast<unsigned>(rows), kRowThreads, 0, stream>>>(xb, wb, cs, sn, ob, dim,
                                                                                       tokens_per_batch, eps);
  }
#undef VB_RMS_CASE
  VB_CUDA_OK(cudaGetLastError());
  return VB_OK;
}

}  // namespace vb
