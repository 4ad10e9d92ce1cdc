// layernorm.cu -- LayerNorm fused with the residual add around it, forward and backward, at HBM speed.
//
// The blocks of the path interleave every attention / Mlp call with a LayerNorm and a residual add
// (swin_v2_module.py:299-302 post-norm, swinfusion_module.py:345,377-378,491-492,535-539 pre-norm,
// crossmodal_transformer.py:143-165).  PyTorch runs them as separate kernels on an fp32 residual stream (autocast), plus the
// bf16 casts feeding the next GEMM; at the Swin widths (C = 96 ... 1536, ~1e5 rows) ATen's layer_norm kernels are far
// from the memory roofline (one block per 96-element row).  Here one kernel does, per row:
//
//   mode PRE  (pre-norm blocks):   s = resid + delta;   out_sum = s;   out_norm = LN(s) * gamma + beta
//   mode POST (SwinV2 res-post-norm):   s = resid + LN(delta) * gamma + beta;   out_sum = s;   out_norm = s (cast)
//
// either input may be absent (PRE with delta == null is a plain LayerNorm), either output may be skipped, and every
// tensor is fp32 or bf16 independently (residual stream fp32, activations bf16 under autocast).  mean / rstd per row are
// kept for the backward, which returns d resid, d delta and (accumulated with atomics over row blocks) d gamma, d beta.
// Deterministic mode hands the backward kernels a `part` buffer: block b writes its column sums to part[0 / 1][b][c] (d gamma
// / d beta) instead, and reduce_partials adds them into the caller's buffers in block order.
//
// One warp per row; lane l owns the column pairs 2 (l + 32 k): 4-byte (bf16x2) or 8-byte (float2) accesses, fully
// coalesced, values stay in registers between the statistics pass and the normalisation pass.  fp32 arithmetic.
#include <unordered_map>
#include <mutex>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mmn_b200.h"
#include "generic_launch.h"

namespace mmn {

namespace {

struct LnTensor {            // (rows, cols) matrix, contiguous rows
  const void* p;
  int dt;                    // MMN_DT_F32 / MMN_DT_BF16
};
struct LnOut {
  void* p;
  int dt;
};

__device__ __forceinline__ float2 ld2(const LnTensor& t, long long idx) {       // idx: element index of an even column
  if (t.dt == MMN_DT_F32) return __ldg(reinterpret_cast<const float2*>(static_cast<const float*>(t.p) + idx));
  const uint32_t u = __ldg(reinterpret_cast<const uint32_t*>(static_cast<const __nv_bfloat16*>(t.p) + idx));
  return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u));
}
__device__ __forceinline__ void st2(const LnOut& t, long long idx, float2 v) {
  if (t.dt == MMN_DT_F32) {
    *reinterpret_cast<float2*>(static_cast<float*>(t.p) + idx) = v;
  } else {
    __nv_bfloat162 b = __floats2bfloat162_rn(v.x, v.y);
    *reinterpret_cast<__nv_bfloat162*>(static_cast<__nv_bfloat16*>(t.p) + idx) = b;
  }
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

constexpr int kLnWarps = 8;

// K = column pairs per lane = ceil(cols / 64)
template <int K>
__global__ void __launch_bounds__(kLnWarps * 32)
ln_fwd_kernel(LnTensor resid, LnTensor delta, const float* __restrict__ gamma, const float* __restrict__ beta, float eps, int mode,
              LnOut out_sum, LnOut out_norm, float* __restrict__ mean, float* __restrict__ rstd, long long rows, int cols) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float2 g[K], b[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const int c = 2 * (lane + 32 * k);
    g[k] = c < cols ? __ldg(reinterpret_cast<const float2*>(gamma + c)) : make_float2(0.f, 0.f);
    b[k] = c < cols && beta ? __ldg(reinterpret_cast<const float2*>(beta + c)) : make_float2(0.f, 0.f);
  }
  const float inv_n = 1.f / (float)cols;
  for (long long row = (long long)blockIdx.x * kLnWarps + warp; row < rows; row += (long long)gridDim.x * kLnWarps) {
    const long long base = row * cols;
    float2 x[K], r[K];          // x: the normalised quantity (PRE: resid + delta; POST: delta); r: the residual (POST)
    float s1 = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int c = 2 * (lane + 32 * k);
      x[k] = make_float2(0.f, 0.f);
      r[k] = make_float2(0.f, 0.f);
      if (c < cols) {
        if (mode == 0) {
          if (resid.p) x[k] = ld2(resid, base + c);
          if (delta.p) { const float2 d = ld2(delta, base + c); x[k].x += d.x; x[k].y += d.y; }
        } else {
          x[k] = ld2(delta, base + c);
          if (resid.p) r[k] = ld2(resid, base + c);
        }
        s1 += x[k].x + x[k].y;
      }
    }
    const float mu = warp_sum(s1) * inv_n;
    float s2 = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int c = 2 * (lane + 32 * k);
      if (c < cols) { const float a = x[k].x - mu, d = x[k].y - mu; s2 += a * a + d * d; }
    }
    const float rs = rsqrtf(warp_sum(s2) * inv_n + eps);
    if (lane == 0) { mean[row] = mu; rstd[row] = rs; }
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int c = 2 * (lane + 32 * k);
      if (c < cols) {
        const float2 n = make_float2((x[k].x - mu) * rs * g[k].x + b[k].x, (x[k].y - mu) * rs * g[k].y + b[k].y);
        if (mode == 0) {
          if (out_sum.p) st2(out_sum, base + c, x[k]);
          if (out_norm.p) st2(out_norm, base + c, n);
        } else {
          const float2 s = make_float2(r[k].x + n.x, r[k].y + n.y);
          if (out_sum.p) st2(out_sum, base + c, s);
          if (out_norm.p) st2(out_norm, base + c, s);
        }
      }
    }
  }
}

// Backward.  gs: gradient w.r.t. out_sum (optional), gn: gradient w.r.t. out_norm (optional), x: the normalised quantity
// (PRE: out_sum; POST: delta).
//   PRE :  g_x = gs + LN'(gn)      d resid = d delta = g_x          d gamma += sum_rows gn * xhat,  d beta += sum_rows gn
//   POST:  g   = gs + gn           d resid = g,  d delta = LN'(g)   d gamma += sum_rows g * xhat,   d beta += sum_rows g
// LN'(u)_c = rstd * (u_c gamma_c - mean_c(u gamma) - xhat_c mean_c(u gamma xhat)).
template <int K>
__global__ void __launch_bounds__(kLnWarps * 32)
ln_bwd_kernel(LnTensor gs, LnTensor gn, LnTensor x, const float* __restrict__ gamma, const float* __restrict__ mean,
              const float* __restrict__ rstd, int mode, LnOut d_resid, LnOut d_delta, float* __restrict__ dgamma,
              float* __restrict__ dbeta, float* __restrict__ part, long long rows, int cols) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float2 g[K], ag[K], ab[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const int c = 2 * (lane + 32 * k);
    g[k] = c < cols ? __ldg(reinterpret_cast<const float2*>(gamma + c)) : make_float2(0.f, 0.f);
    ag[k] = make_float2(0.f, 0.f);
    ab[k] = make_float2(0.f, 0.f);
  }
  const float inv_n = 1.f / (float)cols;
  for (long long row = (long long)blockIdx.x * kLnWarps + warp; row < rows; row += (long long)gridDim.x * kLnWarps) {
    const long long base = row * cols;
    const float mu = __ldg(mean + row), rs = __ldg(rstd + row);
    float2 u[K], xh[K], pass[K];     // u: gradient entering the LayerNorm; pass: gradient bypassing it
    float m1 = 0.f, m2 = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int c = 2 * (lane + 32 * k);
      u[k] = xh[k] = pass[k] = make_float2(0.f, 0.f);
      if (c < cols) {
        const float2 xv = ld2(x, base + c);
        xh[k] = make_float2((xv.x - mu) * rs, (xv.y - mu) * rs);
        float2 a = gs.p ? ld2(gs, base + c) : make_float2(0.f, 0.f);
        float2 n = gn.p ? ld2(gn, base + c) : make_float2(0.f, 0.f);
        if (mode == 0) { u[k] = n; pass[k] = a; }
        else { u[k] = make_float2(a.x + n.x, a.y + n.y); pass[k] = u[k]; }
        ag[k].x += u[k].x * xh[k].x; ag[k].y += u[k].y * xh[k].y;
        ab[k].x += u[k].x; ab[k].y += u[k].y;
        const float ux = u[k].x * g[k].x, uy = u[k].y * g[k].y;
        m1 += ux + uy;
        m2 += ux * xh[k].x + uy * xh[k].y;
      }
    }
    m1 = warp_sum(m1) * inv_n;
    m2 = warp_sum(m2) * inv_n;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int c = 2 * (lane + 32 * k);
      if (c < cols) {
        const float2 ln = make_float2(rs * (u[k].x * g[k].x - m1 - xh[k].x * m2), rs * (u[k].y * g[k].y - m1 - xh[k].y * m2));
        if (mode == 0) {
          const float2 t = make_float2(pass[k].x + ln.x, pass[k].y + ln.y);
          if (d_resid.p) st2(d_resid, base + c, t);
          if (d_delta.p) st2(d_delta, base + c, t);
        } else {
          if (d_resid.p) st2(d_resid, base + c, pass[k]);
          if (d_delta.p) st2(d_delta, base + c, ln);
        }
      }
    }
  }
  // column sums over this block's rows: warps -> shared memory -> one atomic per column and block (64 columns per round)
  __shared__ float red[kLnWarps][64];
  for (int pass_id = 0; pass_id < 2; ++pass_id) {
    float* dst = pass_id == 0 ? dgamma : dbeta;
    if (!dst) continue;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const float2 v = pass_id == 0 ? ag[k] : ab[k];
      red[warp][2 * lane] = v.x;
      red[warp][2 * lane + 1] = v.y;
      __syncthreads();
      const int c = 64 * k + threadIdx.x;
      if (threadIdx.x < 64 && c < cols) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kLnWarps; ++w) s += red[w][threadIdx.x];
        if (part) part[((size_t)pass_id * gridDim.x + blockIdx.x) * cols + c] = s;
        else atomicAdd(dst + c, s);
      }
      __syncthreads();
    }
  }
}

// ------------------------------------------------------------------------------------------
// Vectorised kernels (cols % 4 == 0, cols <= 768): LPR lanes share a row, each lane owns V chunks of four consecutive
// columns (16-byte fp32 / 8-byte bf16 accesses), a warp works on 32 / LPR rows at once.  At C = 96 that is 8 lanes x 3
// chunks per row, four rows per warp: ~25 warp instructions per row where the one-row-per-warp kernels above need ~280
// (they were issue-bound at a quarter of the HBM roofline; tools/bench_blocks.py).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 ld4(const LnTensor& t, long long idx) {
  if (t.dt == MMN_DT_F32) return __ldg(reinterpret_cast<const float4*>(static_cast<const float*>(t.p) + idx));
  const uint2 u = __ldg(reinterpret_cast<const uint2*>(static_cast<const __nv_bfloat16*>(t.p) + idx));
  return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16),
                     __uint_as_float(u.y & 0xffff0000u));
}
__device__ __forceinline__ void st4(const LnOut& t, long long idx, float4 v) {
  if (t.dt == MMN_DT_F32) {
    *reinterpret_cast<float4*>(static_cast<float*>(t.p) + idx) = v;
  } else {
    const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 u;
    u.x = *reinterpret_cast<const uint32_t*>(&a);
    u.y = *reinterpret_cast<const uint32_t*>(&b);
    *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(t.p) + idx) = u;
  }
}
template <int LPR>
__device__ __forceinline__ float row_sum(float v) {          // sum over the LPR lanes that share a row
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float4 f4zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }

// MODE (pre- / post-norm) is a template parameter: the pre-norm forward keeps no residual copy and fits 64 registers (four
// blocks per SM); the post-norm one took 80-85 (three blocks) until it was asked for four as well: 32.3 -> 30.7 us at 110 592 x 96.  U row groups per iteration with all their loads issued up front (U = 2 at two blocks per SM measured
// no better than U = 1 at three or four: tools/bench_blocks.py, r2o vs r2k), so the launches use U = 1.
template <int LPR, int V, int MODE, int U>
__global__ void __launch_bounds__(kLnWarps * 32, V <= 3 ? 4 : 0)      // 0 = no occupancy request (as before) for the wide rows
ln_fwd_v4_kernel(LnTensor resid, LnTensor delta, const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                 LnOut out_sum, LnOut out_norm, float* __restrict__ mean, float* __restrict__ rstd, long long rows, int cols) {
  constexpr int R = 32 / LPR;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lr = lane % LPR, sub = lane / LPR;
  const float inv_n = 1.f / (float)cols;
  const long long stride = (long long)gridDim.x * kLnWarps * R * U;
  for (long long row0 = ((long long)blockIdx.x * kLnWarps + warp) * R * U; row0 < rows; row0 += stride) {
    float4 x[U][V], r[MODE == 0 ? 1 : U][MODE == 0 ? 1 : V];
    float s1[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long row = row0 + u * R + sub;
      const bool live = row < rows;
      const long long base = row * cols;
      s1[u] = 0.f;
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const int c = 4 * (lr + LPR * v);
        x[u][v] = f4zero();
        if (MODE != 0) r[u][v] = f4zero();
        if (live && c < cols) {
          if (MODE == 0) {
            if (resid.p) x[u][v] = ld4(resid, base + c);
            if (delta.p) { const float4 d = ld4(delta, base + c); x[u][v].x += d.x; x[u][v].y += d.y; x[u][v].z += d.z; x[u][v].w += d.w; }
          } else {
            x[u][v] = ld4(delta, base + c);
            if (resid.p) r[u][v] = ld4(resid, base + c);
          }
          s1[u] += (x[u][v].x + x[u][v].y) + (x[u][v].z + x[u][v].w);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long row = row0 + u * R + sub;
      const bool live = row < rows;
      const long long base = row * cols;
      const float mu = row_sum<LPR>(s1[u]) * inv_n;
      float s2 = 0.f;
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const int c = 4 * (lr + LPR * v);
        if (c < cols) {
          const float a0 = x[u][v].x - mu, a1 = x[u][v].y - mu, a2 = x[u][v].z - mu, a3 = x[u][v].w - mu;
          s2 += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
        }
      }
      const float rs = rsqrtf(row_sum<LPR>(s2) * inv_n + eps);
      if (live && lr == 0) { mean[row] = mu; rstd[row] = rs; }
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const int c = 4 * (lr + LPR * v);
        if (live && c < cols) {
          // gamma / beta: 16-byte loads that hit L1 (keeping them in registers cost half the occupancy)
          const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
          const float4 b = beta ? __ldg(reinterpret_cast<const float4*>(beta + c)) : f4zero();
          const float4 xv = x[u][v];
          const float4 n = make_float4((xv.x - mu) * rs * g.x + b.x, (xv.y - mu) * rs * g.y + b.y,
                                       (xv.z - mu) * rs * g.z + b.z, (xv.w - mu) * rs * g.w + b.w);
          if (MODE == 0) {
            if (out_sum.p) st4(out_sum, base + c, xv);
            if (out_norm.p) st4(out_norm, base + c, n);
          } else {
            const float4 rv = r[u][v];
            const float4 s = make_float4(rv.x + n.x, rv.y + n.y, rv.z + n.z, rv.w + n.w);
            if (out_sum.p) st4(out_sum, base + c, s);
            if (out_norm.p) st4(out_norm, base + c, s);
          }
        }
      }
    }
  }
}

template <int LPR, int V, int MODE, int U>
__global__ void __launch_bounds__(kLnWarps * 32, V <= 3 ? 3 : 1)
ln_bwd_v4_kernel(LnTensor gs, LnTensor gn, LnTensor x, const float* __restrict__ gamma, const float* __restrict__ mean,
                 const float* __restrict__ rstd, LnOut d_resid, LnOut d_delta, float* __restrict__ dgamma,
                 float* __restrict__ dbeta, float* __restrict__ part, long long rows, int cols) {
  constexpr int R = 32 / LPR;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lr = lane % LPR, sub = lane / LPR;
  float4 ag[V], ab[V];
#pragma unroll
  for (int v = 0; v < V; ++v) { ag[v] = f4zero(); ab[v] = f4zero(); }
  const float inv_n = 1.f / (float)cols;
  const long long stride = (long long)gridDim.x * kLnWarps * R * U;
  for (long long row0 = ((long long)blockIdx.x * kLnWarps + warp) * R * U; row0 < rows; row0 += stride) {
    // raw loads of all U row groups first
    float4 xv[U][V], a[U][V], n[U][V];
    float mu[U], rs[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long row = row0 + u * R + sub;
      const bool live = row < rows;
      const long long base = row * cols;
      mu[u] = live ? __ldg(mean + row) : 0.f;
      rs[u] = live ? __ldg(rstd + row) : 0.f;
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const int c = 4 * (lr + LPR * v);
        xv[u][v] = a[u][v] = n[u][v] = f4zero();
        if (live && c < cols) {
          xv[u][v] = ld4(x, base + c);
          if (gs.p) a[u][v] = ld4(gs, base + c);
          if (gn.p) n[u][v] = ld4(gn, base + c);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long row = row0 + u * R + sub;
      const bool live = row < rows;
      const long long base = row * cols;
      // w = (gradient bypassing the LayerNorm) + rstd * u * gamma, u = gradient entering it: the row's output is
      // w - rstd * (m1 + xhat * m2), so only w and xhat live across the row reductions
      float4 w[V], xh[V];
      float m1 = 0.f, m2 = 0.f;
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const int c = 4 * (lr + LPR * v);
        w[v] = xh[v] = f4zero();
        if (live && c < cols) {
          const float4 t = xv[u][v];
          xh[v] = make_float4((t.x - mu[u]) * rs[u], (t.y - mu[u]) * rs[u], (t.z - mu[u]) * rs[u], (t.w - mu[u]) * rs[u]);
          const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
          float4 uu;
          if (MODE == 0) { uu = n[u][v]; w[v] = a[u][v]; }
          else {
            uu = make_float4(a[u][v].x + n[u][v].x, a[u][v].y + n[u][v].y, a[u][v].z + n[u][v].z, a[u][v].w + n[u][v].w);
            if (d_resid.p) st4(d_resid, base + c, uu);
          }
          ag[v].x += uu.x * xh[v].x; ag[v].y += uu.y * xh[v].y; ag[v].z += uu.z * xh[v].z; ag[v].w += uu.w * xh[v].w;
          ab[v].x += uu.x; ab[v].y += uu.y; ab[v].z += uu.z; ab[v].w += uu.w;
          const float u0 = uu.x * g.x, u1 = uu.y * g.y, u2 = uu.z * g.z, u3 = uu.w * g.w;
          m1 += (u0 + u1) + (u2 + u3);
          m2 += (u0 * xh[v].x + u1 * xh[v].y) + (u2 * xh[v].z + u3 * xh[v].w);
          w[v].x = fmaf(rs[u], u0, w[v].x); w[v].y = fmaf(rs[u], u1, w[v].y); w[v].z = fmaf(rs[u], u2, w[v].z); w[v].w = fmaf(rs[u], u3, w[v].w);
        }
      }
      m1 = row_sum<LPR>(m1) * inv_n * rs[u];
      m2 = row_sum<LPR>(m2) * inv_n * rs[u];
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const int c = 4 * (lr + LPR * v);
        if (live && c < cols) {
          const float4 t = make_float4(w[v].x - m1 - xh[v].x * m2, w[v].y - m1 - xh[v].y * m2, w[v].z - m1 - xh[v].z * m2,
                                       w[v].w - m1 - xh[v].w * m2);
          if (MODE == 0) {
            if (d_resid.p) st4(d_resid, base + c, t);
            if (d_delta.p) st4(d_delta, base + c, t);
          } else {
            if (d_delta.p) st4(d_delta, base + c, t);
          }
        }
      }
    }
  }
  // column sums: rows of a warp (shuffles) -> warps (shared memory) -> one atomic per column and block
  __shared__ float red[kLnWarps][4 * LPR * V];
  for (int pass_id = 0; pass_id < 2; ++pass_id) {
    float* dst = pass_id == 0 ? dgamma : dbeta;
    if (!dst) continue;                                      // uniform
#pragma unroll
    for (int v = 0; v < V; ++v) {
      float4 acc = pass_id == 0 ? ag[v] : ab[v];
#pragma unroll
      for (int o = LPR; o < 32; o <<= 1) {
        acc.x += __shfl_xor_sync(0xffffffffu, acc.x, o); acc.y += __shfl_xor_sync(0xffffffffu, acc.y, o);
        acc.z += __shfl_xor_sync(0xffffffffu, acc.z, o); acc.w += __shfl_xor_sync(0xffffffffu, acc.w, o);
      }
      if (sub == 0) *reinterpret_cast<float4*>(&red[warp][4 * (lr + LPR * v)]) = acc;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < cols; c += kLnWarps * 32) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < kLnWarps; ++w) s += red[w][c];
      if (part) part[((size_t)pass_id * gridDim.x + blockIdx.x) * cols + c] = s;
      else atomicAdd(dst + c, s);
    }
    __syncthreads();
  }
}

struct V4Cfg { int lpr, v; };
// lanes per row / chunks per lane for cols / 4 chunks; {0, 0} when the vectorised kernels do not apply
V4Cfg v4_cfg(int cols) {
  if (cols % 4 != 0 || cols > 768) return {0, 0};
  const int ch = cols / 4;
  const V4Cfg table[] = {{8, 1}, {8, 2}, {8, 3}, {16, 2}, {16, 3}, {32, 2}, {32, 3}, {32, 4}, {32, 6}};
  for (const V4Cfg& c : table) if (ch <= c.lpr * c.v) return c;
  return {0, 0};
}
bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Blocks of `kern` that fit on one SM at kLnWarps * 32 threads (registers decide: 64 -> 4, 80 -> 3).  The grid-stride kernels
// are launched as whole resident waves: 8 blocks per SM for a kernel of which 3 fit ran 2.67 waves -- the last one a third
// empty -- and cost the LayerNorm backward 9-12 % at cfg3's 110 592 rows (tools/bench_ln.py: 46.6 -> 42.5 us pre-norm,
// 44.3 -> 39.3 us post-norm; two waves are no better than one at any width); its per-block column-sum flush (192 atomics)
// also runs 2.7x less often.
int resident_blocks(const void* kern) {
  static std::mutex mu;
  static std::unordered_map<const void*, int> cache;
  std::lock_guard<std::mutex> g(mu);
  auto it = cache.find(kern);
  if (it != cache.end()) return it->second;
  int b = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, kern, kLnWarps * 32, 0) != cudaSuccess || b < 1) {
    cudaGetLastError();
    b = 2;
  }
  cache[kern] = b;
  return b;
}

// up to blocks_per_sm x 148 blocks (grid-stride loops inside)
int ln_grid_v4(long long rows, int lpr, int unroll, int blocks_per_sm) {
  const long long per_block = (long long)kLnWarps * (32 / lpr) * unroll;
  long long want = (rows + per_block - 1) / per_block;
  const long long cap = 148ll * blocks_per_sm;
  return (int)(want < cap ? want : cap);
}

int ln_grid(long long rows) {
  long long want = (rows + kLnWarps - 1) / kLnWarps;
  const long long cap = 148ll * 8;
  return (int)(want < cap ? want : cap);
}

// blocks the backward launched (both kernels are one-wave grid-stride launches); adds their partials in block order
cudaError_t ln_reduce(const float* part, int blocks, int cols, float* dgamma, float* dbeta, cudaStream_t st, int* launches) {
  cudaError_t e = cudaSuccess;
  if (dgamma) e = reduce_partials(part, blocks, cols, dgamma, st, launches);
  if (e == cudaSuccess && dbeta) e = reduce_partials(part + (size_t)blocks * cols, blocks, cols, dbeta, st, launches);
  return e;
}

}  // namespace

#define MMN_LN_DISPATCH(K_, call)                       \
  switch (K_) {                                         \
    case 1: { constexpr int K = 1; call; } break;       \
    case 2: { constexpr int K = 2; call; } break;       \
    case 3: { constexpr int K = 3; call; } break;       \
    case 4: { constexpr int K = 4; call; } break;       \
    case 6: { constexpr int K = 6; call; } break;       \
    case 8: { constexpr int K = 8; call; } break;       \
    case 12: { constexpr int K = 12; call; } break;     \
    case 16: { constexpr int K = 16; call; } break;     \
    case 24: { constexpr int K = 24; call; } break;     \
    default: return cudaErrorInvalidValue;              \
  }

static int ln_pairs(int cols) {
  const int k = (cols + 63) / 64;
  const int sizes[] = {1, 2, 3, 4, 6, 8, 12, 16, 24};
  for (int s : sizes) if (k <= s) return s;
  return 0;
}

bool layernorm_supported(int cols) { return cols >= 2 && cols % 2 == 0 && ln_pairs(cols) > 0; }

cudaError_t layernorm_fwd(const void* resid, int resid_dt, const void* delta, int delta_dt, const float* gamma, const float* beta,
                          float eps, int mode, void* out_sum, int sum_dt, void* out_norm, int norm_dt, float* mean, float* rstd,
                          long long rows, int cols, cudaStream_t st, int* launches) {
  const int kk = ln_pairs(cols);
  LnTensor r{resid, resid_dt}, d{delta, delta_dt};
  LnOut os{out_sum, sum_dt}, on{out_norm, norm_dt};
  const V4Cfg vc = v4_cfg(cols);
  if (vc.lpr && aligned16(resid) && aligned16(delta) && aligned16(out_sum) && aligned16(out_norm) && aligned16(gamma) && aligned16(beta)) {
#define MMN_LN_V4(L_, V_) if (vc.lpr == L_ && vc.v == V_) {                                                                       \
      constexpr int U0 = 1, U1 = 1;                                                                  \
      auto k0 = ln_fwd_v4_kernel<L_, V_, 0, U0>;                                                     \
      auto k1 = ln_fwd_v4_kernel<L_, V_, 1, U1>;                                                     \
      if (mode == 0) k0<<<ln_grid_v4(rows, L_, U0, resident_blocks((const void*)k0)), kLnWarps * 32, 0, st>>>(r, d, gamma, beta, eps, os, on, mean, rstd, rows, cols); \
      else k1<<<ln_grid_v4(rows, L_, U1, resident_blocks((const void*)k1)), kLnWarps * 32, 0, st>>>(r, d, gamma, beta, eps, os, on, mean, rstd, rows, cols);           \
    }
    MMN_LN_V4(8, 1) MMN_LN_V4(8, 2) MMN_LN_V4(8, 3) MMN_LN_V4(16, 2) MMN_LN_V4(16, 3) MMN_LN_V4(32, 2) MMN_LN_V4(32, 3) MMN_LN_V4(32, 4) MMN_LN_V4(32, 6)
#undef MMN_LN_V4
    cudaError_t e4 = cudaGetLastError();
    if (e4 == cudaSuccess) ++*launches;
    return e4;
  }
  MMN_LN_DISPATCH(kk, (ln_fwd_kernel<K><<<ln_grid(rows), kLnWarps * 32, 0, st>>>(r, d, gamma, beta, eps, mode, os, on, mean, rstd, rows, cols)));
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) ++*launches;
  return e;
}

cudaError_t layernorm_bwd(const void* g_sum, int gs_dt, const void* g_norm, int gn_dt, const void* x, int x_dt, const float* gamma,
                          const float* mean, const float* rstd, int mode, void* d_resid, int dr_dt, void* d_delta, int dd_dt,
                          float* dgamma, float* dbeta, float* part, long long rows, int cols, cudaStream_t st, int* launches) {
  const int kk = ln_pairs(cols);
  if (!dgamma && !dbeta) part = nullptr;
  int blocks = 0;
  LnTensor gs{g_sum, gs_dt}, gn{g_norm, gn_dt}, xx{x, x_dt};
  LnOut dr{d_resid, dr_dt}, dd{d_delta, dd_dt};
  const V4Cfg vc = v4_cfg(cols);
  if (vc.lpr && aligned16(g_sum) && aligned16(g_norm) && aligned16(x) && aligned16(d_resid) && aligned16(d_delta) && aligned16(gamma)) {
#define MMN_LN_V4(L_, V_) if (vc.lpr == L_ && vc.v == V_) {                                                                       \
      constexpr int U = 1;                                                                           \
      auto k0 = ln_bwd_v4_kernel<L_, V_, 0, U>;                                                      \
      auto k1 = ln_bwd_v4_kernel<L_, V_, 1, U>;                                                      \
      if (mode == 0) { blocks = ln_grid_v4(rows, L_, U, resident_blocks((const void*)k0)); k0<<<blocks, kLnWarps * 32, 0, st>>>(gs, gn, xx, gamma, mean, rstd, dr, dd, dgamma, dbeta, part, rows, cols); } \
      else { blocks = ln_grid_v4(rows, L_, U, resident_blocks((const void*)k1)); k1<<<blocks, kLnWarps * 32, 0, st>>>(gs, gn, xx, gamma, mean, rstd, dr, dd, dgamma, dbeta, part, rows, cols); }        \
    }
    MMN_LN_V4(8, 1) MMN_LN_V4(8, 2) MMN_LN_V4(8, 3) MMN_LN_V4(16, 2) MMN_LN_V4(16, 3) MMN_LN_V4(32, 2) MMN_LN_V4(32, 3) MMN_LN_V4(32, 4) MMN_LN_V4(32, 6)
#undef MMN_LN_V4
    cudaError_t e4 = cudaGetLastError();
    if (e4 != cudaSuccess) return e4;
    ++*launches;
    return part ? ln_reduce(part, blocks, cols, dgamma, dbeta, st, launches) : cudaSuccess;
  }
  blocks = ln_grid(rows);
  MMN_LN_DISPATCH(kk, (ln_bwd_kernel<K><<<blocks, kLnWarps * 32, 0, st>>>(gs, gn, xx, gamma, mean, rstd, mode, dr, dd, dgamma, dbeta, part, rows, cols)));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  ++*launches;
  return part ? ln_reduce(part, blocks, cols, dgamma, dbeta, st, launches) : cudaSuccess;
}

// Either kernel launches at most 148 x 8 blocks (a 256-thread block per 8 rows at least), two rows of partials per block.
size_t layernorm_bwd_workspace_floats(long long rows, int cols) {
  const long long want = (rows + kLnWarps - 1) / kLnWarps, blocks = want < 148ll * 8 ? want : 148ll * 8;
  return (size_t)(blocks > 0 ? blocks : 0) * 2 * cols;
}

}  // namespace mmn
