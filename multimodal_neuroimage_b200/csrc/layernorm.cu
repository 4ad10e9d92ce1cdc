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
// One kernel family for every width: LPR lanes share a row and each lane owns V chunks of W consecutive columns, so a warp
// works on 32 / LPR rows at once.  W = 4 (16-byte fp32 / 8-byte bf16 accesses) when cols % 4 == 0 and every operand is
// 16-byte aligned, else W = 2.  At C = 96 that is 8 lanes x 3 chunks per row, four rows per warp: ~25 warp instructions per
// row where one row per warp needs ~280 and is issue-bound at a quarter of the HBM roofline (tools/bench_blocks.py).  Values
// stay in registers between the statistics pass and the normalisation pass; fp32 arithmetic.
#include <initializer_list>
#include <mutex>
#include <tuple>
#include <type_traits>
#include <unordered_map>
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

template <int W> using Vec = std::conditional_t<W == 4, float4, float2>;   // W consecutive columns of one row

template <int W>
__device__ __forceinline__ Vec<W> ld(const LnTensor& t, long long idx) {       // idx: element index of the chunk's first column
  if (t.dt == MMN_DT_F32) return __ldg(reinterpret_cast<const Vec<W>*>(static_cast<const float*>(t.p) + idx));
  if constexpr (W == 4) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(static_cast<const __nv_bfloat16*>(t.p) + idx));
    return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16),
                       __uint_as_float(u.y & 0xffff0000u));
  } else {
    const uint32_t u = __ldg(reinterpret_cast<const uint32_t*>(static_cast<const __nv_bfloat16*>(t.p) + idx));
    return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u));
  }
}
template <int W>
__device__ __forceinline__ void st(const LnOut& t, long long idx, Vec<W> v) {
  if (t.dt == MMN_DT_F32) {
    *reinterpret_cast<Vec<W>*>(static_cast<float*>(t.p) + idx) = v;
  } else if constexpr (W == 4) {
    const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 u;
    u.x = *reinterpret_cast<const uint32_t*>(&a);
    u.y = *reinterpret_cast<const uint32_t*>(&b);
    *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(t.p) + idx) = u;
  } else {
    *reinterpret_cast<__nv_bfloat162*>(static_cast<__nv_bfloat16*>(t.p) + idx) = __floats2bfloat162_rn(v.x, v.y);
  }
}
template <int W>
__device__ __forceinline__ Vec<W> vzero() {
  if constexpr (W == 4) return make_float4(0.f, 0.f, 0.f, 0.f); else return make_float2(0.f, 0.f);
}
// f applied column by column: vmap(f, a, b) = {f(a.x, b.x), f(a.y, b.y), ...}
template <class F, class... T>
__device__ __forceinline__ float4 vmap(F f, float4 a, T... b) {
  return make_float4(f(a.x, b.x...), f(a.y, b.y...), f(a.z, b.z...), f(a.w, b.w...));
}
template <class F, class... T>
__device__ __forceinline__ float2 vmap(F f, float2 a, T... b) { return make_float2(f(a.x, b.x...), f(a.y, b.y...)); }
// sum of a chunk's columns and dot product of two chunks, in pairs: (x + y) + (z + w)
__device__ __forceinline__ float vsum(float4 a) { return (a.x + a.y) + (a.z + a.w); }
__device__ __forceinline__ float vsum(float2 a) { return a.x + a.y; }
__device__ __forceinline__ float vdot(float4 a, float4 b) { return (a.x * b.x + a.y * b.y) + (a.z * b.z + a.w * b.w); }
__device__ __forceinline__ float vdot(float2 a, float2 b) { return a.x * b.x + a.y * b.y; }
template <int LPR>
__device__ __forceinline__ float row_sum(float v) {          // sum over the LPR lanes that share a row
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

constexpr int kLnWarps = 8;

// MODE (pre- / post-norm) is a template parameter: the pre-norm forward keeps no residual copy and fits 64 registers (four
// blocks per SM); the post-norm one took 80-85 (three blocks) until it was asked for four as well: 32.3 -> 30.7 us at 110 592 x 96.
template <int W, int LPR, int V, int MODE>
__global__ void __launch_bounds__(kLnWarps * 32, V <= 3 ? 4 : 0)      // 0 = no occupancy request for the wide rows
layernorm_fwd_kernel(LnTensor resid, LnTensor delta, const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                     LnOut out_sum, LnOut out_norm, float* __restrict__ mean, float* __restrict__ rstd, long long rows, int cols) {
  constexpr int R = 32 / LPR;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lr = lane % LPR, sub = lane / LPR;
  const float inv_n = 1.f / (float)cols;
  const long long stride = (long long)gridDim.x * kLnWarps * R;
  for (long long row0 = ((long long)blockIdx.x * kLnWarps + warp) * R; row0 < rows; row0 += stride) {
    const long long row = row0 + sub;
    const bool live = row < rows;
    const long long base = row * cols;
    Vec<W> x[V], r[MODE == 0 ? 1 : V];    // x: the normalised quantity (PRE: resid + delta; POST: delta); r: the residual (POST)
    float s1 = 0.f;
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const int c = W * (lr + LPR * v);
      x[v] = vzero<W>();
      if (MODE != 0) r[v] = vzero<W>();
      if (live && c < cols) {
        if (MODE == 0) {
          if (resid.p) x[v] = ld<W>(resid, base + c);
          if (delta.p) x[v] = vmap([](float p, float q) { return p + q; }, x[v], ld<W>(delta, base + c));
        } else {
          x[v] = ld<W>(delta, base + c);
          if (resid.p) r[v] = ld<W>(resid, base + c);
        }
        s1 += vsum(x[v]);
      }
    }
    const float mu = row_sum<LPR>(s1) * inv_n;
    float s2 = 0.f;
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const int c = W * (lr + LPR * v);
      if (c < cols) {
        const Vec<W> a = vmap([&](float p) { return p - mu; }, x[v]);
        s2 += vdot(a, a);
      }
    }
    const float rs = rsqrtf(row_sum<LPR>(s2) * inv_n + eps);
    if (live && lr == 0) { mean[row] = mu; rstd[row] = rs; }
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const int c = W * (lr + LPR * v);
      if (live && c < cols) {
        // gamma / beta: loads that hit L1 (keeping them in registers cost half the occupancy)
        const Vec<W> g = __ldg(reinterpret_cast<const Vec<W>*>(gamma + c));
        const Vec<W> b = beta ? __ldg(reinterpret_cast<const Vec<W>*>(beta + c)) : vzero<W>();
        const Vec<W> n = vmap([&](float p, float gg, float bb) { return (p - mu) * rs * gg + bb; }, x[v], g, b);
        if (MODE == 0) {
          if (out_sum.p) st<W>(out_sum, base + c, x[v]);
          if (out_norm.p) st<W>(out_norm, base + c, n);
        } else {
          const Vec<W> s = vmap([](float p, float q) { return p + q; }, r[v], n);
          if (out_sum.p) st<W>(out_sum, base + c, s);
          if (out_norm.p) st<W>(out_norm, base + c, s);
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
template <int W, int LPR, int V, int MODE>
__global__ void __launch_bounds__(kLnWarps * 32, V <= 3 ? 3 : 1)
layernorm_bwd_kernel(LnTensor gs, LnTensor gn, LnTensor x, const float* __restrict__ gamma, const float* __restrict__ mean,
                     const float* __restrict__ rstd, LnOut d_resid, LnOut d_delta, float* __restrict__ dgamma,
                     float* __restrict__ dbeta, float* __restrict__ part, long long rows, int cols) {
  constexpr int R = 32 / LPR;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lr = lane % LPR, sub = lane / LPR;
  Vec<W> ag[V], ab[V];
#pragma unroll
  for (int v = 0; v < V; ++v) { ag[v] = vzero<W>(); ab[v] = vzero<W>(); }
  const float inv_n = 1.f / (float)cols;
  const long long stride = (long long)gridDim.x * kLnWarps * R;
  for (long long row0 = ((long long)blockIdx.x * kLnWarps + warp) * R; row0 < rows; row0 += stride) {
    const long long row = row0 + sub;
    const bool live = row < rows;
    const long long base = row * cols;
    // raw loads of the whole row first
    Vec<W> xv[V], a[V], n[V];
    const float mu = live ? __ldg(mean + row) : 0.f;
    const float rs = live ? __ldg(rstd + row) : 0.f;
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const int c = W * (lr + LPR * v);
      xv[v] = a[v] = n[v] = vzero<W>();
      if (live && c < cols) {
        xv[v] = ld<W>(x, base + c);
        if (gs.p) a[v] = ld<W>(gs, base + c);
        if (gn.p) n[v] = ld<W>(gn, base + c);
      }
    }
    // w = (gradient bypassing the LayerNorm) + rstd * u * gamma, u = gradient entering it: the row's output is
    // w - rstd * (m1 + xhat * m2), so only w and xhat live across the row reductions
    Vec<W> w[V], xh[V];
    float m1 = 0.f, m2 = 0.f;
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const int c = W * (lr + LPR * v);
      w[v] = xh[v] = vzero<W>();
      if (live && c < cols) {
        xh[v] = vmap([&](float p) { return (p - mu) * rs; }, xv[v]);
        const Vec<W> g = __ldg(reinterpret_cast<const Vec<W>*>(gamma + c));
        Vec<W> uu;
        if (MODE == 0) { uu = n[v]; w[v] = a[v]; }
        else {
          uu = vmap([](float p, float q) { return p + q; }, a[v], n[v]);
          if (d_resid.p) st<W>(d_resid, base + c, uu);
        }
        ag[v] = vmap([](float acc, float p, float q) { return acc + p * q; }, ag[v], uu, xh[v]);
        ab[v] = vmap([](float acc, float p) { return acc + p; }, ab[v], uu);
        const Vec<W> ug = vmap([](float p, float q) { return p * q; }, uu, g);
        m1 += vsum(ug);
        m2 += vdot(ug, xh[v]);
        w[v] = vmap([&](float p, float q) { return fmaf(rs, p, q); }, ug, w[v]);
      }
    }
    m1 = row_sum<LPR>(m1) * inv_n * rs;
    m2 = row_sum<LPR>(m2) * inv_n * rs;
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const int c = W * (lr + LPR * v);
      if (live && c < cols) {
        const Vec<W> t = vmap([&](float p, float q) { return p - m1 - q * m2; }, w[v], xh[v]);
        if (MODE == 0) {
          if (d_resid.p) st<W>(d_resid, base + c, t);
          if (d_delta.p) st<W>(d_delta, base + c, t);
        } else {
          if (d_delta.p) st<W>(d_delta, base + c, t);
        }
      }
    }
  }
  // column sums: rows of a warp (shuffles) -> warps (shared memory) -> one atomic per column and block
  __shared__ float red[kLnWarps][W * LPR * V];
  for (int pass_id = 0; pass_id < 2; ++pass_id) {
    float* dst = pass_id == 0 ? dgamma : dbeta;
    if (!dst) continue;                                      // uniform
#pragma unroll
    for (int v = 0; v < V; ++v) {
      Vec<W> acc = pass_id == 0 ? ag[v] : ab[v];
#pragma unroll
      for (int o = LPR; o < 32; o <<= 1) acc = vmap([&](float p) { return p + __shfl_xor_sync(0xffffffffu, p, o); }, acc);
      if (sub == 0) *reinterpret_cast<Vec<W>*>(&red[warp][W * (lr + LPR * v)]) = acc;
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

// The configurations {W, LPR, V} the kernels are built for: a row of cols columns runs on the first one of its chunk width
// whose LPR x V chunks cover it.  Past 768 columns (only cfg5's last stage, 64 rows) and at W = 2 (no workload) a few
// configurations cover the range instead of a full ladder.
template <int W_, int LPR_, int V_>
struct LnCfg { static constexpr int W = W_, LPR = LPR_, V = V_; };
using LnCfgs = std::tuple<LnCfg<4, 8, 1>, LnCfg<4, 8, 2>, LnCfg<4, 8, 3>, LnCfg<4, 16, 2>, LnCfg<4, 16, 3>, LnCfg<4, 32, 2>,
                          LnCfg<4, 32, 3>, LnCfg<4, 32, 4>, LnCfg<4, 32, 6>, LnCfg<4, 32, 8>, LnCfg<4, 32, 12>,
                          LnCfg<2, 32, 3>, LnCfg<2, 32, 16>, LnCfg<2, 32, 24>>;

// calls f(LnCfg<...>{}) with the configuration for (w, cols); false when the table has none
template <class F>
bool with_cfg(int w, int cols, F&& f) {
  return std::apply([&](auto... c) {
    return ((decltype(c)::W == w && cols <= decltype(c)::W * decltype(c)::LPR * decltype(c)::V && (f(c), true)) || ...);
  }, LnCfgs{});
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int chunk_width(int cols, std::initializer_list<const void*> operands) {
  if (cols % 4 != 0) return 2;
  for (const void* p : operands) if (!aligned16(p)) return 2;
  return 4;
}

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

// 256-thread blocks resident on one SM at most (2048 threads)
constexpr int kLnMaxBlocksPerSm = 2048 / (kLnWarps * 32);

// up to blocks_per_sm x 148 blocks (grid-stride loops inside)
int ln_grid(long long rows, int lpr, int blocks_per_sm) {
  const long long per_block = (long long)kLnWarps * (32 / lpr);
  const long long want = (rows + per_block - 1) / per_block;
  const long long cap = 148ll * (blocks_per_sm < kLnMaxBlocksPerSm ? blocks_per_sm : kLnMaxBlocksPerSm);
  return (int)(want < cap ? want : cap);
}

// adds the partials of the `blocks` the backward launched in block order
cudaError_t ln_reduce(const float* part, int blocks, int cols, float* dgamma, float* dbeta, cudaStream_t st, int* launches) {
  cudaError_t e = cudaSuccess;
  if (dgamma) e = reduce_partials(part, blocks, cols, dgamma, st, launches);
  if (e == cudaSuccess && dbeta) e = reduce_partials(part + (size_t)blocks * cols, blocks, cols, dbeta, st, launches);
  return e;
}

}  // namespace

bool layernorm_supported(int cols) { return cols >= 2 && cols % 2 == 0 && with_cfg(2, cols, [](auto) {}); }

cudaError_t layernorm_fwd(const void* resid, int resid_dt, const void* delta, int delta_dt, const float* gamma, const float* beta,
                          float eps, int mode, void* out_sum, int sum_dt, void* out_norm, int norm_dt, float* mean, float* rstd,
                          long long rows, int cols, cudaStream_t st, int* launches) {
  const LnTensor r{resid, resid_dt}, d{delta, delta_dt};
  const LnOut os{out_sum, sum_dt}, on{out_norm, norm_dt};
  const int w = chunk_width(cols, {resid, delta, out_sum, out_norm, gamma, beta});
  const bool found = with_cfg(w, cols, [&](auto c) {
    using C = decltype(c);
    auto k = mode == 0 ? layernorm_fwd_kernel<C::W, C::LPR, C::V, 0> : layernorm_fwd_kernel<C::W, C::LPR, C::V, 1>;
    k<<<ln_grid(rows, C::LPR, resident_blocks((const void*)k)), kLnWarps * 32, 0, st>>>(r, d, gamma, beta, eps, os, on, mean, rstd,
                                                                                        rows, cols);
  });
  if (!found) return cudaErrorInvalidValue;
  const cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) ++*launches;
  return e;
}

cudaError_t layernorm_bwd(const void* g_sum, int gs_dt, const void* g_norm, int gn_dt, const void* x, int x_dt, const float* gamma,
                          const float* mean, const float* rstd, int mode, void* d_resid, int dr_dt, void* d_delta, int dd_dt,
                          float* dgamma, float* dbeta, float* part, long long rows, int cols, cudaStream_t st, int* launches) {
  if (!dgamma && !dbeta) part = nullptr;
  const LnTensor gs{g_sum, gs_dt}, gn{g_norm, gn_dt}, xx{x, x_dt};
  const LnOut dr{d_resid, dr_dt}, dd{d_delta, dd_dt};
  const int w = chunk_width(cols, {g_sum, g_norm, x, d_resid, d_delta, gamma});
  int blocks = 0;
  const bool found = with_cfg(w, cols, [&](auto c) {
    using C = decltype(c);
    auto k = mode == 0 ? layernorm_bwd_kernel<C::W, C::LPR, C::V, 0> : layernorm_bwd_kernel<C::W, C::LPR, C::V, 1>;
    blocks = ln_grid(rows, C::LPR, resident_blocks((const void*)k));
    k<<<blocks, kLnWarps * 32, 0, st>>>(gs, gn, xx, gamma, mean, rstd, dr, dd, dgamma, dbeta, part, rows, cols);
  });
  if (!found) return cudaErrorInvalidValue;
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  ++*launches;
  return part ? ln_reduce(part, blocks, cols, dgamma, dbeta, st, launches) : cudaSuccess;
}

// A block covers kLnWarps * 32 / LPR >= kLnWarps rows and at most kLnMaxBlocksPerSm blocks are resident per SM, so this bounds
// the grid of every configuration; two rows of partials per block.
size_t layernorm_bwd_workspace_floats(long long rows, int cols) {
  return (size_t)(rows > 0 ? ln_grid(rows, 32, kLnMaxBlocksPerSm) : 0) * 2 * cols;
}

}  // namespace mmn
