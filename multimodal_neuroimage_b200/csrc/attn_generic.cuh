// attn_generic.cuh -- shape-generic attention kernels (CUDA cores, fp32 arithmetic).
//
// This is the fp32 parity path (north star: outputs and gradients within 1e-5 relative
// of the reference in fp32) and the path for the reference's own tiny shapes (head_dim
// 2..14, 9/36-token windows, SURVEY.md F8) where tensor cores have nothing to chew on.
// One kernel family serves both attention flavours of the hot path:
//   kind 0  window attention: item = (window, head); rows are gathered straight from the
//           un-windowed, un-shifted token grid, so torch.roll / window_partition /
//           window_reverse / roll-back never touch HBM.
//   kind 1  multi-head attention: item = (batch, head); rows addressed by (t, b) strides.
// Forward is flash-style: one thread owns one query row, keys/values are staged through
// shared memory in chunks, softmax is online so nothing N x N is ever materialised.
// Backward is two kernels with the same structure and roles swapped (dq: thread per
// query row; dkv: thread per key row), recomputing probabilities from the saved
// log-sum-exp; no atomics except the cross-window reductions dbias / dhead_scale.  The
// backward never reads the forward output: delta = rowsum(P o dP) is recomputed exactly.
// Deterministic mode passes no reduction outputs to those two kernels and computes them afterwards in a fixed order:
// attn_bias_grad_generic (dbias, dhead_scale partials) and the column-sum partials below (dcolsum).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "dropout_rng.cuh"

namespace mmn {

constexpr int kGenericThreads = 128;

struct GenericProblem {
  int kind;                       // 0 window, 1 mha
  int n_items, nq, nk, d, nH;
  int nW;                         // windows per sample (kind 0)
  int grid[3], win[3], shift[3], nwin[3];   // right-aligned: unused leading axes are 1 / 0
  long long q_s0, q_s1, k_s0, k_s1, v_s0, v_s1, o_s0, o_s1;
  long long do_s0, do_s1, dq_s0, dq_s1, dk_s0, dk_s1, dv_s0, dv_s1;
  int cosine;                     // 1: normalise q,k rows and multiply by head_scale[h]
  int mask_kind, mask_diag, mask_windows;
  float scale, dropout_p;
  unsigned long long seed, offset;
  DropoutCfg drop;                // the mask generator's constants (make_dropout(dropout_p, seed, offset))
  const float* bias;              // (nH, nq, nk) or null
  const float* head_scale;        // (nH) when cosine
  const float* mask;              // MMN_MASK_TENSOR
};

enum { kMaskNone = 0, kMaskShift = 1, kMaskTensor = 2, kMaskFuture = 3 };

__device__ __forceinline__ float ldf(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ldf(const __nv_bfloat16* p) { return __bfloat162float(*p); }
__device__ __forceinline__ void stf(float* p, float v) { *p = v; }
__device__ __forceinline__ void stf(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

// Token index (un-windowed, un-shifted order) of position p of window w: the composite of
// roll(-s) and window_partition (SURVEY.md a3), and the region id of the same position in
// the shifted frame (SURVEY.md a4).
__device__ __forceinline__ long long win_token(const GenericProblem& P, int w, int p, int* rid) {
  int b = w / P.nW, wl = w - b * P.nW;
  int i2 = wl % P.nwin[2]; int t = wl / P.nwin[2];
  int i1 = t % P.nwin[1];  int i0 = t / P.nwin[1];
  int a2 = p % P.win[2]; t = p / P.win[2];
  int a1 = t % P.win[1]; int a0 = t / P.win[1];
  int v0 = i0 * P.win[0] + a0, v1 = i1 * P.win[1] + a1, v2 = i2 * P.win[2] + a2;
  int r0 = P.shift[0] == 0 ? 0 : (v0 < P.grid[0] - P.win[0] ? 0 : (v0 < P.grid[0] - P.shift[0] ? 1 : 2));
  int r1 = P.shift[1] == 0 ? 0 : (v1 < P.grid[1] - P.win[1] ? 0 : (v1 < P.grid[1] - P.shift[1] ? 1 : 2));
  int r2 = P.shift[2] == 0 ? 0 : (v2 < P.grid[2] - P.win[2] ? 0 : (v2 < P.grid[2] - P.shift[2] ? 1 : 2));
  *rid = (r0 * 3 + r1) * 3 + r2;
  int c0 = v0 + P.shift[0]; if (c0 >= P.grid[0]) c0 -= P.grid[0];
  int c1 = v1 + P.shift[1]; if (c1 >= P.grid[1]) c1 -= P.grid[1];
  int c2 = v2 + P.shift[2]; if (c2 >= P.grid[2]) c2 -= P.grid[2];
  return (((long long)b * P.grid[0] + c0) * P.grid[1] + c1) * P.grid[2] + c2;
}

// Element offset of row `row` of item `item` for a tensor with strides (s0, s1).
__device__ __forceinline__ long long row_offset(const GenericProblem& P, int item, int row,
                                                long long s0, long long s1, int* rid) {
  int outer = item / P.nH, h = item - outer * P.nH;
  if (P.kind == 0) return win_token(P, outer, row, rid) * s0 + (long long)h * P.d;
  *rid = 0;
  return (long long)row * s0 + (long long)outer * s1 + (long long)h * P.d;
}

// Dropout keep-scale for probability (item, i, j): 0 or 1/(1-p).  Counter-based (dropout_rng.cuh), so the
// forward and both backward kernels -- and the tensor-core MHA kernels -- regenerate the same mask without storing it.
__device__ __forceinline__ float keep_scale(const GenericProblem& P, int item, int i, int j) {
  if (P.dropout_p <= 0.f) return 1.f;
  return dropout_keep(P.drop, item, i, j) ? P.drop.inv_keep : 0.f;
}

// Logit for (i, j) from the raw dot product.
__device__ __forceinline__ float logit(const GenericProblem& P, int item, float dot, int i, int j,
                                       int rid_i, int rid_j, float hscale) {
  float s = P.cosine ? dot * hscale : dot;
  int outer = item / P.nH, h = item - outer * P.nH;
  if (P.bias) s += __ldg(P.bias + ((long long)h * P.nq + i) * P.nk + j);
  if (P.mask_kind == kMaskShift) {
    s += (rid_i == rid_j) ? 0.f : -100.f;
  } else if (P.mask_kind == kMaskTensor) {
    long long m = P.kind == 0 ? (long long)(outer % P.mask_windows) * P.nq + i : (long long)i;
    s += __ldg(P.mask + m * P.nk + j);
  } else if (P.mask_kind == kMaskFuture) {
    if (j - i >= P.mask_diag) s = -INFINITY;
  }
  return s;
}

// 1 / max(||x||, 1e-12): F.normalize's denominator (swin_v2_module.py:153).
__device__ __forceinline__ float inv_norm(float sumsq) { return 1.f / fmaxf(sqrtf(sumsq), 1e-12f); }

// Stage `cnt` rows (row0 .. row0+cnt) of every slot's item into shared memory.
// dst: [slots][cap*d] floats; offs: [slots][cap] element offsets scratch; rid: [slots][cap].
// mode 0: raw.  mode 1: row-normalised (cosine).  `mul` scales every element (q scale).
template <typename T>
__device__ __forceinline__ void stage_rows(const GenericProblem& P, const T* __restrict__ src, long long s0,
                                           long long s1, int item0, int slots, int row0, int cnt, int cap,
                                           float* dst, long long* offs, int* rid, int mode, float mul) {
  const int t = threadIdx.x;
  for (int idx = t; idx < slots * cnt; idx += kGenericThreads) {
    int s = idx / cnt, j = idx - s * cnt, it = item0 + s, r = 0;
    long long o = 0;
    if (it < P.n_items) o = row_offset(P, it, row0 + j, s0, s1, &r);
    offs[s * cap + j] = o;
    if (rid) rid[s * cap + j] = r;
  }
  __syncthreads();
  const int per = cnt * P.d;
  for (int idx = t; idx < slots * per; idx += kGenericThreads) {
    int s = idx / per, rem = idx - s * per, j = rem / P.d, c = rem - j * P.d;
    float x = 0.f;
    if (item0 + s < P.n_items) x = ldf(src + offs[s * cap + j] + c) * mul;
    dst[(s * cap + j) * P.d + c] = x;
  }
  __syncthreads();
  if (mode == 1) {
    for (int idx = t; idx < slots * cnt; idx += kGenericThreads) {
      int s = idx / cnt, j = idx - s * cnt;
      float* rowp = dst + (s * cap + j) * P.d;
      float ss = 0.f;
      for (int c = 0; c < P.d; ++c) ss += rowp[c] * rowp[c];
      float inv = inv_norm(ss);
      for (int c = 0; c < P.d; ++c) rowp[c] *= inv;
    }
    __syncthreads();
  }
}

struct GenericLaunch {
  int rows_per_slot;   // min(rows, 128)
  int slots;           // items per block
  int chunk;           // rows of the "other side" staged per iteration
  size_t smem_bytes;
};

// ---------------------------------------------------------------------------------------
// Forward.  grid = (ceil(n_items / slots), ceil(nq / rows_per_slot)).
// ---------------------------------------------------------------------------------------
template <typename T, int DMAX>
__global__ void __launch_bounds__(kGenericThreads)
attn_fwd_generic(GenericProblem P, GenericLaunch L, const T* __restrict__ q, const T* __restrict__ k,
                 const T* __restrict__ v, T* __restrict__ out, float* __restrict__ lse) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int cap = L.chunk, slots = L.slots, d = P.d;
  long long* sOff = reinterpret_cast<long long*>(smem_raw);
  int* sRid = reinterpret_cast<int*>(sOff + slots * cap);
  float* sK = reinterpret_cast<float*>(sRid + slots * cap);
  float* sV = sK + slots * cap * d;

  const int t = threadIdx.x;
  const int slot = t / L.rows_per_slot, r_in = t - slot * L.rows_per_slot;
  const int item0 = blockIdx.x * slots;
  const int item = item0 + slot;
  const int row = blockIdx.y * L.rows_per_slot + r_in;
  const bool active = slot < slots && item < P.n_items && row < P.nq;

  float qr[DMAX], acc[DMAX];
  int rid_i = 0;
  long long o_off = 0;
  float hscale = 1.f;
  if (active) {
    long long qo = row_offset(P, item, row, P.q_s0, P.q_s1, &rid_i);
    o_off = row_offset(P, item, row, P.o_s0, P.o_s1, &rid_i);
    float ss = 0.f;
#pragma unroll
    for (int c = 0; c < DMAX; ++c) {
      qr[c] = c < d ? ldf(q + qo + c) : 0.f;
      ss += qr[c] * qr[c];
      acc[c] = 0.f;
    }
    float mul = P.cosine ? inv_norm(ss) : P.scale;
#pragma unroll
    for (int c = 0; c < DMAX; ++c) qr[c] *= mul;
    if (P.cosine) hscale = __ldg(P.head_scale + item % P.nH);
  }
  float m = -INFINITY, l = 0.f;

  for (int k0 = 0; k0 < P.nk; k0 += cap) {
    const int cnt = min(cap, P.nk - k0);
    stage_rows(P, k, P.k_s0, P.k_s1, item0, slots, k0, cnt, cap, sK, sOff, sRid, P.cosine ? 1 : 0, 1.f);
    stage_rows(P, v, P.v_s0, P.v_s1, item0, slots, k0, cnt, cap, sV, sOff, (int*)nullptr, 0, 1.f);
    if (active) {
      const float* Ks = sK + slot * cap * d;
      const float* Vs = sV + slot * cap * d;
      const int* Rs = sRid + slot * cap;
      for (int j = 0; j < cnt; ++j) {
        float dot = 0.f;
#pragma unroll
        for (int c = 0; c < DMAX; ++c) if (c < d) dot += qr[c] * Ks[j * d + c];
        float s = logit(P, item, dot, row, k0 + j, rid_i, Rs[j], hscale);
        if (s == -INFINITY) continue;
        float mn = fmaxf(m, s);
        float corr = expf(m - mn);                      // exp(-inf) = 0 on the first valid key
        float p = expf(s - mn);
        l = l * corr + p;
        float pk = p * keep_scale(P, item, row, k0 + j);
#pragma unroll
        for (int c = 0; c < DMAX; ++c) if (c < d) acc[c] = acc[c] * corr + pk * Vs[j * d + c];
        m = mn;
      }
    }
    __syncthreads();
  }
  if (active) {
    float inv = 1.f / l;
#pragma unroll
    for (int c = 0; c < DMAX; ++c) if (c < d) stf(out + o_off + c, acc[c] * inv);
    lse[(long long)item * P.nq + row] = m + logf(l);
  }
}

// ---------------------------------------------------------------------------------------
// Backward, query side: dq (+ dbias, dhead_scale).  Same launch geometry as forward.
// ---------------------------------------------------------------------------------------
template <typename T, int DMAX>
__global__ void __launch_bounds__(kGenericThreads)
attn_bwd_dq_generic(GenericProblem P, GenericLaunch L, const T* __restrict__ q, const T* __restrict__ k,
                    const T* __restrict__ v, const float* __restrict__ lse,
                    const T* __restrict__ dout, T* __restrict__ dq, float* __restrict__ dbias,
                    float* __restrict__ dhead_scale, float* __restrict__ delta_ws, float* __restrict__ dcolsum) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int cap = L.chunk, slots = L.slots, d = P.d;
  long long* sOff = reinterpret_cast<long long*>(smem_raw);
  int* sRid = reinterpret_cast<int*>(sOff + slots * cap);
  float* sK = reinterpret_cast<float*>(sRid + slots * cap);
  float* sV = sK + slots * cap * d;

  const int t = threadIdx.x;
  const int slot = t / L.rows_per_slot, r_in = t - slot * L.rows_per_slot;
  const int item0 = blockIdx.x * slots;
  const int item = item0 + slot;
  const int row = blockIdx.y * L.rows_per_slot + r_in;
  const bool active = slot < slots && item < P.n_items && row < P.nq;

  float qr[DMAX], dor[DMAX], dqr[DMAX];
  int rid_i = 0;
  long long dq_off = 0;
  float hscale = 1.f, delta = 0.f, psum = 0.f, lse_i = 0.f, qinv = 1.f, dscale = 0.f;
  if (active) {
    long long qo = row_offset(P, item, row, P.q_s0, P.q_s1, &rid_i);
    long long doo = row_offset(P, item, row, P.do_s0, P.do_s1, &rid_i);
    dq_off = row_offset(P, item, row, P.dq_s0, P.dq_s1, &rid_i);
    float ss = 0.f;
#pragma unroll
    for (int c = 0; c < DMAX; ++c) {
      qr[c] = c < d ? ldf(q + qo + c) : 0.f;
      dor[c] = c < d ? ldf(dout + doo + c) : 0.f;
      ss += qr[c] * qr[c];
      dqr[c] = 0.f;
    }
    qinv = P.cosine ? inv_norm(ss) : P.scale;
#pragma unroll
    for (int c = 0; c < DMAX; ++c) qr[c] *= qinv;
    if (P.cosine) hscale = __ldg(P.head_scale + item % P.nH);
    lse_i = lse[(long long)item * P.nq + row];
  }

  // Pass 0: delta_i = sum_j P_ij dP_ij (== dO_i . O_i), from the recomputed probabilities so
  // that no rounding of a low-precision `out` leaks into the cancellation-heavy reductions
  // (dhead_scale, dbias).  It is handed to the key-side kernel through `delta_ws`.
  for (int k0 = 0; k0 < P.nk; k0 += cap) {
    const int cnt = min(cap, P.nk - k0);
    stage_rows(P, k, P.k_s0, P.k_s1, item0, slots, k0, cnt, cap, sK, sOff, sRid, P.cosine ? 1 : 0, 1.f);
    stage_rows(P, v, P.v_s0, P.v_s1, item0, slots, k0, cnt, cap, sV, sOff, (int*)nullptr, 0, 1.f);
    if (active) {
      const float* Ks = sK + slot * cap * d;
      const float* Vs = sV + slot * cap * d;
      const int* Rs = sRid + slot * cap;
      for (int j = 0; j < cnt; ++j) {
        float dot = 0.f, dp = 0.f;
#pragma unroll
        for (int c = 0; c < DMAX; ++c) if (c < d) { dot += qr[c] * Ks[j * d + c]; dp += dor[c] * Vs[j * d + c]; }
        float s = logit(P, item, dot, row, k0 + j, rid_i, Rs[j], hscale);
        if (s == -INFINITY) continue;
        float p = expf(s - lse_i);
        psum += p;
        delta += p * dp * keep_scale(P, item, row, k0 + j);
      }
    }
    __syncthreads();
  }
  // exp(s - lse) sums to 1 only to within ulp(lse); with logits of magnitude ~100 that is
  // ~1e-5, and ds = p (dp - delta) turns a row-sum error into a bias that the reductions
  // over rows do not cancel.  Renormalise by the row sum actually obtained.
  const float pnorm = 1.f / psum;
  delta *= pnorm;
  if (active) {
    delta_ws[(long long)item * P.nq + row] = delta;
    delta_ws[(long long)P.n_items * P.nq + (long long)item * P.nq + row] = pnorm;
  }

  for (int k0 = 0; k0 < P.nk; k0 += cap) {
    const int cnt = min(cap, P.nk - k0);
    stage_rows(P, k, P.k_s0, P.k_s1, item0, slots, k0, cnt, cap, sK, sOff, sRid, P.cosine ? 1 : 0, 1.f);
    stage_rows(P, v, P.v_s0, P.v_s1, item0, slots, k0, cnt, cap, sV, sOff, (int*)nullptr, 0, 1.f);
    if (active) {
      const float* Ks = sK + slot * cap * d;
      const float* Vs = sV + slot * cap * d;
      const int* Rs = sRid + slot * cap;
      const int h = item % P.nH;
      for (int j = 0; j < cnt; ++j) {
        float dot = 0.f, dp = 0.f;
#pragma unroll
        for (int c = 0; c < DMAX; ++c) if (c < d) { dot += qr[c] * Ks[j * d + c]; dp += dor[c] * Vs[j * d + c]; }
        float s = logit(P, item, dot, row, k0 + j, rid_i, Rs[j], hscale);
        if (s == -INFINITY) continue;
        float p = expf(s - lse_i) * pnorm;
        float ds = p * (dp * keep_scale(P, item, row, k0 + j) - delta);
        float g = ds * hscale;
#pragma unroll
        for (int c = 0; c < DMAX; ++c) if (c < d) dqr[c] += g * Ks[j * d + c];
        if (dbias) atomicAdd(dbias + ((long long)h * P.nq + row) * P.nk + k0 + j, ds);
        dscale += ds * dot;
      }
    }
    __syncthreads();
  }
  if (active) {
    if (P.cosine) {
      // d/dq of q / max(||q||, eps): (g - qhat (qhat . g)) / ||q||   (qr holds qhat)
      float proj = 0.f;
#pragma unroll
      for (int c = 0; c < DMAX; ++c) proj += qr[c] * dqr[c];
      bool tiny = qinv >= 1e12f;                         // ||q|| < eps: qhat = q / eps, linear
#pragma unroll
      for (int c = 0; c < DMAX; ++c) dqr[c] = (dqr[c] - (tiny ? 0.f : qr[c] * proj)) * qinv;
      if (dhead_scale) atomicAdd(dhead_scale + item % P.nH, dscale);
    } else {
#pragma unroll
      for (int c = 0; c < DMAX; ++c) dqr[c] *= P.scale;
    }
#pragma unroll
    for (int c = 0; c < DMAX; ++c) if (c < d) {
      stf(dq + dq_off + c, dqr[c]);
      if (dcolsum) atomicAdd(dcolsum + (item % P.nH) * d + c, dqr[c]);
    }
  }
}

// ---------------------------------------------------------------------------------------
// Backward, key side: dk, dv.  Thread per key row; queries staged in chunks.
// grid = (ceil(n_items / slots), ceil(nk / rows_per_slot)), slots derived from nk.
// ---------------------------------------------------------------------------------------
template <typename T, int DMAX>
__global__ void __launch_bounds__(kGenericThreads)
attn_bwd_dkv_generic(GenericProblem P, GenericLaunch L, const T* __restrict__ q, const T* __restrict__ k,
                     const T* __restrict__ v, const float* __restrict__ lse, const float* __restrict__ delta_ws,
                     const T* __restrict__ dout, T* __restrict__ dk, T* __restrict__ dv, float* __restrict__ dcolsum) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int cap = L.chunk, slots = L.slots, d = P.d;
  long long* sOff = reinterpret_cast<long long*>(smem_raw);
  int* sRid = reinterpret_cast<int*>(sOff + slots * cap);
  float* sLse = reinterpret_cast<float*>(sRid + slots * cap);
  float* sDelta = sLse + slots * cap;
  float* sNorm = sDelta + slots * cap;
  float* sQ = sNorm + slots * cap;
  float* sDO = sQ + slots * cap * d;

  const int t = threadIdx.x;
  const int slot = t / L.rows_per_slot, r_in = t - slot * L.rows_per_slot;
  const int item0 = blockIdx.x * slots;
  const int item = item0 + slot;
  const int col = blockIdx.y * L.rows_per_slot + r_in;
  const bool active = slot < slots && item < P.n_items && col < P.nk;

  float kr[DMAX], vr[DMAX], dkr[DMAX], dvr[DMAX];
  int rid_j = 0;
  long long dk_off = 0, dv_off = 0;
  float hscale = 1.f, kinv = 1.f;
  if (active) {
    long long ko = row_offset(P, item, col, P.k_s0, P.k_s1, &rid_j);
    long long vo = row_offset(P, item, col, P.v_s0, P.v_s1, &rid_j);
    dk_off = row_offset(P, item, col, P.dk_s0, P.dk_s1, &rid_j);
    dv_off = row_offset(P, item, col, P.dv_s0, P.dv_s1, &rid_j);
    float ss = 0.f;
#pragma unroll
    for (int c = 0; c < DMAX; ++c) {
      kr[c] = c < d ? ldf(k + ko + c) : 0.f;
      vr[c] = c < d ? ldf(v + vo + c) : 0.f;
      ss += kr[c] * kr[c];
      dkr[c] = 0.f; dvr[c] = 0.f;
    }
    if (P.cosine) {
      kinv = inv_norm(ss);
#pragma unroll
      for (int c = 0; c < DMAX; ++c) kr[c] *= kinv;
      hscale = __ldg(P.head_scale + item % P.nH);
    }
  }

  for (int q0 = 0; q0 < P.nq; q0 += cap) {
    const int cnt = min(cap, P.nq - q0);
    stage_rows(P, q, P.q_s0, P.q_s1, item0, slots, q0, cnt, cap, sQ, sOff, sRid, P.cosine ? 1 : 0,
               P.cosine ? 1.f : P.scale);
    stage_rows(P, dout, P.do_s0, P.do_s1, item0, slots, q0, cnt, cap, sDO, sOff, (int*)nullptr, 0, 1.f);
    for (int idx = t; idx < slots * cnt; idx += kGenericThreads) {
      int s = idx / cnt, i = idx - s * cnt, it = item0 + s;
      float dl = 0.f, ls = 0.f, pn = 0.f;
      if (it < P.n_items) {
        dl = delta_ws[(long long)it * P.nq + q0 + i];
        pn = delta_ws[(long long)P.n_items * P.nq + (long long)it * P.nq + q0 + i];
        ls = lse[(long long)it * P.nq + q0 + i];
      }
      sDelta[s * cap + i] = dl;
      sNorm[s * cap + i] = pn;
      sLse[s * cap + i] = ls;
    }
    __syncthreads();
    if (active) {
      const float* Qs = sQ + slot * cap * d;
      const float* DOs = sDO + slot * cap * d;
      const int* Rs = sRid + slot * cap;
      for (int i = 0; i < cnt; ++i) {
        float dot = 0.f, dp = 0.f;
#pragma unroll
        for (int c = 0; c < DMAX; ++c) if (c < d) { dot += Qs[i * d + c] * kr[c]; dp += DOs[i * d + c] * vr[c]; }
        float s = logit(P, item, dot, q0 + i, col, Rs[i], rid_j, hscale);
        if (s == -INFINITY) continue;
        float p = expf(s - sLse[slot * cap + i]) * sNorm[slot * cap + i];
        float ks = keep_scale(P, item, q0 + i, col);
        float ds = p * (dp * ks - sDelta[slot * cap + i]);
        float pk = p * ks, g = ds * hscale;
#pragma unroll
        for (int c = 0; c < DMAX; ++c) if (c < d) { dvr[c] += pk * DOs[i * d + c]; dkr[c] += g * Qs[i * d + c]; }
      }
    }
    __syncthreads();
  }
  if (active) {
    float proj = 0.f;
    if (P.cosine) {
#pragma unroll
      for (int c = 0; c < DMAX; ++c) proj += kr[c] * dkr[c];
      if (kinv >= 1e12f) proj = 0.f;
    }
#pragma unroll
    for (int c = 0; c < DMAX; ++c) if (c < d) {
      const float dkc = P.cosine ? (dkr[c] - kr[c] * proj) * kinv : dkr[c];
      stf(dk + dk_off + c, dkc);
      stf(dv + dv_off + c, dvr[c]);
      if (dcolsum) {
        const int C = P.nH * d, hc = (item % P.nH) * d + c;
        atomicAdd(dcolsum + C + hc, dkc);
        atomicAdd(dcolsum + 2 * C + hc, dvr[c]);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------
// Deterministic mode: dbias and dhead_scale without atomics.  Thread per (h, i, j): walks head h's windows in order and
// recomputes ds_ij exactly as attn_bwd_dq_generic does (delta and the row normaliser come from delta_ws), adds sum_w ds
// into dbias[h][i][j] and writes sum_w ds * dot to dsp[(i * nk + j) * nH + h], which reduce_partials turns into
// dhead_scale.  Window attention (kind 0) only.
// ---------------------------------------------------------------------------------------
template <typename T, int DMAX>
__global__ void __launch_bounds__(kGenericThreads)
attn_bias_grad_generic(GenericProblem P, const T* __restrict__ q, const T* __restrict__ k, const T* __restrict__ v,
                       const float* __restrict__ lse, const T* __restrict__ dout, const float* __restrict__ delta_ws,
                       float* __restrict__ dbias, float* __restrict__ dsp) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)P.nH * P.nq * P.nk) return;
  const int j = (int)(idx % P.nk);
  const long long r = idx / P.nk;
  const int i = (int)(r % P.nq), h = (int)(r / P.nq), d = P.d;
  const float hscale = P.cosine ? __ldg(P.head_scale + h) : 1.f;
  float db = 0.f, dsd = 0.f;
  for (int outer = 0; outer < P.n_items / P.nH; ++outer) {
    const int item = outer * P.nH + h;
    int rid_i, rid_j;
    const long long qo = row_offset(P, item, i, P.q_s0, P.q_s1, &rid_i), doo = row_offset(P, item, i, P.do_s0, P.do_s1, &rid_i);
    const long long ko = row_offset(P, item, j, P.k_s0, P.k_s1, &rid_j), vo = row_offset(P, item, j, P.v_s0, P.v_s1, &rid_j);
    float qr[DMAX], kr[DMAX];
    float qss = 0.f, kss = 0.f;
#pragma unroll
    for (int c = 0; c < DMAX; ++c) {
      qr[c] = c < d ? ldf(q + qo + c) : 0.f;
      kr[c] = c < d ? ldf(k + ko + c) : 0.f;
      qss += qr[c] * qr[c];
    }
    for (int c = 0; c < d; ++c) kss += kr[c] * kr[c];
    const float qmul = P.cosine ? inv_norm(qss) : P.scale, kmul = P.cosine ? inv_norm(kss) : 1.f;
    float dot = 0.f, dp = 0.f;
#pragma unroll
    for (int c = 0; c < DMAX; ++c)
      if (c < d) { dot += (qr[c] * qmul) * (kr[c] * kmul); dp += ldf(dout + doo + c) * ldf(v + vo + c); }
    const float s = logit(P, item, dot, i, j, rid_i, rid_j, hscale);
    if (s == -INFINITY) continue;
    const long long row = (long long)item * P.nq + i;
    const float p = expf(s - lse[row]) * delta_ws[(long long)P.n_items * P.nq + row];
    const float ds = p * (dp * keep_scale(P, item, i, j) - delta_ws[row]);
    db += ds;
    dsd += ds * dot;
  }
  if (dbias) dbias[idx] += db;
  if (dsp) dsp[((long long)i * P.nk + j) * P.nH + h] = dsd;
}

// Deterministic column sums, any width: block b sums rows [b * rpb, (b + 1) * rpb) of every column into part[b][c].
template <typename T>
__global__ void __launch_bounds__(256)
colsum_part_any(const T* __restrict__ x, long long rows, int cols, long long row_stride, long long rpb, float* __restrict__ part) {
  const long long r0 = (long long)blockIdx.x * rpb, r1 = r0 + rpb < rows ? r0 + rpb : rows;
  for (int c = threadIdx.x; c < cols; c += blockDim.x) {
    float acc = 0.f;
    for (long long r = r0; r < r1; ++r) acc += ldf(x + r * row_stride + c);
    part[(size_t)blockIdx.x * cols + c] = acc;
  }
}

// ---------------------------------------------------------------------------------------
// Head-averaged attention probabilities (multihead_attention.py:131-133): thread per (b,i,j).
// ---------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
mha_avg_weights_generic(GenericProblem P, int B, const T* __restrict__ q, const T* __restrict__ k,
                        const float* __restrict__ lse, float* __restrict__ avg) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = (long long)B * P.nq * P.nk;
  if (idx >= total) return;
  int j = (int)(idx % P.nk);
  long long r = idx / P.nk;
  int i = (int)(r % P.nq), b = (int)(r / P.nq);
  float sum = 0.f;
  for (int h = 0; h < P.nH; ++h) {
    int item = b * P.nH + h, rid;
    const T* qp = q + row_offset(P, item, i, P.q_s0, P.q_s1, &rid);
    const T* kp = k + row_offset(P, item, j, P.k_s0, P.k_s1, &rid);
    float dot = 0.f;
    for (int c = 0; c < P.d; ++c) dot += ldf(qp + c) * P.scale * ldf(kp + c);
    float s = logit(P, item, dot, i, j, 0, 0, 1.f);
    if (s != -INFINITY) sum += expf(s - lse[(long long)item * P.nq + i]) * keep_scale(P, item, i, j);
  }
  avg[idx] = sum / (float)P.nH;
}


// ---------------------------------------------------------------------------------------
// Column sums of a (rows, cols) matrix into fp32 (accumulated): the bias gradient of a
// projection, at memory speed.  Thread = 8 consecutive columns; a block strides over rows.
// part != null (deterministic mode): the block's sums go to part[blockIdx.x][c] instead of atomics into out.
// ---------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
colsum_kernel(const T* __restrict__ x, long long rows, int cols, long long row_stride, float* __restrict__ out,
              float* __restrict__ part) {
  constexpr int V = 8;
  const int vcols = cols / V;
  const int rpb = 256 / vcols;                        // rows handled in parallel by a block
  const int tx = threadIdx.x % vcols, ty = threadIdx.x / vcols;
  float acc[V];
#pragma unroll
  for (int e = 0; e < V; ++e) acc[e] = 0.f;
  if (ty < rpb) {
    const long long r0 = (long long)blockIdx.x * rpb + ty, step = (long long)gridDim.x * rpb;
    if (sizeof(T) == 2 && row_stride % 8 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0) {
      // bf16 rows: one 16-byte load per row and thread, four rows in flight
      long long r = r0;
      for (; r + 3 * step < rows; r += 4 * step) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = __ldg(reinterpret_cast<const uint4*>(x + (r + u * step) * row_stride + tx * V));
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint32_t w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
          for (int e = 0; e < 4; ++e) { acc[2 * e] += __uint_as_float(w[e] << 16); acc[2 * e + 1] += __uint_as_float(w[e] & 0xffff0000u); }
        }
      }
      for (; r < rows; r += step) {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(x + r * row_stride + tx * V));
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) { acc[2 * e] += __uint_as_float(w[e] << 16); acc[2 * e + 1] += __uint_as_float(w[e] & 0xffff0000u); }
      }
    } else {
      for (long long r = r0; r < rows; r += step) {
        const T* p = x + r * row_stride + tx * V;
#pragma unroll
        for (int e = 0; e < V; ++e) acc[e] += ldf(p + e);
      }
    }
  }
  __shared__ float red[256 * V];
#pragma unroll
  for (int e = 0; e < V; ++e) red[threadIdx.x * V + e] = ty < rpb ? acc[e] : 0.f;
  __syncthreads();
  for (int c = threadIdx.x; c < vcols * V; c += 256) {   // column (cols may exceed the block size: up to 2048)
    float s = 0.f;
    for (int y = 0; y < rpb; ++y) s += red[(y * vcols + c / V) * V + c % V];
    if (part) part[(size_t)blockIdx.x * cols + c] = s;
    else atomicAdd(out + c, s);
  }
}

}  // namespace mmn
