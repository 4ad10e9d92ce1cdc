// cpb_bias.cu -- SwinV2's continuous relative-position bias (swin_v2_module.py:158-162) as two small kernels
// forward and three backward, instead of the ~25 ATen/cuBLAS launches autograd spends on it every step:
//
//   tab[t][h]   = sum_j W2[h][j] relu(W1[j] . coords[t] + b1[j])          t < T = prod(2w-1), hidden j < J (512)
//   bias[h][e]  = 16 sigmoid(tab[index[e]][h])                            e < N*N
//
// The sizes are tiny (T = 343, J = 512, nH = 3 at BASELINE cfg2); the point is launch count, not flops.
// fp32 throughout (the bias feeds logits that reach +-100; the parity bar for this row is 1e-5).
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>

#include "generic_launch.h"
#include "zero_fill.h"

namespace mmn {

constexpr int kCpbMaxIn = 3;      // spatial dims of the coordinate table
constexpr int kCpbMaxHeads = 64;

// grid = T blocks, 128 threads: tab16[t][h] = 16 sigmoid(...)
__global__ void __launch_bounds__(128)
cpb_table_kernel(const float* __restrict__ coords, const float* __restrict__ w1, const float* __restrict__ b1,
                 const float* __restrict__ w2, int n_in, int J, int nH, float* __restrict__ tab16) {
  __shared__ float red[4][kCpbMaxHeads];
  const int t = blockIdx.x, tid = threadIdx.x;
  float c[kCpbMaxIn];
  for (int a = 0; a < kCpbMaxIn; ++a) c[a] = a < n_in ? __ldg(coords + t * n_in + a) : 0.f;
  // each thread: a strided subset of the hidden units, partial dot products with every head's W2 row
  for (int h0 = 0; h0 < nH; h0 += 8) {
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int j = tid; j < J; j += 128) {
      float z = __ldg(b1 + j);
      for (int a = 0; a < n_in; ++a) z = fmaf(__ldg(w1 + j * n_in + a), c[a], z);
      z = fmaxf(z, 0.f);
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (h0 + k < nH) acc[k] = fmaf(__ldg(w2 + (h0 + k) * J + j), z, acc[k]);
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float v = acc[k];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if ((tid & 31) == 0 && h0 + k < nH) red[tid >> 5][h0 + k] = v;
    }
  }
  __syncthreads();
  if (tid < nH) {
    const float s = (red[0][tid] + red[1][tid]) + (red[2][tid] + red[3][tid]);
    tab16[t * nH + tid] = 16.f / (1.f + __expf(-s));
  }
}

// bias[h][e] = tab16[index[e]][h]
__global__ void cpb_gather_kernel(const float* __restrict__ tab16, const long long* __restrict__ index, int NN, int nH,
                                  float* __restrict__ bias) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= NN) return;
  const long long t = index[e];
  for (int h = 0; h < nH; ++h) bias[(size_t)h * NN + e] = __ldg(tab16 + t * nH + h);
}

// dtab16[index[e]][h] += dbias[h][e]   (dtab16 zeroed by the caller of this kernel)
__global__ void cpb_scatter_kernel(const float* __restrict__ dbias, const long long* __restrict__ index, int NN, int nH,
                                   float* __restrict__ dtab16) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= NN) return;
  const long long t = index[e];
  for (int h = 0; h < nH; ++h) atomicAdd(dtab16 + t * nH + h, __ldg(dbias + (size_t)h * NN + e));
}

// Deterministic variant of the scatter: a gather over the inverse of `index` in CSR form (inv_perm = the entries e sorted
// by (index[e], e), inv_offsets = the run of each table entry).  Thread per (t, h) sums dbias[h][e] over its run in
// increasing e.  An inverse that does not cover NN entries is not the inverse of this index: the output becomes NaN.
__global__ void cpb_gather_grad_kernel(const float* __restrict__ dbias, const int* __restrict__ inv_perm, const int* __restrict__ inv_offsets,
                                       int T, int NN, int nH, float* __restrict__ dtab16) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= T * nH) return;
  const int t = x / nH, h = x - t * nH;
  float acc = 0.f;
  if (__ldg(inv_offsets + T) != NN) {
    acc = __int_as_float(0x7fffffff);
  } else {
    const float* row = dbias + (size_t)h * NN;
    for (int k = __ldg(inv_offsets + t), k1 = __ldg(inv_offsets + t + 1); k < k1; ++k) acc += __ldg(row + __ldg(inv_perm + k));
  }
  dtab16[x] = acc;
}

// dtab[t][h] = sum over e with index[e] == t of dbias[h][e]: the scatter (after zeroing) or, with the inverse index, the gather
cudaError_t table_grad(const float* dbias, const long long* index, const int* inv_perm, const int* inv_offsets, int T, int nH, int NN,
                       float* dtab, cudaStream_t st) {
  if (inv_perm) {
    cpb_gather_grad_kernel<<<(T * nH + 255) / 256, 256, 0, st>>>(dbias, inv_perm, inv_offsets, T, NN, nH, dtab);
    return cudaGetLastError();
  }
  cudaError_t e = zero_words_async(dtab, (size_t)T * nH, st);
  if (e != cudaSuccess) return e;
  cpb_scatter_kernel<<<(NN + 255) / 256, 256, 0, st>>>(dbias, index, NN, nH, dtab);
  return cudaGetLastError();
}

// Backward of the MLP.  A block owns 32 hidden units; its 16 warps split the T table entries (warp w takes
// t = w, w + 16, ...), every thread recomputes its unit's activation and accumulates dW2[:, j], dW1[j, :], db1[j] for
// its slice in registers; the 16 slices are then summed through shared memory in a fixed order (this kernel uses no
// atomics; the scatter of dbias into the table before it, cpb_scatter_kernel, does -- float atomicAdd, so the
// last bits of the CPB gradients can differ from run to run unless the deterministic gather replaces it).  g[t][h] = d tab[t][h] is staged in shared memory eight heads at a time:
// d/dx 16 sigmoid(x) = tab16 (1 - tab16 / 16).  (One thread per hidden unit walking all T entries alone -- four blocks
// on four SMs -- took 58 us at BASELINE cfg2, 4 % of the whole fused-module step.)
constexpr int kCpbBwdUnits = 32, kCpbBwdSlices = 16;
__global__ void __launch_bounds__(kCpbBwdUnits * kCpbBwdSlices)
cpb_mlp_bwd_kernel(const float* __restrict__ coords, const float* __restrict__ w1, const float* __restrict__ b1,
                   const float* __restrict__ w2, const float* __restrict__ tab16, const float* __restrict__ dtab16, int T, int n_in,
                   int J, int nH, float* __restrict__ dw1, float* __restrict__ db1, float* __restrict__ dw2) {
  extern __shared__ float sm[];
  float* sc = sm;                              // [T][3] coordinates (zero-padded to 3)
  float* g = sc + ((T * kCpbMaxIn + 3) & ~3);  // [T][8] (16-byte aligned) gradient w.r.t. the pre-sigmoid table, current head group
  float* red = g + T * 8;                      // [slices][8][units]
  const int tid = threadIdx.x, js = tid & (kCpbBwdUnits - 1), ts = tid / kCpbBwdUnits;
  const int j = blockIdx.x * kCpbBwdUnits + js;
  const bool live = j < J;
  for (int i = tid; i < T * kCpbMaxIn; i += blockDim.x) {
    const int t = i / kCpbMaxIn, a = i - t * kCpbMaxIn;
    sc[i] = a < n_in ? __ldg(coords + t * n_in + a) : 0.f;
  }
  float wj[kCpbMaxIn], dwj[kCpbMaxIn] = {0.f, 0.f, 0.f};
  for (int a = 0; a < kCpbMaxIn; ++a) wj[a] = (live && a < n_in) ? __ldg(w1 + j * n_in + a) : 0.f;
  const float bj = live ? __ldg(b1 + j) : 0.f;
  float dbj = 0.f;
  // sum `v` over the slices (fixed order); valid in the threads of slice 0
  auto reduce8 = [&](const float (&v)[8], float (&out)[8]) {
#pragma unroll
    for (int k = 0; k < 8; ++k) red[(ts * 8 + k) * kCpbBwdUnits + js] = v[k];
    __syncthreads();
    if (ts == 0) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        float acc = 0.f;
        for (int s2 = 0; s2 < kCpbBwdSlices; ++s2) acc += red[(s2 * 8 + k) * kCpbBwdUnits + js];
        out[k] = acc;
      }
    }
    __syncthreads();
  };
  for (int h0 = 0; h0 < nH; h0 += 8) {         // heads in groups of 8 register accumulators
    __syncthreads();                           // previous group's g is no longer read
    for (int i = tid; i < T * 8; i += blockDim.x) {
      const int t = i >> 3, k = i & 7;
      float v = 0.f;
      if (h0 + k < nH) {
        const float s16 = __ldg(tab16 + t * nH + h0 + k);
        v = __ldg(dtab16 + t * nH + h0 + k) * s16 * (1.f - s16 * (1.f / 16.f));
      }
      g[i] = v;
    }
    __syncthreads();
    float w2j[8], dw2j[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { w2j[k] = (live && h0 + k < nH) ? __ldg(w2 + (h0 + k) * J + j) : 0.f; dw2j[k] = 0.f; }
    for (int t = ts; t < T; t += kCpbBwdSlices) {
      const float c0 = sc[t * 3], c1 = sc[t * 3 + 1], c2 = sc[t * 3 + 2];
      const float z = fmaf(wj[2], c2, fmaf(wj[1], c1, fmaf(wj[0], c0, bj)));
      const float act = fmaxf(z, 0.f);
      const float4 ga = *reinterpret_cast<const float4*>(g + t * 8), gb = *reinterpret_cast<const float4*>(g + t * 8 + 4);
      const float gt[8] = {ga.x, ga.y, ga.z, ga.w, gb.x, gb.y, gb.z, gb.w};
      float dh = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        dw2j[k] = fmaf(gt[k], act, dw2j[k]);
        dh = fmaf(gt[k], w2j[k], dh);
      }
      if (z > 0.f) {
        dbj += dh;
        dwj[0] = fmaf(dh, c0, dwj[0]); dwj[1] = fmaf(dh, c1, dwj[1]); dwj[2] = fmaf(dh, c2, dwj[2]);
      }
    }
    float tot[8];
    reduce8(dw2j, tot);
    if (ts == 0 && live) {
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (h0 + k < nH) dw2[(h0 + k) * J + j] = tot[k];
    }
  }
  const float rest[8] = {dbj, dwj[0], dwj[1], dwj[2], 0.f, 0.f, 0.f, 0.f};
  float tot[8];
  reduce8(rest, tot);
  if (ts == 0 && live) {
    db1[j] = tot[0];
    for (int a = 0; a < n_in; ++a) dw1[j * n_in + a] = tot[1 + a];
  }
}

// dynamic shared memory of cpb_mlp_bwd_kernel: coords [T][3] + g [T][8] + the slice-reduction buffer
size_t cpb_bwd_smem_bytes(int T) {
  return ((size_t)((T * kCpbMaxIn + 3) & ~3) + (size_t)T * 8 + (size_t)kCpbBwdSlices * 8 * kCpbBwdUnits) * sizeof(float);
}

// Learned relative-position bias table (swinfusion_module.py:127-130): the same gather / scatter without the MLP.
cudaError_t table_bias_fwd(const float* table, const long long* index, int nH, int NN, float* bias, cudaStream_t st, int* launches) {
  cpb_gather_kernel<<<(NN + 255) / 256, 256, 0, st>>>(table, index, NN, nH, bias);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) *launches += 1;
  return e;
}

cudaError_t table_bias_bwd(const float* dbias, const long long* index, const int* inv_perm, const int* inv_offsets, int T, int nH, int NN,
                           float* dtable, cudaStream_t st, int* launches) {
  cudaError_t e = table_grad(dbias, index, inv_perm, inv_offsets, T, nH, NN, dtable, st);
  if (e == cudaSuccess) *launches += 1;
  return e;
}

cudaError_t cpb_bias_fwd(const float* coords, const float* w1, const float* b1, const float* w2, const long long* index, int T,
                         int n_in, int J, int nH, int NN, float* tab16, float* bias, cudaStream_t st, int* launches) {
  cpb_table_kernel<<<T, 128, 0, st>>>(coords, w1, b1, w2, n_in, J, nH, tab16);
  cpb_gather_kernel<<<(NN + 255) / 256, 256, 0, st>>>(tab16, index, NN, nH, bias);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) *launches += 2;
  return e;
}

cudaError_t cpb_bias_bwd(const float* coords, const float* w1, const float* b1, const float* w2, const long long* index,
                         const int* inv_perm, const int* inv_offsets, const float* tab16, const float* dbias, int T, int n_in, int J,
                         int nH, int NN, float* dtab16, float* dw1, float* db1, float* dw2, cudaStream_t st, int* launches) {
  cudaError_t e = table_grad(dbias, index, inv_perm, inv_offsets, T, nH, NN, dtab16, st);
  if (e != cudaSuccess) return e;
  const size_t smem = cpb_bwd_smem_bytes(T);
  if (smem > 48 * 1024) {      // 2-D windows of 16 (T = 961), 3-D windows of 6 / 7 (T = 1331 / 2197): opt in to large dynamic smem
    static std::once_flag once;
    std::call_once(once, [] { cudaFuncSetAttribute(cpb_mlp_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024); });
  }
  cpb_mlp_bwd_kernel<<<(J + kCpbBwdUnits - 1) / kCpbBwdUnits, kCpbBwdUnits * kCpbBwdSlices, smem, st>>>(coords, w1, b1, w2, tab16, dtab16, T,
                                                                                                    n_in, J, nH, dw1, db1, dw2);
  e = cudaGetLastError();
  if (e == cudaSuccess) *launches += 2;
  return e;
}

}  // namespace mmn
