// generic_launch.cu -- instantiates and launches the shape-generic kernels.
#include "generic_launch.h"
#include "zero_fill.h"

#include "../../include/mmn_b200.h"

namespace mmn {

// out[e] += sum over s < nparts of part[s * n + e], s in increasing order within each of 32 slices, the slices added in
// a fixed tree (as gemm_reduce_kernel: a latency-bound reduction wants at most a few loads per thread).
constexpr int kRedSlices = 32;
__global__ void __launch_bounds__(kRedSlices * 32)
reduce_partials_kernel(const float* __restrict__ part, int nparts, long long n, float* __restrict__ out) {
  __shared__ float red[kRedSlices][33];
  const int lane = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const long long e = (long long)blockIdx.x * 32 + lane;
  float acc = 0.f;
  if (e < n) {
#pragma unroll 4
    for (int s = sl; s < nparts; s += kRedSlices) acc += __ldg(part + (size_t)s * n + e);
  }
  red[sl][lane] = acc;
  __syncthreads();
  if (sl < 4) {
    acc = red[8 * sl][lane];
#pragma unroll
    for (int k = 1; k < 8; ++k) acc += red[8 * sl + k][lane];
    red[8 * sl][lane] = acc;
  }
  __syncthreads();
  if (sl == 0 && e < n) out[e] += (acc + red[8][lane]) + (red[16][lane] + red[24][lane]);
}

namespace {

// rows: extent of the thread-per-row side; other: extent of the staged side;
// floats_per_staged_row: shared floats per staged row excluding the 12-byte offset/rid.
mmn::GenericLaunch plan(int rows, int other, int bytes_per_staged_row) {
  mmn::GenericLaunch L{};
  L.rows_per_slot = rows < mmn::kGenericThreads ? rows : mmn::kGenericThreads;
  L.slots = mmn::kGenericThreads / L.rows_per_slot;
  const size_t budget = 96 * 1024;
  int cap = (int)(budget / ((size_t)L.slots * bytes_per_staged_row));
  if (cap > other) cap = other;
  if (cap > 256) cap = 256;
  if (cap < 1) cap = 1;
  L.chunk = cap;
  L.smem_bytes = (size_t)L.slots * cap * bytes_per_staged_row;
  return L;
}

constexpr int kMaxSmem = 100 * 1024;

template <typename T, int DMAX>
cudaError_t launch_fwd(const mmn::GenericProblem& P, const void* q, const void* k, const void* v, void* out, float* lse, cudaStream_t st, int* launches) {
  mmn::GenericLaunch L = plan(P.nq, P.nk, 2 * P.d * 4 + 12);
  auto kern = mmn::attn_fwd_generic<T, DMAX>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
  dim3 grid((P.n_items + L.slots - 1) / L.slots, (P.nq + L.rows_per_slot - 1) / L.rows_per_slot);
  kern<<<grid, mmn::kGenericThreads, L.smem_bytes, st>>>(P, L, (const T*)q, (const T*)k, (const T*)v, (T*)out, lse);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) ++*launches;
  return e;
}

long long tokens(const mmn::GenericProblem& P) { return (long long)(P.n_items / P.nH / P.nW) * P.grid[0] * P.grid[1] * P.grid[2]; }
int colsum_any_blocks(long long rows) { return (int)((rows + 63) / 64 < 592 ? (rows + 63) / 64 : 592); }

template <typename T>
cudaError_t colsum_det_any(const T* x, long long rows, int cols, long long row_stride, float* out, float* part, cudaStream_t st,
                           int* launches) {
  const int blocks = colsum_any_blocks(rows);
  colsum_part_any<T><<<blocks, 256, 0, st>>>(x, rows, cols, row_stride, (rows + blocks - 1) / blocks, part);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  ++*launches;
  return reduce_partials(part, blocks, cols, out, st, launches);
}

template <typename T, int DMAX>
cudaError_t launch_bwd(const mmn::GenericProblem& P, const void* q, const void* k, const void* v, const float* lse,
               const void* dout, void* dq, void* dk, void* dv, float* dbias, float* dhs, float* ws, float* dcs, bool det, cudaStream_t st,
               int* launches) {
  if (det) {
    cudaError_t e = launch_bwd<T, DMAX>(P, q, k, v, lse, dout, dq, dk, dv, nullptr, nullptr, ws, nullptr, false, st, launches);
    if (e != cudaSuccess) return e;
    float* dsp = ws + 2 * (long long)P.n_items * P.nq;          // after delta / row normaliser
    float* cpart = dsp + (long long)P.nH * P.nq * P.nk;
    if (dbias || dhs) {
      const long long n = (long long)P.nH * P.nq * P.nk;
      mmn::attn_bias_grad_generic<T, DMAX><<<(unsigned)((n + kGenericThreads - 1) / kGenericThreads), kGenericThreads, 0, st>>>(
          P, (const T*)q, (const T*)k, (const T*)v, lse, (const T*)dout, ws, dbias, dhs ? dsp : nullptr);
      e = cudaGetLastError();
      if (e != cudaSuccess) return e;
      ++*launches;
      if (dhs && (e = reduce_partials(dsp, P.nq * P.nk, P.nH, dhs, st, launches)) != cudaSuccess) return e;
    }
    if (dcs) {                                                  // column sums of the dq, dk, dv just written
      const long long rows = tokens(P);
      const int C = P.nH * P.d;
      if ((e = colsum_det_any((const T*)dq, rows, C, P.dq_s0, dcs, cpart, st, launches)) != cudaSuccess) return e;
      if ((e = colsum_det_any((const T*)dk, rows, C, P.dk_s0, dcs + C, cpart, st, launches)) != cudaSuccess) return e;
      if ((e = colsum_det_any((const T*)dv, rows, C, P.dv_s0, dcs + 2 * C, cpart, st, launches)) != cudaSuccess) return e;
    }
    return cudaSuccess;
  }
  {
    mmn::GenericLaunch L = plan(P.nq, P.nk, 2 * P.d * 4 + 12);
    auto kern = mmn::attn_bwd_dq_generic<T, DMAX>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    dim3 grid((P.n_items + L.slots - 1) / L.slots, (P.nq + L.rows_per_slot - 1) / L.rows_per_slot);
    kern<<<grid, mmn::kGenericThreads, L.smem_bytes, st>>>(P, L, (const T*)q, (const T*)k, (const T*)v, lse,
                                                          (const T*)dout, (T*)dq, dbias, dhs, ws, dcs);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    ++*launches;
  }
  {
    mmn::GenericLaunch L = plan(P.nk, P.nq, 2 * P.d * 4 + 24);
    auto kern = mmn::attn_bwd_dkv_generic<T, DMAX>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    dim3 grid((P.n_items + L.slots - 1) / L.slots, (P.nk + L.rows_per_slot - 1) / L.rows_per_slot);
    kern<<<grid, mmn::kGenericThreads, L.smem_bytes, st>>>(P, L, (const T*)q, (const T*)k, (const T*)v, lse, ws,
                                                          (const T*)dout, (T*)dk, (T*)dv, dcs);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) ++*launches;
    return e;
  }
}

#define MMN_DISPATCH_D(T, FN, ...)                                            \
  do {                                                                         \
    if (P.d <= 4) return FN<T, 4>(__VA_ARGS__);                                \
    if (P.d <= 8) return FN<T, 8>(__VA_ARGS__);                                \
    if (P.d <= 16) return FN<T, 16>(__VA_ARGS__);                              \
    if (P.d <= 32) return FN<T, 32>(__VA_ARGS__);                              \
    if (P.d <= 64) return FN<T, 64>(__VA_ARGS__);                              \
    return FN<T, 128>(__VA_ARGS__);                                            \
  } while (0)

}  // namespace

cudaError_t generic_fwd(const GenericProblem& P, int dt, const void* q, const void* k, const void* v, void* out, float* lse,
                        cudaStream_t st, int* launches) {
  if (dt == MMN_DT_F32) MMN_DISPATCH_D(float, launch_fwd, P, q, k, v, out, lse, st, launches);
  MMN_DISPATCH_D(__nv_bfloat16, launch_fwd, P, q, k, v, out, lse, st, launches);
}

cudaError_t generic_bwd(const GenericProblem& P, int dt, const void* q, const void* k, const void* v, const float* lse,
                        const void* dout, void* dq, void* dk, void* dv, float* dbias, float* dhs, float* ws, float* dcs, bool det,
                        cudaStream_t st, int* launches) {
  if (dt == MMN_DT_F32) MMN_DISPATCH_D(float, launch_bwd, P, q, k, v, lse, dout, dq, dk, dv, dbias, dhs, ws, dcs, det, st, launches);
  MMN_DISPATCH_D(__nv_bfloat16, launch_bwd, P, q, k, v, lse, dout, dq, dk, dv, dbias, dhs, ws, dcs, det, st, launches);
}

size_t generic_bwd_workspace_floats(const GenericProblem& P, bool det) {
  size_t n = 2 * (size_t)P.n_items * P.nq;
  if (det) n += (size_t)P.nH * P.nq * P.nk + (size_t)colsum_any_blocks(tokens(P)) * P.nH * P.d;
  return n;
}

cudaError_t reduce_partials(const float* part, int nparts, long long n, float* out, cudaStream_t st, int* launches) {
  reduce_partials_kernel<<<(unsigned)((n + 31) / 32), kRedSlices * 32, 0, st>>>(part, nparts, n, out);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) ++*launches;
  return e;
}

cudaError_t generic_avg_weights(const GenericProblem& P, int dt, int batch, const void* q, const void* k, const float* lse,
                                float* avg, cudaStream_t st, int* launches) {
  long long total = (long long)batch * P.nq * P.nk;
  int blocks = (int)((total + 255) / 256);
  if (dt == MMN_DT_F32)
    mha_avg_weights_generic<float><<<blocks, 256, 0, st>>>(P, batch, (const float*)q, (const float*)k, lse, avg);
  else
    mha_avg_weights_generic<__nv_bfloat16><<<blocks, 256, 0, st>>>(P, batch, (const __nv_bfloat16*)q, (const __nv_bfloat16*)k, lse, avg);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) ++*launches;
  return e;
}

int colsum_blocks(long long rows, int cols) {
  const int rpb = 256 / (cols / 8);
  long long want = (rows + rpb - 1) / rpb;
  // four blocks per SM: with eight, the per-block flush (one atomic per column and block, all on the same few cache lines)
  // weighs more than the extra loads in flight help -- 10.0 -> 7.4 us at 110 592 x 96, 30.8 -> 25.7 us at x 384, equal at 8x the rows
  return (int)(want < 148 * 4 ? want : 148 * 4);
}

size_t colsum_workspace_floats(long long rows, int cols) { return rows > 0 ? (size_t)colsum_blocks(rows, cols) * cols : 0; }

cudaError_t colsum(int dt, const void* x, long long rows, int cols, long long row_stride, float* out, float* part, cudaStream_t st,
                   int* launches) {
  const int blocks = colsum_blocks(rows, cols);
  if (dt == MMN_DT_F32) colsum_kernel<float><<<blocks, 256, 0, st>>>((const float*)x, rows, cols, row_stride, out, part);
  else colsum_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)x, rows, cols, row_stride, out, part);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  ++*launches;
  return part ? reduce_partials(part, blocks, cols, out, st, launches) : cudaSuccess;
}

__global__ void zero_words_kernel(uint32_t* __restrict__ p, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = 0u;
}

cudaError_t zero_words_async(void* p, size_t words, cudaStream_t st) {
  if (words == 0) return cudaSuccess;
  const size_t want = (words + 255) / 256;
  zero_words_kernel<<<(unsigned)(want < 592 ? want : 592), 256, 0, st>>>(static_cast<uint32_t*>(p), words);
  return cudaGetLastError();
}

}  // namespace mmn


