// generic_launch.h -- host entry points of the shape-generic kernels (attn_generic.cuh),
// compiled in their own translation unit so that the tensor-core kernels rebuild quickly.
#pragma once
#include <cuda_runtime.h>
#include "attn_generic.cuh"

namespace mmn {
// Each returns cudaSuccess or the launch error; `*launches` is incremented per kernel launched.
cudaError_t generic_fwd(const GenericProblem& P, int io_dtype, const void* q, const void* k, const void* v, void* out,
                        float* lse, cudaStream_t st, int* launches);
cudaError_t generic_bwd(const GenericProblem& P, int io_dtype, const void* q, const void* k, const void* v, const float* lse,
                        const void* dout, void* dq, void* dk, void* dv, float* dbias, float* dhs, float* ws, float* dcolsum,
                        bool deterministic, cudaStream_t st, int* launches);
// floats of `ws` generic_bwd needs: the row statistics, plus in deterministic mode the partial sums
size_t generic_bwd_workspace_floats(const GenericProblem& P, bool deterministic);
// out[e] += sum over s < nparts of part[s * n + e] in a fixed order (deterministic mode's second pass)
cudaError_t reduce_partials(const float* part, int nparts, long long n, float* out, cudaStream_t st, int* launches);
cudaError_t generic_avg_weights(const GenericProblem& P, int io_dtype, int batch, const void* q, const void* k,
                                const float* lse, float* avg, cudaStream_t st, int* launches);
// part: null (float atomics into out) or colsum_workspace_floats(rows, cols) floats (per-block partials + fixed-order reduce)
cudaError_t colsum(int io_dtype, const void* x, long long rows, int cols, long long row_stride, float* out, float* part, cudaStream_t st,
                   int* launches);
size_t colsum_workspace_floats(long long rows, int cols);
// continuous relative-position bias (cpb_bias.cu)
size_t cpb_bwd_smem_bytes(int T);
cudaError_t table_bias_fwd(const float* table, const long long* index, int nH, int NN, float* bias, cudaStream_t st, int* launches);
cudaError_t table_bias_bwd(const float* dbias, const long long* index, const int* inv_perm, const int* inv_offsets, int T, int nH, int NN,
                           float* dtable, cudaStream_t st, int* launches);
cudaError_t cpb_bias_fwd(const float* coords, const float* w1, const float* b1, const float* w2, const long long* index, int T,
                         int n_in, int J, int nH, int NN, float* tab16, float* bias, cudaStream_t st, int* launches);
cudaError_t cpb_bias_bwd(const float* coords, const float* w1, const float* b1, const float* w2, const long long* index,
                         const int* inv_perm, const int* inv_offsets, const float* tab16, const float* dbias, int T, int n_in, int J, int nH, int NN, float* dtab16, float* dw1,
                         float* db1, float* dw2, cudaStream_t st, int* launches);
// LayerNorm fused with the residual add around it (layernorm.cu)
bool layernorm_supported(int cols);
cudaError_t layernorm_fwd(const void* resid, int resid_dt, const void* delta, int delta_dt, const float* gamma, const float* beta,
                          float eps, int mode, void* out_sum, int sum_dt, void* out_norm, int norm_dt, float* mean, float* rstd,
                          long long rows, int cols, cudaStream_t st, int* launches);
cudaError_t layernorm_bwd(const void* g_sum, int gs_dt, const void* g_norm, int gn_dt, const void* x, int x_dt, const float* gamma,
                          const float* mean, const float* rstd, int mode, void* d_resid, int dr_dt, void* d_delta, int dd_dt,
                          float* dgamma, float* dbeta, float* part, long long rows, int cols, cudaStream_t st, int* launches);
// floats of the deterministic LayerNorm backward's per-block partials (an upper bound over its kernels)
size_t layernorm_bwd_workspace_floats(long long rows, int cols);
}  // namespace mmn
