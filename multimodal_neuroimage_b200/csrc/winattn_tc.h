// winattn_tc.h -- host entry points of the tcgen05 window-attention kernels (winattn_tc.cu).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include "../../include/mmn_b200.h"

namespace mmn { namespace tc {
// nullptr when the descriptor qualifies for the tensor-core path, else the reason it does not.
const char* fwd_why_not(const mmn_winattn_desc* d);
const char* bwd_why_not(const mmn_winattn_desc* d);
int winattn_fwd(const mmn_winattn_desc* d, const void* q, const void* k, const void* v, const float* bias,
                const float* head_scale, const float* mask, void* out, float* lse, void* workspace, cudaStream_t st, char* err,
                size_t errlen);
int winattn_bwd(const mmn_winattn_desc* d, const void* q, const void* k, const void* v, const float* bias,
                const float* head_scale, const float* mask, const void* out, const float* lse, const void* dout, void* dq,
                void* dk, void* dv, float* dbias, float* dhead_scale, float* dcolsum, float* workspace, cudaStream_t st,
                char* err, size_t errlen, int* launches);
// workspace of the deterministic backward (desc->deterministic != 0): one slot of partial sums per CTA
size_t bwd_det_workspace_bytes(const mmn_winattn_desc* d);
// fused projection backward (linbwd_tc.cu)
const char* linbwd_why_not(int io_dtype, long long rows, int in_features, int out_features, long long ld_dy, long long ld_x, long long ld_dx);
size_t linbwd_workspace_bytes(int out_features);
int linbwd(const void* dy, const void* x, const void* w, void* dx, float* dw, float* db, float* workspace, long long rows,
           int in_features, int out_features, long long ld_dy, long long ld_x, long long ld_dx, cudaStream_t st, char* err,
           size_t errlen, int* launches);
// tensor-core projections for any width that is a multiple of 32 (gemm_tc.cu)
const char* linear_why_not(int io_dtype, long long rows, int in_features, int out_features, long long ld_x, long long ld_y);
int linear_fwd(const void* x, const void* w, const float* bias, void* y, void* y_pre, int act, long long rows, int in_features,
               int out_features, long long ld_x, long long ld_y, cudaStream_t st, char* err, size_t errlen, int* launches);
size_t linear_wgrad_workspace_bytes(long long rows, int in_features, int out_features);
int linear_bwd_general(const void* dy, const void* x, const void* w, void* dx, float* dw, float* workspace, const void* aux, long long ld_aux,
                       int act_grad, long long rows, int in_features, int out_features, long long ld_dy, long long ld_x, long long ld_dx,
                       cudaStream_t st, char* err, size_t errlen, int* launches);
// cross-modal multi-head attention on the tensor cores (mha_tc.cu): bf16, head_dim 32 / 64, no attention dropout
const char* mha_why_not(const mmn_mha_desc* d, bool backward);
int mha_fwd(const mmn_mha_desc* d, const void* q, const void* k, const void* v, const float* mask, void* out, float* lse, cudaStream_t st,
            char* err, size_t errlen, int* launches);
int mha_bwd(const mmn_mha_desc* d, const void* q, const void* k, const void* v, const float* mask, const void* out, const float* lse,
            const void* dout, void* dq, void* dk, void* dv, float* workspace, cudaStream_t st, char* err, size_t errlen, int* launches);
}}  // namespace mmn::tc
