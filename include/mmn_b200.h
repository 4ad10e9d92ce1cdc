/* mmn_b200.h -- C ABI of libmmn_b200.so: the B200 (sm_100a) attention hot path of
 * Transconnectome/multimodal_neuroimage.
 *
 * The reference has no FFI/plugin interface for this path (it is pure PyTorch); the
 * boundary it exposes is the nn.Module API of modules/*.py.  The entry points below are
 * what a binding for that path binds, one per reference call site:
 *
 *   mmn_winattn_fwd / _bwd   replace, between `qkv = F.linear(x, ...)` and `self.proj(x)`:
 *       modules/swin_v2_module.py:149-175      (WindowAttention.forward, cosine + CPB bias)
 *       modules/swinfusion_module.py:121-142   (WindowAttention_fusion.forward)
 *       modules/swinfusion_module.py:221-243   (Cross_WindowAttention.forward)
 *     and, fused into the same kernel, the data movement of the enclosing blocks:
 *       torch.roll / window_partition / window_reverse / roll back
 *       modules/swin_v2_module.py:277-297, modules/swinfusion_module.py:350-373,497-530
 *       and the shift mask of swin_v2_module.py:244-266 (generated in-kernel).
 *   mmn_mha_fwd / _bwd       replace modules/multihead_attention.py:85-127
 *       (q*scaling, bmm, +attn_mask, softmax, dropout, bmm) incl. the future mask of
 *       modules/crossmodal_transformer.py:179-186 (generated in-kernel).
 *   mmn_mha_avg_weights      replaces modules/multihead_attention.py:131-133.
 *
 * Conventions: plain C structs, device pointers owned by the caller, the callee never
 * allocates or frees device memory, launches on the given stream of the given device and
 * never synchronises.  Return 0 on success, a negative MMN_ERR_* otherwise;
 * mmn_last_error() gives the thread-local message.  There is NO CPU path: every entry
 * point fails with MMN_ERR_CUDA when no CUDA device is usable.
 *
 * Deterministic mode.  By default the backward entry points accumulate cross-block sums (bias and scale gradients,
 * column sums, LayerNorm dgamma / dbeta, bias-table gradients) with float atomics, so their last bits can change from run
 * to run.  mmn_winattn_desc.deterministic, the `deterministic` arguments and the inverse bias index select kernels that
 * write per-block partial sums and add them in a fixed order instead: the same inputs then give bit-identical outputs
 * on one GPU model with one build (grid sizes follow the SM count, so not across GPU models).  Their workspace sizes
 * come from the *_workspace_bytes queries; with the flag off the queries return what the default kernels need.
 *
 * Token addressing.  A "token row" is num_heads*head_dim contiguous elements; row r of
 * head h of tensor X lives at  X + row_offset(r) + h*head_dim  (element units).
 *   window attention: tokens are indexed in the UN-windowed, UN-shifted (batch, grid...)
 *     order, row_offset = token * X_row_stride.  Packed qkv of shape (..., 3C) is passed
 *     as q = base, k = base + C, v = base + 2C with row stride 3C.
 *   multi-head attention: row (t, b) has row_offset = t*X_stride_t + b*X_stride_b.
 */
#ifndef MMN_B200_H_
#define MMN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMN_ABI_VERSION 5
/* scratch every window-attention launch needs: the tensor-core kernels keep the counters of their run-time work queue
 * there (zeroed by the library on the launch's stream; one buffer per launch, never shared between launches in flight) */
#define MMN_WINATTN_WORK_BYTES 2048

enum { MMN_OK = 0, MMN_ERR_INVALID = -1, MMN_ERR_UNSUPPORTED = -2, MMN_ERR_CUDA = -3 };
enum { MMN_DT_F32 = 0, MMN_DT_BF16 = 1 };
enum { MMN_SCORE_SCALED = 0,   /* s = (q*scale) . k            swinfusion_module.py:124-125 */
       MMN_SCORE_COSINE = 1 }; /* s = g_h * q^ . k^            swin_v2_module.py:153-156    */
enum { MMN_MASK_NONE = 0,
       MMN_MASK_SHIFT = 1,     /* {0,-100} region mask of the shifted frame, made in-kernel  */
       MMN_MASK_TENSOR = 2,    /* additive fp32 tensor: (mask_windows,N,N) or (T,S)          */
       MMN_MASK_FUTURE = 3 };  /* -inf where j - i >= mask_diagonal, made in-kernel          */
enum { MMN_PATH_AUTO = 0, MMN_PATH_GENERIC = 1, MMN_PATH_TCGEN05 = 2 };

typedef struct mmn_winattn_desc {
  int32_t ndim;            /* 1..3 spatial dims; unused trailing entries below are ignored   */
  int32_t batch;
  int32_t grid[3];         /* tokens per axis                                                 */
  int32_t window[3];       /* window extent per axis, divides grid                            */
  int32_t shift[3];        /* cyclic shift per axis, 0 <= shift < window                      */
  int32_t num_heads, head_dim;
  int32_t score_kind;      /* MMN_SCORE_*                                                     */
  int32_t mask_kind;       /* NONE | SHIFT | TENSOR                                           */
  int32_t mask_windows;    /* TENSOR: leading extent nW of the mask, window w uses w % nW     */
  int32_t io_dtype;        /* MMN_DT_*: dtype of q,k,v,out,dout,dq,dk,dv                      */
  int32_t path;            /* MMN_PATH_*; AUTO picks tcgen05 when the shape qualifies         */
  float scale;             /* SCALED: multiplier on q                                         */
  float dropout_p;         /* attention-probability dropout; 0 disables                       */
  uint64_t seed, offset;   /* Philox stream for dropout (same values in fwd and bwd)          */
  int64_t q_row_stride, k_row_stride, v_row_stride, o_row_stride;
  int64_t do_row_stride, dq_row_stride, dk_row_stride, dv_row_stride;   /* bwd only          */
  int32_t deterministic;   /* bwd: nonzero selects the fixed-order reductions (see above)     */
} mmn_winattn_desc;

typedef struct mmn_mha_desc {
  int32_t tgt_len, src_len, batch, num_heads, head_dim;
  int32_t mask_kind;       /* NONE | FUTURE | TENSOR                                          */
  int32_t mask_diagonal;   /* FUTURE: 1 + |S - T|   (crossmodal_transformer.py:183)           */
  int32_t io_dtype, path;
  float scale;             /* multiplier on q (head_dim^-0.5, multihead_attention.py:85)      */
  float dropout_p;
  uint64_t seed, offset;
  int64_t q_stride_t, q_stride_b, k_stride_t, k_stride_b, v_stride_t, v_stride_b;
  int64_t o_stride_t, o_stride_b;
  int64_t do_stride_t, do_stride_b, dq_stride_t, dq_stride_b, dk_stride_t, dk_stride_b;
  int64_t dv_stride_t, dv_stride_b;
} mmn_mha_desc;

int mmn_abi_version(void);
const char* mmn_last_error(void);
/* Name of the code path AUTO would take for this descriptor: "tcgen05" or "generic". */
const char* mmn_winattn_path(const mmn_winattn_desc* desc);
const char* mmn_mha_path(const mmn_mha_desc* desc);
/* Number of kernels this library has launched in the calling process (monotonic). */
uint64_t mmn_launch_count(void);

/* bias (num_heads,N,N) fp32 or NULL; head_scale (num_heads) fp32, COSINE only;
 * mask (mask_windows,N,N) fp32, TENSOR only; out: token rows; lse: FOUR slabs of batch*nW*num_heads*N fp32 --
 * [0] log-sum-exp (batch*nW, num_heads, N) by window position; [1..3] one record per window and head,
 * (batch*nW, num_heads, 3, N) = 1/max(||q||,eps) | 1/max(||k||,eps) | log2-domain lse in the kernel's tile row order,
 * written by the tensor-core forward kernel for mmn_winattn_bwd, which must be given the same buffer
 * (the generic kernels read and write slab 0 only).  `workspace`: MMN_WINATTN_WORK_BYTES of scratch owned by this
 * launch until it has completed, contents undefined on return. */
int mmn_winattn_fwd(const mmn_winattn_desc* desc, const void* q, const void* k, const void* v,
                    const float* bias, const float* head_scale, const float* mask,
                    void* out, float* lse, void* workspace, int device, void* stream);

/* dbias (num_heads,N,N) fp32 and dhead_scale (num_heads) fp32 are ACCUMULATED into (the
 * caller zeroes them); either may be NULL to skip.  `out` is the forward output (may be NULL:
 * the kernels recompute rowsum(P o dP) instead of reading it).  dcolsum (3, num_heads*head_dim) fp32,
 * ACCUMULATED, may be NULL: column sums over all tokens of dq, dk, dv -- the bias gradients of the
 * projections that produced q, k, v (replaces the reductions autograd does for F.linear's bias,
 * swin_v2_module.py:147-148, swinfusion_module.py:121,221-222).  `workspace`: scratch of
 * mmn_winattn_bwd_workspace_bytes(desc) bytes (16-byte aligned), owned by this launch until it has completed, contents
 * undefined on return.  With desc->deterministic == 0 that is max(2*batch*nW*num_heads*N floats, MMN_WINATTN_WORK_BYTES). */
size_t mmn_winattn_bwd_workspace_bytes(const mmn_winattn_desc* desc);
int mmn_winattn_bwd(const mmn_winattn_desc* desc, const void* q, const void* k, const void* v,
                    const float* bias, const float* head_scale, const float* mask,
                    const void* out, const float* lse, const void* dout,
                    void* dq, void* dk, void* dv, float* dbias, float* dhead_scale, float* dcolsum,
                    float* workspace, int device, void* stream);

/* mask (T,S) fp32, TENSOR only; out (T,B,E)-addressed rows; lse (batch*num_heads*T) fp32. */
int mmn_mha_fwd(const mmn_mha_desc* desc, const void* q, const void* k, const void* v,
                const float* mask, void* out, float* lse, int device, void* stream);

int mmn_mha_bwd(const mmn_mha_desc* desc, const void* q, const void* k, const void* v,
                const float* mask, const void* out, const float* lse, const void* dout,
                void* dq, void* dk, void* dv, float* workspace /* 2*batch*num_heads*roundup(T,128) floats */,
                int device, void* stream);

/* avg (batch,T,S) fp32 = mean over heads of the (dropped-out) attention probabilities. */
int mmn_mha_avg_weights(const mmn_mha_desc* desc, const void* q, const void* k, const float* mask,
                        const float* lse, float* avg, int device, void* stream);

/* out[c] += sum over rows of x[r*row_stride + c]: the bias gradient of the output projection
 * (F.linear backward, swin_v2_module.py:176) at memory speed.  cols % 8 == 0, cols <= 2048.
 * deterministic != 0: per-block partial sums in `workspace` (mmn_colsum_workspace_bytes(rows, cols) bytes), then a
 * fixed-order reduction; workspace may be NULL otherwise. */
size_t mmn_colsum_workspace_bytes(int64_t rows, int32_t cols);
int mmn_colsum(const void* x, int io_dtype, int64_t rows, int32_t cols, int64_t row_stride, float* out,
               float* workspace, int deterministic, int device, void* stream);

/* SwinV2 continuous relative-position bias (swin_v2_module.py:158-162), fp32:
 *   bias[h][e] = 16 sigmoid(tab[index[e]][h]),  tab[t][h] = sum_j w2[h][j] relu(w1[j] . coords[t] + b1[j])
 * coords (T, n_in) with n_in <= 3, w1 (J, n_in), b1 (J), w2 (nH, J) with nH <= 64, index (NN) int64 in [0, T).
 * fwd writes tab16 (T, nH) [= 16 sigmoid(tab), kept for the backward] and bias (nH, NN).
 * bwd: dbias (nH, NN) -> dw1 (J, n_in), db1 (J), dw2 (nH, J), all OVERWRITTEN; scratch (T, nH) floats.
 * inv_perm / inv_offsets: NULL, or the inverse of `index` in CSR form -- inv_perm (NN) int32 = the entries e in increasing
 * order of (index[e], e), inv_offsets (T + 1) int32 = where each table entry's run starts, inv_offsets[T] == NN.  Given,
 * the table gradient is a gather that sums each entry's dbias values in increasing e (deterministic); NULL, a scatter with
 * float atomics.  A kernel that finds inv_offsets[T] != NN writes NaN into its output.
 * T * nH <= 12288 (the backward stages d tab in shared memory); MMN_ERR_UNSUPPORTED otherwise. */
int mmn_cpb_bias_fwd(const float* coords, const float* w1, const float* b1, const float* w2, const int64_t* index,
                     int32_t T, int32_t n_in, int32_t J, int32_t num_heads, int32_t NN,
                     float* tab16, float* bias, int device, void* stream);
int mmn_cpb_bias_bwd(const float* coords, const float* w1, const float* b1, const float* w2, const int64_t* index,
                     const int32_t* inv_perm, const int32_t* inv_offsets,
                     const float* tab16, const float* dbias, int32_t T, int32_t n_in, int32_t J, int32_t num_heads, int32_t NN,
                     float* scratch, float* dw1, float* db1, float* dw2, int device, void* stream);

/* Learned relative-position bias table of the fusion blocks (swinfusion_module.py:58-60,127-130,228-231), fp32:
 *   fwd: bias[h][e] = table[index[e]][h]            table (T, nH), index (NN) int64 in [0, T), bias (nH, NN)
 *   bwd: dtable[t][h] = sum over e with index[e] == t of dbias[h][e]     (dtable OVERWRITTEN; float atomics, or with
 *        inv_perm / inv_offsets given a fixed-order gather: see mmn_cpb_bias_bwd)
 * i.e. `table[index].view(N, N, nH).permute(2, 0, 1).contiguous()` and its backward in one launch each (PyTorch: index_select +
 * permute copy forward, zeros + index_add backward). */
int mmn_table_bias_fwd(const float* table, const int64_t* index, int32_t T, int32_t num_heads, int32_t NN, float* bias,
                       int device, void* stream);
int mmn_table_bias_bwd(const float* dbias, const int64_t* index, const int32_t* inv_perm, const int32_t* inv_offsets, int32_t T,
                       int32_t num_heads, int32_t NN, float* dtable, int device, void* stream);

/* Projections on the tensor cores (csrc/gemm_tc.cu, csrc/linbwd_tc.cu).  They replace the F.linear calls of the path and
 * their autograd backward: swin_v2_module.py:148,176 (qkv, proj) and :27-31 (Mlp: fc1 -> GELU -> fc2),
 * swinfusion_module.py:121,143,221-222,244, crossmodal_transformer.py:158-160 (fc1 -> relu -> fc2).
 * bf16 operands, fp32 accumulation, in_features and out_features multiples of 32 (mmn_linear_supported tells; other shapes
 * -- the reference's own 12/24/48/84/168-wide layers -- are plain library GEMMs on the caller's side).
 *   forward:  y (rows, out) = act(x (rows, in) w^T + bias);  w is (out, in) row-major contiguous, bias (out) fp32 or NULL;
 *             y_pre (rows, out), optional, receives act'(x w^T + bias), the activation's DERIVATIVE at the pre-activation
 *             (GELU: Phi(v) + v phi(v); ReLU: 0 / 1) -- what the backward multiplies with, computed where exp(-v^2/2) is at hand;
 *             x has leading dimension ld_x, y and y_pre ld_y (elements).
 *   backward: dx (rows, in) = (dy w) o act_aux   -- act != NONE says the layer BELOW this one (whose output was this layer's
 *             input) had an activation; act_aux is the y_pre ITS forward wrote, (rows, in) with leading dimension ld_aux;
 *             dw (out, in) fp32 = dy^T x, OVERWRITTEN; db (out) fp32 = column sums of dy, OVERWRITTEN.  dx or dw may be NULL
 *             to skip that half (then db is skipped with dw == NULL only if db is NULL too).
 *             workspace: mmn_linear_bwd_workspace_bytes(rows, in, out, deterministic) bytes, contents undefined on return.
 *             deterministic != 0: db of the dgrad + wgrad path is summed in a fixed order (the fused pass always is).
 *             in = 96 and out in {96, 192, 288, 384} with no activation run as ONE pass over dy and x (linbwd_tc.cu). */
enum { MMN_ACT_NONE = 0, MMN_ACT_RELU = 1, MMN_ACT_GELU = 2 };
int mmn_linear_supported(int io_dtype, int64_t rows, int32_t in_features, int32_t out_features, int64_t ld_x, int64_t ld_y);
int mmn_linear_fwd(const void* x, const void* w, const float* bias, void* y, void* y_pre, int act, int io_dtype, int64_t rows,
                   int32_t in_features, int32_t out_features, int64_t ld_x, int64_t ld_y, int device, void* stream);
int mmn_linear_bwd_supported(int io_dtype, int64_t rows, int32_t in_features, int32_t out_features,
                             int64_t ld_dy, int64_t ld_x, int64_t ld_dx);
size_t mmn_linear_bwd_workspace_bytes(int64_t rows, int32_t in_features, int32_t out_features, int deterministic);
int mmn_linear_bwd(const void* dy, const void* x, const void* w, void* dx, float* dw, float* db, void* workspace,
                   const void* act_aux, int64_t ld_aux, int act, int io_dtype, int64_t rows, int32_t in_features,
                   int32_t out_features, int64_t ld_dy, int64_t ld_x, int64_t ld_dx, int deterministic, int device, void* stream);

/* LayerNorm fused with the residual add around it (csrc/layernorm.cu), one pass over the rows forward, one backward.
 * Replaces the norm + add (+ autocast cast) sequences of swin_v2_module.py:299,302 (res-post-norm),
 * swinfusion_module.py:345,377-378,491-492,535-539 (pre-norm) and crossmodal_transformer.py:143-165.  Per row of `cols`:
 *   MMN_LN_PRE :  s = resid + delta;                       out_sum = s,  out_norm = LN(s) * gamma + beta
 *   MMN_LN_POST:  s = resid + (LN(delta) * gamma + beta);  out_sum = s,  out_norm = s
 * resid or (PRE only) delta may be NULL (= 0), out_sum or out_norm may be NULL (skipped); each tensor is MMN_DT_F32 or
 * MMN_DT_BF16 on its own, rows contiguous; gamma / beta (cols) fp32, beta may be NULL; mean / rstd (rows) fp32 are written
 * for the backward.  cols even and <= 1536.
 * Backward: g_sum / g_norm = gradients w.r.t. out_sum / out_norm (either may be NULL), x = the normalised quantity (PRE: s,
 * i.e. out_sum or the lone input; POST: delta).  d_resid / d_delta may be NULL.  dgamma / dbeta (cols) fp32 are ACCUMULATED
 * into (the caller zeroes them); either may be NULL.  By default each block adds its column sums with atomics;
 * deterministic != 0 has each block write them to `workspace` (mmn_layernorm_bwd_workspace_bytes(rows, cols) bytes) and
 * adds them in block order.  workspace may be NULL otherwise. */
enum { MMN_LN_PRE = 0, MMN_LN_POST = 1 };
int mmn_layernorm_supported(int32_t cols);
int mmn_layernorm_fwd(const void* resid, int resid_dtype, const void* delta, int delta_dtype, const float* gamma, const float* beta,
                      float eps, int mode, void* out_sum, int sum_dtype, void* out_norm, int norm_dtype, float* mean, float* rstd,
                      int64_t rows, int32_t cols, int device, void* stream);
size_t mmn_layernorm_bwd_workspace_bytes(int64_t rows, int32_t cols);
int mmn_layernorm_bwd(const void* g_sum, int gs_dtype, const void* g_norm, int gn_dtype, const void* x, int x_dtype,
                      const float* gamma, const float* mean, const float* rstd, int mode, void* d_resid, int dr_dtype,
                      void* d_delta, int dd_dtype, float* dgamma, float* dbeta, float* workspace, int deterministic,
                      int64_t rows, int32_t cols, int device, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MMN_B200_H_ */
