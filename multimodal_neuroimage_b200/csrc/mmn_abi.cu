// mmn_abi.cu -- the extern "C" surface declared in include/mmn_b200.h.
// Validates descriptors, picks a code path (tcgen05 tensor-core kernels for the tuned
// bf16 shapes, the generic fp32-arithmetic kernels for everything else) and launches on
// the caller's stream.  No ATen / pybind here: plain pointers and sizes only.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "../../include/mmn_b200.h"
#include "generic_launch.h"
#include "zero_fill.h"
#include "winattn_tc.h"

namespace {

thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

struct DeviceGuard {
  int prev = -1;
  bool ok = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); return; }
    if (dev != prev && cudaSetDevice(dev) != cudaSuccess) { cudaGetLastError(); return; }
    ok = true;
  }
  ~DeviceGuard() { if (ok && prev >= 0) cudaSetDevice(prev); }
};

int finish(cudaError_t e, int launches, const char* what) {
  g_launches.fetch_add((uint64_t)launches, std::memory_order_relaxed);
  if (e != cudaSuccess) return fail(MMN_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  return MMN_OK;
}

int validate_win(const mmn_winattn_desc* d) {
  if (!d) return fail(MMN_ERR_INVALID, "null descriptor");
  if (d->ndim < 1 || d->ndim > 3) return fail(MMN_ERR_INVALID, "ndim %d not in 1..3", d->ndim);
  if (d->batch < 1 || d->num_heads < 1 || d->head_dim < 1) return fail(MMN_ERR_INVALID, "batch/heads/head_dim must be positive");
  for (int a = 0; a < d->ndim; ++a) {
    if (d->window[a] < 1 || d->grid[a] < 1 || d->grid[a] % d->window[a] != 0)
      return fail(MMN_ERR_INVALID, "axis %d: window %d does not divide grid %d", a, d->window[a], d->grid[a]);
    if (d->shift[a] < 0 || d->shift[a] >= d->window[a])
      return fail(MMN_ERR_INVALID, "axis %d: shift %d not in [0, window %d)", a, d->shift[a], d->window[a]);
  }
  if (d->score_kind != MMN_SCORE_SCALED && d->score_kind != MMN_SCORE_COSINE) return fail(MMN_ERR_INVALID, "bad score_kind");
  if (d->mask_kind != MMN_MASK_NONE && d->mask_kind != MMN_MASK_SHIFT && d->mask_kind != MMN_MASK_TENSOR)
    return fail(MMN_ERR_INVALID, "bad mask_kind %d for window attention", d->mask_kind);
  if (d->mask_kind == MMN_MASK_TENSOR && d->mask_windows < 1) return fail(MMN_ERR_INVALID, "mask_windows must be >= 1");
  if (d->io_dtype != MMN_DT_F32 && d->io_dtype != MMN_DT_BF16) return fail(MMN_ERR_INVALID, "bad io_dtype");
  if (d->dropout_p < 0.f || d->dropout_p >= 1.f) return fail(MMN_ERR_INVALID, "dropout_p must be in [0,1)");
  if (d->head_dim > 128) return fail(MMN_ERR_UNSUPPORTED, "head_dim %d > 128", d->head_dim);
  return MMN_OK;
}

int validate_mha(const mmn_mha_desc* d) {
  if (!d) return fail(MMN_ERR_INVALID, "null descriptor");
  if (d->tgt_len < 1 || d->src_len < 1 || d->batch < 1 || d->num_heads < 1 || d->head_dim < 1)
    return fail(MMN_ERR_INVALID, "sizes must be positive");
  if (d->mask_kind != MMN_MASK_NONE && d->mask_kind != MMN_MASK_FUTURE && d->mask_kind != MMN_MASK_TENSOR)
    return fail(MMN_ERR_INVALID, "bad mask_kind %d for multi-head attention", d->mask_kind);
  if (d->io_dtype != MMN_DT_F32 && d->io_dtype != MMN_DT_BF16) return fail(MMN_ERR_INVALID, "bad io_dtype");
  if (d->dropout_p < 0.f || d->dropout_p >= 1.f) return fail(MMN_ERR_INVALID, "dropout_p must be in [0,1)");
  if (d->head_dim > 128) return fail(MMN_ERR_UNSUPPORTED, "head_dim %d > 128", d->head_dim);
  return MMN_OK;
}

mmn::GenericProblem problem_from(const mmn_winattn_desc* d, const float* bias, const float* head_scale, const float* mask) {
  mmn::GenericProblem P{};
  P.kind = 0;
  for (int a = 0; a < 3; ++a) { P.grid[a] = 1; P.win[a] = 1; P.shift[a] = 0; P.nwin[a] = 1; }
  for (int a = 0; a < d->ndim; ++a) {          // right-align the used axes
    int t = 3 - d->ndim + a;
    P.grid[t] = d->grid[a]; P.win[t] = d->window[a]; P.shift[t] = d->shift[a]; P.nwin[t] = d->grid[a] / d->window[a];
  }
  P.nW = P.nwin[0] * P.nwin[1] * P.nwin[2];
  P.nq = P.nk = P.win[0] * P.win[1] * P.win[2];
  P.d = d->head_dim; P.nH = d->num_heads;
  P.n_items = d->batch * P.nW * P.nH;
  P.q_s0 = d->q_row_stride; P.k_s0 = d->k_row_stride; P.v_s0 = d->v_row_stride; P.o_s0 = d->o_row_stride;
  P.do_s0 = d->do_row_stride; P.dq_s0 = d->dq_row_stride; P.dk_s0 = d->dk_row_stride; P.dv_s0 = d->dv_row_stride;
  P.cosine = d->score_kind == MMN_SCORE_COSINE;
  P.mask_kind = d->mask_kind; P.mask_windows = d->mask_windows > 0 ? d->mask_windows : 1;
  P.scale = d->scale; P.dropout_p = d->dropout_p; P.seed = d->seed; P.offset = d->offset;
  P.drop = mmn::make_dropout(d->dropout_p, d->seed, d->offset);
  P.rng = reinterpret_cast<const unsigned long long*>(d->rng);
  P.bias = bias; P.head_scale = head_scale; P.mask = mask;
  return P;
}

mmn::GenericProblem problem_from(const mmn_mha_desc* d, const float* mask) {
  mmn::GenericProblem P{};
  P.kind = 1;
  for (int a = 0; a < 3; ++a) { P.grid[a] = 1; P.win[a] = 1; P.shift[a] = 0; P.nwin[a] = 1; }
  P.nW = 1;
  P.nq = d->tgt_len; P.nk = d->src_len; P.d = d->head_dim; P.nH = d->num_heads;
  P.n_items = d->batch * d->num_heads;
  P.q_s0 = d->q_stride_t; P.q_s1 = d->q_stride_b; P.k_s0 = d->k_stride_t; P.k_s1 = d->k_stride_b;
  P.v_s0 = d->v_stride_t; P.v_s1 = d->v_stride_b; P.o_s0 = d->o_stride_t; P.o_s1 = d->o_stride_b;
  P.do_s0 = d->do_stride_t; P.do_s1 = d->do_stride_b; P.dq_s0 = d->dq_stride_t; P.dq_s1 = d->dq_stride_b;
  P.dk_s0 = d->dk_stride_t; P.dk_s1 = d->dk_stride_b; P.dv_s0 = d->dv_stride_t; P.dv_s1 = d->dv_stride_b;
  P.cosine = 0;
  P.mask_kind = d->mask_kind; P.mask_diag = d->mask_diagonal; P.mask_windows = 1;
  P.scale = d->scale; P.dropout_p = d->dropout_p; P.seed = d->seed; P.offset = d->offset;
  P.drop = mmn::make_dropout(d->dropout_p, d->seed, d->offset);
  P.rng = reinterpret_cast<const unsigned long long*>(d->rng);
  P.mask = mask;
  return P;
}

bool have_device() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return false; }
  return n > 0;
}

}  // namespace

extern "C" {

int mmn_abi_version(void) { return MMN_ABI_VERSION; }
const char* mmn_last_error(void) { return g_err; }
uint64_t mmn_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

const char* mmn_winattn_path(const mmn_winattn_desc* d) {
  if (validate_win(d) != MMN_OK) return "invalid";
  if (d->path == MMN_PATH_GENERIC) return "generic";
  return mmn::tc::fwd_why_not(d) == nullptr ? "tcgen05" : "generic";
}

const char* mmn_mha_path(const mmn_mha_desc* d) {
  if (validate_mha(d) != MMN_OK) return "invalid";
  if (d->path == MMN_PATH_GENERIC) return "generic";
  return mmn::tc::mha_why_not(d, false) == nullptr ? "tcgen05" : "generic";
}

int mmn_winattn_fwd(const mmn_winattn_desc* d, const void* q, const void* k, const void* v, const float* bias,
                    const float* head_scale, const float* mask, void* out, float* lse, void* workspace, int device,
                    void* stream) {
  int rc = validate_win(d);
  if (rc) return rc;
  if (!q || !k || !v || !out || !lse || !workspace) return fail(MMN_ERR_INVALID, "null tensor pointer");
  if (d->score_kind == MMN_SCORE_COSINE && !head_scale) return fail(MMN_ERR_INVALID, "cosine attention needs head_scale");
  if (d->mask_kind == MMN_MASK_TENSOR && !mask) return fail(MMN_ERR_INVALID, "MMN_MASK_TENSOR needs a mask");
  if (!have_device()) return fail(MMN_ERR_CUDA, "no CUDA device: libmmn_b200 has no CPU path");
  DeviceGuard g(device);
  if (!g.ok) return fail(MMN_ERR_CUDA, "cannot select device %d", device);
  cudaStream_t st = (cudaStream_t)stream;
  const char* why = mmn::tc::fwd_why_not(d);
  bool tc_ok = why == nullptr;
  if (d->path == MMN_PATH_TCGEN05 && !tc_ok) return fail(MMN_ERR_UNSUPPORTED, "shape not supported by the tcgen05 path: %s", why);
  if (d->path != MMN_PATH_GENERIC && tc_ok) {
    rc = mmn::tc::winattn_fwd(d, q, k, v, bias, head_scale, mask, out, lse, workspace, st, g_err, sizeof(g_err));
    if (rc == MMN_OK) g_launches.fetch_add(1, std::memory_order_relaxed);
    return rc;
  }
  int n = 0;
  cudaError_t e = mmn::generic_fwd(problem_from(d, bias, head_scale, mask), d->io_dtype, q, k, v, out, lse, st, &n);
  return finish(e, n, "attn_fwd_generic");
}

const char* mmn_winattn_qkv_path(const mmn_winattn_desc* d, int in_channels) {
  if (validate_win(d) != MMN_OK) return "invalid";
  if (d->path == MMN_PATH_GENERIC) return "generic path requested";
  const char* why = mmn::tc::qkv_fwd_why_not(d, in_channels);
  return why ? why : "tcgen05-fused";
}

int mmn_winattn_qkv_fwd(const mmn_winattn_desc* d, const void* x, const void* w_qkv, const float* b_qkv, const float* bias,
                        const float* head_scale, const float* mask, void* qkv_out, void* out, float* lse, void* workspace,
                        int device, void* stream) {
  int rc = validate_win(d);
  if (rc) return rc;
  if (!x || !w_qkv || !qkv_out || !out || !lse || !workspace) return fail(MMN_ERR_INVALID, "null tensor pointer");
  if (d->score_kind == MMN_SCORE_COSINE && !head_scale) return fail(MMN_ERR_INVALID, "cosine attention needs head_scale");
  if (d->mask_kind == MMN_MASK_TENSOR && !mask) return fail(MMN_ERR_INVALID, "MMN_MASK_TENSOR needs a mask");
  if (!have_device()) return fail(MMN_ERR_CUDA, "no CUDA device: libmmn_b200 has no CPU path");
  if (d->path == MMN_PATH_GENERIC) return fail(MMN_ERR_UNSUPPORTED, "the fused qkv forward has no generic path");
  if (const char* why = mmn::tc::qkv_fwd_why_not(d, d->num_heads * d->head_dim))
    return fail(MMN_ERR_UNSUPPORTED, "shape not supported by the fused qkv forward: %s", why);
  DeviceGuard g(device);
  if (!g.ok) return fail(MMN_ERR_CUDA, "cannot select device %d", device);
  rc = mmn::tc::winattn_qkv_fwd(d, x, w_qkv, b_qkv, bias, head_scale, mask, qkv_out, out, lse, workspace, (cudaStream_t)stream,
                                g_err, sizeof(g_err));
  if (rc == MMN_OK) g_launches.fetch_add(1, std::memory_order_relaxed);
  return rc;
}

size_t mmn_winattn_bwd_workspace_bytes(const mmn_winattn_desc* d) {
  if (validate_win(d) != MMN_OK) return 0;
  const mmn::GenericProblem P = problem_from(d, nullptr, nullptr, nullptr);
  const size_t base = mmn::generic_bwd_workspace_floats(P, false) * sizeof(float);
  size_t bytes = base > MMN_WINATTN_WORK_BYTES ? base : MMN_WINATTN_WORK_BYTES;
  if (!d->deterministic) return bytes;
  const size_t det = d->path != MMN_PATH_GENERIC && mmn::tc::bwd_why_not(d) == nullptr ? mmn::tc::bwd_det_workspace_bytes(d)
                                                                                      : mmn::generic_bwd_workspace_floats(P, true) * sizeof(float);
  return det > bytes ? det : bytes;
}

int mmn_winattn_bwd(const mmn_winattn_desc* d, const void* q, const void* k, const void* v, const float* bias,
                    const float* head_scale, const float* mask, const void* out, const float* lse, const void* dout,
                    void* dq, void* dk, void* dv, float* dbias, float* dhead_scale, float* dcolsum, float* workspace,
                    int device, void* stream) {
  int rc = validate_win(d);
  if (rc) return rc;
  if (!q || !k || !v || !lse || !dout || !dq || !dk || !dv || !workspace) return fail(MMN_ERR_INVALID, "null tensor pointer");
  if (d->score_kind == MMN_SCORE_COSINE && !head_scale) return fail(MMN_ERR_INVALID, "cosine attention needs head_scale");
  if (d->mask_kind == MMN_MASK_TENSOR && !mask) return fail(MMN_ERR_INVALID, "MMN_MASK_TENSOR needs a mask");
  if (!have_device()) return fail(MMN_ERR_CUDA, "no CUDA device: libmmn_b200 has no CPU path");
  DeviceGuard g(device);
  if (!g.ok) return fail(MMN_ERR_CUDA, "cannot select device %d", device);
  cudaStream_t st = (cudaStream_t)stream;
  const char* why = mmn::tc::bwd_why_not(d);
  bool tc_ok = why == nullptr;
  if (d->path == MMN_PATH_TCGEN05 && !tc_ok) return fail(MMN_ERR_UNSUPPORTED, "shape not supported by the tcgen05 backward path: %s", why);
  if (d->path != MMN_PATH_GENERIC && tc_ok) {
    int n = 0;
    rc = mmn::tc::winattn_bwd(d, q, k, v, bias, head_scale, mask, out, lse, dout, dq, dk, dv, dbias, dhead_scale, dcolsum, workspace, st, g_err, sizeof(g_err), &n);
    g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed);
    return rc;
  }
  mmn::GenericProblem P = problem_from(d, bias, head_scale, mask);
  int n = 0;
  cudaError_t e = mmn::generic_bwd(P, d->io_dtype, q, k, v, lse, dout, dq, dk, dv, bias ? dbias : nullptr,
                                 P.cosine ? dhead_scale : nullptr, workspace, dcolsum, d->deterministic != 0, st, &n);
  return finish(e, n, "attn_bwd_generic");
}

int mmn_mha_fwd(const mmn_mha_desc* d, const void* q, const void* k, const void* v, const float* mask, void* out,
                float* lse, int device, void* stream) {
  int rc = validate_mha(d);
  if (rc) return rc;
  if (!q || !k || !v || !out || !lse) return fail(MMN_ERR_INVALID, "null tensor pointer");
  if (d->mask_kind == MMN_MASK_TENSOR && !mask) return fail(MMN_ERR_INVALID, "MMN_MASK_TENSOR needs a mask");
  if (!have_device()) return fail(MMN_ERR_CUDA, "no CUDA device: libmmn_b200 has no CPU path");
  DeviceGuard g(device);
  if (!g.ok) return fail(MMN_ERR_CUDA, "cannot select device %d", device);
  int n = 0;
  const char* why = mmn::tc::mha_why_not(d, false);
  if (d->path == MMN_PATH_TCGEN05 && why) return fail(MMN_ERR_UNSUPPORTED, "shape not supported by the tcgen05 MHA path: %s", why);
  if (d->path != MMN_PATH_GENERIC && !why) {
    rc = mmn::tc::mha_fwd(d, q, k, v, mask, out, lse, (cudaStream_t)stream, g_err, sizeof(g_err), &n);
    g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed);
    return rc;
  }
  cudaError_t e = mmn::generic_fwd(problem_from(d, mask), d->io_dtype, q, k, v, out, lse, (cudaStream_t)stream, &n);
  return finish(e, n, "attn_fwd_generic");
}

int mmn_mha_bwd(const mmn_mha_desc* d, const void* q, const void* k, const void* v, const float* mask, const void* out,
                const float* lse, const void* dout, void* dq, void* dk, void* dv, float* workspace, int device,
                void* stream) {
  int rc = validate_mha(d);
  if (rc) return rc;
  if (!q || !k || !v || !lse || !dout || !dq || !dk || !dv || !workspace) return fail(MMN_ERR_INVALID, "null tensor pointer");
  if (d->mask_kind == MMN_MASK_TENSOR && !mask) return fail(MMN_ERR_INVALID, "MMN_MASK_TENSOR needs a mask");
  if (!have_device()) return fail(MMN_ERR_CUDA, "no CUDA device: libmmn_b200 has no CPU path");
  DeviceGuard g(device);
  if (!g.ok) return fail(MMN_ERR_CUDA, "cannot select device %d", device);
  int n = 0;
  const char* why = mmn::tc::mha_why_not(d, true);
  if (d->path == MMN_PATH_TCGEN05 && why) return fail(MMN_ERR_UNSUPPORTED, "shape not supported by the tcgen05 MHA backward path: %s", why);
  if (d->path != MMN_PATH_GENERIC && !why) {
    rc = mmn::tc::mha_bwd(d, q, k, v, mask, out, lse, dout, dq, dk, dv, workspace, (cudaStream_t)stream, g_err, sizeof(g_err), &n);
    g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed);
    return rc;
  }
  cudaError_t e = mmn::generic_bwd(problem_from(d, mask), d->io_dtype, q, k, v, lse, dout, dq, dk, dv, nullptr, nullptr, workspace,
                                 nullptr, false, (cudaStream_t)stream, &n);
  return finish(e, n, "attn_bwd_generic");
}

int mmn_mha_avg_weights(const mmn_mha_desc* d, const void* q, const void* k, const float* mask, const float* lse,
                        float* avg, int device, void* stream) {
  int rc = validate_mha(d);
  if (rc) return rc;
  if (!q || !k || !lse || !avg) return fail(MMN_ERR_INVALID, "null tensor pointer");
  if (!have_device()) return fail(MMN_ERR_CUDA, "no CUDA device: libmmn_b200 has no CPU path");
  DeviceGuard g(device);
  if (!g.ok) return fail(MMN_ERR_CUDA, "cannot select device %d", device);
  int n = 0;
  cudaError_t e = mmn::generic_avg_weights(problem_from(d, mask), d->io_dtype, d->batch, q, k, lse, avg, (cudaStream_t)stream, &n);
  return finish(e, n, "mha_avg_weights_generic");
}

size_t mmn_colsum_workspace_bytes(int64_t rows, int32_t cols) {
  if (rows < 1 || cols < 8 || cols % 8 != 0 || cols > 2048) return 0;
  return mmn::colsum_workspace_floats(rows, cols) * sizeof(float);
}

int mmn_colsum(const void* x, int io_dtype, int64_t rows, int32_t cols, int64_t row_stride, float* out, float* workspace,
               int deterministic, int device, void* stream) {
  if (!x || !out || rows < 0 || cols < 1) return fail(MMN_ERR_INVALID, "bad colsum arguments");
  if (deterministic && !workspace) return fail(MMN_ERR_INVALID, "deterministic colsum needs a workspace");
  if (io_dtype != MMN_DT_F32 && io_dtype != MMN_DT_BF16) return fail(MMN_ERR_INVALID, "bad io_dtype");
  if (cols % 8 != 0 || cols > 2048) return fail(MMN_ERR_UNSUPPORTED, "colsum needs cols %% 8 == 0 and cols <= 2048 (got %d)", cols);
  if (!have_device()) return fail(MMN_ERR_CUDA, "no CUDA device: libmmn_b200 has no CPU path");
  DeviceGuard g(device);
  if (!g.ok) return fail(MMN_ERR_CUDA, "cannot select device %d", device);
  if (rows == 0) return MMN_OK;
  int n = 0;
  cudaError_t e = mmn::colsum(io_dtype, x, rows, cols, row_stride, out, deterministic ? workspace : nullptr, (cudaStream_t)stream, &n);
  return finish(e, n, "colsum_kernel");
}

static int cpb_check(int T, int n_in, int J, int nH, int NN) {
  if (T < 1 || n_in < 1 || n_in > 3 || J < 1 || nH < 1 || nH > 64 || NN < 1) return fail(MMN_ERR_INVALID, "bad cpb_bias sizes");
  if ((long long)T * nH > 12288) return fail(MMN_ERR_UNSUPPORTED, "cpb_bias: T * num_heads = %lld > 12288", (long long)T * nH);
  if (mmn::cpb_bwd_smem_bytes(T) > 227 * 1024) return fail(MMN_ERR_UNSUPPORTED, "cpb_bias: table of %d entries exceeds the backward kernel's shared memory", T);
  if (!have_device()) return fail(MMN_ERR_CUDA, "no CUDA device: libmmn_b200 has no CPU path");
  return MMN_OK;
}

int mmn_table_bias_fwd(const float* table, const int64_t* index, int32_t T, int32_t nH, int32_t NN, float* bias, int device, void* stream) {
  if (!table || !index || !bias) return fail(MMN_ERR_INVALID, "null tensor pointer");
  if (T < 1 || nH < 1 || NN < 1) return fail(MMN_ERR_INVALID, "bad bias table dimensions");
  if (!have_device()) return fail(MMN_ERR_CUDA, "no CUDA device: libmmn_b200 has no CPU path");
  DeviceGuard g(device);
  if (!g.ok) return fail(MMN_ERR_CUDA, "cannot select device %d", device);
  int n = 0;
  cudaError_t e = mmn::table_bias_fwd(table, (const long long*)index, nH, NN, bias, (cudaStream_t)stream, &n);
  return finish(e, n, "table_bias_fwd");
}

int mmn_table_bias_bwd(const float* dbias, const int64_t* index, const int32_t* inv_perm, const int32_t* inv_offsets, int32_t T, int32_t nH,
                       int32_t NN, float* dtable, int device, void* stream) {
  if (!dbias || !index || !dtable) return fail(MMN_ERR_INVALID, "null tensor pointer");
  if (!inv_perm != !inv_offsets) return fail(MMN_ERR_INVALID, "inv_perm and inv_offsets go together");
  if (T < 1 || nH < 1 || NN < 1) return fail(MMN_ERR_INVALID, "bad bias table dimensions");
  if (!have_device()) return fail(MMN_ERR_CUDA, "no CUDA device: libmmn_b200 has no CPU path");
  DeviceGuard g(device);
  if (!g.ok) return fail(MMN_ERR_CUDA, "cannot select device %d", device);
  int n = 0;
  cudaError_t e = mmn::table_bias_bwd(dbias, (const long long*)index, inv_perm, inv_offsets, T, nH, NN, dtable, (cudaStream_t)stream, &n);
  return finish(e, n, "table_bias_bwd");
}

int mmn_cpb_bias_fwd(const float* coords, const float* w1, const float* b1, const float* w2, const int64_t* index, int32_t T,
                     int32_t n_in, int32_t J, int32_t nH, int32_t NN, float* tab16, float* bias, int device, void* stream) {
  if (!coords || !w1 || !b1 || !w2 || !index || !tab16 || !bias) return fail(MMN_ERR_INVALID, "null tensor pointer");
  int rc = cpb_check(T, n_in, J, nH, NN);
  if (rc) return rc;
  DeviceGuard g(device);
  if (!g.ok) return fail(MMN_ERR_CUDA, "cannot select device %d", device);
  int n = 0;
  cudaError_t e = mmn::cpb_bias_fwd(coords, w1, b1, w2, (const long long*)index, T, n_in, J, nH, NN, tab16, bias, (cudaStream_t)stream, &n);
  return finish(e, n, "cpb_bias_fwd");
}

int mmn_cpb_bias_bwd(const float* coords, const float* w1, const float* b1, const float* w2, const int64_t* index,
                     const int32_t* inv_perm, const int32_t* inv_offsets,
                     const float* tab16, const float* dbias, int32_t T, int32_t n_in, int32_t J, int32_t nH, int32_t NN,
                     float* scratch, float* dw1, float* db1, float* dw2, int device, void* stream) {
  if (!coords || !w1 || !b1 || !w2 || !index || !tab16 || !dbias || !scratch || !dw1 || !db1 || !dw2)
    return fail(MMN_ERR_INVALID, "null tensor pointer");
  if (!inv_perm != !inv_offsets) return fail(MMN_ERR_INVALID, "inv_perm and inv_offsets go together");
  int rc = cpb_check(T, n_in, J, nH, NN);
  if (rc) return rc;
  DeviceGuard g(device);
  if (!g.ok) return fail(MMN_ERR_CUDA, "cannot select device %d", device);
  int n = 0;
  cudaError_t e = mmn::cpb_bias_bwd(coords, w1, b1, w2, (const long long*)index, inv_perm, inv_offsets, tab16, dbias, T, n_in, J, nH, NN,
                                    scratch, dw1, db1, dw2, (cudaStream_t)stream, &n);
  return finish(e, n, "cpb_bias_bwd");
}

int mmn_linear_supported(int io_dtype, int64_t rows, int32_t in_features, int32_t out_features, int64_t ld_x, int64_t ld_y) {
  return have_device() && mmn::tc::linear_why_not(io_dtype, rows, in_features, out_features, ld_x, ld_y) == nullptr;
}

int mmn_linear_fwd(const void* x, const void* w, const float* bias, void* y, void* y_pre, int act, int io_dtype, int64_t rows,
                   int32_t in_features, int32_t out_features, int64_t ld_x, int64_t ld_y, int device, void* stream) {
  if (!x || !w || !y) return fail(MMN_ERR_INVALID, "null tensor pointer");
  if (act != MMN_ACT_NONE && act != MMN_ACT_RELU && act != MMN_ACT_GELU) return fail(MMN_ERR_INVALID, "bad activation %d", act);
  if (y_pre && act == MMN_ACT_NONE) return fail(MMN_ERR_INVALID, "y_pre only makes sense with an activation");
  if (!have_device()) return fail(MMN_ERR_CUDA, "no CUDA device: libmmn_b200 has no CPU path");
  const char* why = mmn::tc::linear_why_not(io_dtype, rows, in_features, out_features, ld_x, ld_y);
  if (why) return fail(MMN_ERR_UNSUPPORTED, "shape not supported by the tensor-core projection: %s", why);
  DeviceGuard g(device);
  if (!g.ok) return fail(MMN_ERR_CUDA, "cannot select device %d", device);
  int n = 0;
  int rc = mmn::tc::linear_fwd(x, w, bias, y, y_pre, act, rows, in_features, out_features, ld_x, ld_y, (cudaStream_t)stream, g_err,
                               sizeof(g_err), &n);
  g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed);
  return rc;
}

// in = 96, out in {96, 192, 288, 384}: ONE pass over dy and x (linbwd_tc.cu); any other multiple of 32: dgrad + wgrad (gemm_tc.cu)
static bool linbwd_fused_ok(int io_dtype, int64_t rows, int32_t in_features, int32_t out_features, int64_t ld_dy, int64_t ld_x,
                            int64_t ld_dx) {
  return mmn::tc::linbwd_why_not(io_dtype, rows, in_features, out_features, ld_dy, ld_x, ld_dx) == nullptr;
}

int mmn_linear_bwd_supported(int io_dtype, int64_t rows, int32_t in_features, int32_t out_features, int64_t ld_dy, int64_t ld_x,
                             int64_t ld_dx) {
  if (!have_device()) return 0;
  if (linbwd_fused_ok(io_dtype, rows, in_features, out_features, ld_dy, ld_x, ld_dx)) return 1;
  return mmn::tc::linear_why_not(io_dtype, rows, in_features, out_features, ld_x, ld_dy) == nullptr && ld_dx % 8 == 0;
}

// Deterministic mode reuses the workspace for db's column-sum partials once the weight gradient (stream-ordered before them)
// is done with it.
size_t mmn_linear_bwd_workspace_bytes(int64_t rows, int32_t in_features, int32_t out_features, int deterministic) {
  const size_t a = mmn::tc::linbwd_workspace_bytes(out_features);
  const size_t b = mmn::tc::linear_wgrad_workspace_bytes(rows, in_features, out_features);
  size_t bytes = a > b ? a : b;
  if (deterministic && rows > 0 && out_features >= 8) {
    const size_t c = mmn::colsum_workspace_floats(rows, out_features < 2048 ? out_features : 2048) * sizeof(float);
    if (c > bytes) bytes = c;
  }
  return bytes;
}

int mmn_linear_bwd(const void* dy, const void* x, const void* w, void* dx, float* dw, float* db, void* workspace,
                   const void* act_aux, int64_t ld_aux, int act, int io_dtype, int64_t rows, int32_t in_features,
                   int32_t out_features, int64_t ld_dy, int64_t ld_x, int64_t ld_dx, int deterministic, int device, void* stream) {
  if (!dy || !w || !workspace || (!dx && !dw)) return fail(MMN_ERR_INVALID, "null tensor pointer");
  if (dw && !x) return fail(MMN_ERR_INVALID, "dw needs x");
  if (act != MMN_ACT_NONE && act != MMN_ACT_RELU && act != MMN_ACT_GELU) return fail(MMN_ERR_INVALID, "bad activation %d", act);
  if (act != MMN_ACT_NONE && (!act_aux || ld_aux % 8 || reinterpret_cast<uintptr_t>(act_aux) % 16))
    return fail(MMN_ERR_INVALID, "activation gradient needs a 16-byte aligned act'(pre) tensor");
  if (!have_device()) return fail(MMN_ERR_CUDA, "no CUDA device: libmmn_b200 has no CPU path");
  if (!mmn_linear_bwd_supported(io_dtype, rows, in_features, out_features, ld_dy, ld_x ? ld_x : in_features, ld_dx ? ld_dx : in_features))
    return fail(MMN_ERR_UNSUPPORTED, "shape not supported by the tensor-core projection backward (bf16, widths multiples of 32)");
  DeviceGuard g(device);
  if (!g.ok) return fail(MMN_ERR_CUDA, "cannot select device %d", device);
  cudaStream_t st = (cudaStream_t)stream;
  int n = 0, rc;
  if (dx && dw && act == MMN_ACT_NONE && linbwd_fused_ok(io_dtype, rows, in_features, out_features, ld_dy, ld_x, ld_dx)) {
    rc = mmn::tc::linbwd(dy, x, w, dx, dw, db, (float*)workspace, rows, in_features, out_features, ld_dy, ld_x, ld_dx, st, g_err,
                         sizeof(g_err), &n);
  } else {
    rc = mmn::tc::linear_bwd_general(dy, x, w, dx, dw, (float*)workspace, act_aux, ld_aux,
                                     act != MMN_ACT_NONE ? 3 : 0, rows, in_features, out_features, ld_dy,
                                     ld_x, ld_dx, st, g_err, sizeof(g_err), &n);
    if (rc == MMN_OK && db) {
      // bias gradient: column sums of dy, 2048 columns per launch (colsum_kernel's block covers 256 x 8)
      cudaError_t e = mmn::zero_words_async(db, (size_t)out_features, st);
      for (int c0 = 0; e == cudaSuccess && c0 < out_features; c0 += 2048)
        e = mmn::colsum(MMN_DT_BF16, static_cast<const uint16_t*>(dy) + c0, rows, out_features - c0 < 2048 ? out_features - c0 : 2048, ld_dy,
                        db + c0, deterministic ? static_cast<float*>(workspace) : nullptr, st, &n);
      if (e != cudaSuccess) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); return finish(e, 0, "colsum_kernel"); }
    }
  }
  g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed);
  return rc;
}

int mmn_layernorm_supported(int32_t cols) { return have_device() && mmn::layernorm_supported(cols); }

static bool ln_dt_ok(int dt) { return dt == MMN_DT_F32 || dt == MMN_DT_BF16; }

int mmn_layernorm_fwd(const void* resid, int resid_dtype, const void* delta, int delta_dtype, const float* gamma, const float* beta,
                      float eps, int mode, void* out_sum, int sum_dtype, void* out_norm, int norm_dtype, float* mean, float* rstd,
                      int64_t rows, int32_t cols, int device, void* stream) {
  if ((!resid && !delta) || !gamma || !mean || !rstd || (!out_sum && !out_norm)) return fail(MMN_ERR_INVALID, "null tensor pointer");
  if (mode != MMN_LN_PRE && mode != MMN_LN_POST) return fail(MMN_ERR_INVALID, "bad layernorm mode %d", mode);
  if (mode == MMN_LN_POST && !delta) return fail(MMN_ERR_INVALID, "MMN_LN_POST normalises delta: it cannot be null");
  if (!ln_dt_ok(resid_dtype) || !ln_dt_ok(delta_dtype) || !ln_dt_ok(sum_dtype) || !ln_dt_ok(norm_dtype)) return fail(MMN_ERR_INVALID, "bad dtype");
  if (rows < 0) return fail(MMN_ERR_INVALID, "negative row count");
  if (!mmn::layernorm_supported(cols)) return fail(MMN_ERR_UNSUPPORTED, "layernorm: cols = %d (even, <= 1536)", cols);
  if (!have_device()) return fail(MMN_ERR_CUDA, "no CUDA device: libmmn_b200 has no CPU path");
  DeviceGuard g(device);
  if (!g.ok) return fail(MMN_ERR_CUDA, "cannot select device %d", device);
  if (rows == 0) return MMN_OK;
  int n = 0;
  cudaError_t e = mmn::layernorm_fwd(resid, resid_dtype, delta, delta_dtype, gamma, beta, eps, mode, out_sum, sum_dtype, out_norm, norm_dtype,
                                     mean, rstd, rows, cols, (cudaStream_t)stream, &n);
  return finish(e, n, "layernorm_fwd_kernel");
}

size_t mmn_layernorm_bwd_workspace_bytes(int64_t rows, int32_t cols) {
  if (rows < 1 || !mmn::layernorm_supported(cols)) return 0;
  return mmn::layernorm_bwd_workspace_floats(rows, cols) * sizeof(float);
}

int mmn_layernorm_bwd(const void* g_sum, int gs_dtype, const void* g_norm, int gn_dtype, const void* x, int x_dtype, const float* gamma,
                      const float* mean, const float* rstd, int mode, void* d_resid, int dr_dtype, void* d_delta, int dd_dtype,
                      float* dgamma, float* dbeta, float* workspace, int deterministic, int64_t rows, int32_t cols, int device,
                      void* stream) {
  if ((!g_sum && !g_norm) || !x || !gamma || !mean || !rstd) return fail(MMN_ERR_INVALID, "null tensor pointer");
  if (deterministic && (dgamma || dbeta) && !workspace) return fail(MMN_ERR_INVALID, "deterministic layernorm backward needs a workspace");
  if (mode != MMN_LN_PRE && mode != MMN_LN_POST) return fail(MMN_ERR_INVALID, "bad layernorm mode %d", mode);
  if (!ln_dt_ok(gs_dtype) || !ln_dt_ok(gn_dtype) || !ln_dt_ok(x_dtype) || !ln_dt_ok(dr_dtype) || !ln_dt_ok(dd_dtype)) return fail(MMN_ERR_INVALID, "bad dtype");
  if (!mmn::layernorm_supported(cols)) return fail(MMN_ERR_UNSUPPORTED, "layernorm: cols = %d (even, <= 1536)", cols);
  if (!have_device()) return fail(MMN_ERR_CUDA, "no CUDA device: libmmn_b200 has no CPU path");
  DeviceGuard g(device);
  if (!g.ok) return fail(MMN_ERR_CUDA, "cannot select device %d", device);
  if (rows <= 0) return MMN_OK;
  int n = 0;
  cudaError_t e = mmn::layernorm_bwd(g_sum, gs_dtype, g_norm, gn_dtype, x, x_dtype, gamma, mean, rstd, mode, d_resid, dr_dtype, d_delta,
                                     dd_dtype, dgamma, dbeta, deterministic ? workspace : nullptr, rows, cols, (cudaStream_t)stream, &n);
  return finish(e, n, "layernorm_bwd_kernel");
}

}  // extern "C"
