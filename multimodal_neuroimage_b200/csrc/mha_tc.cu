// mha_tc.cu -- cross-modal multi-head attention (modules/multihead_attention.py:85-127: q*scaling, bmm, + attn_mask, fp32
// softmax, bmm) on the Blackwell tensor cores, flash style: nothing T x S ever reaches HBM.
//
// Tuned shapes: bf16, head_dim 32 or 64, any T / S / batch / heads, masks NONE / FUTURE (generated from indices,
// crossmodal_transformer.py:179-186) / TENSOR ((T,S) additive fp32), attention dropout (multihead_attention.py:123; DROP
// instantiations: the mask is regenerated from (seed, offset, item, t, s) by every kernel, dropout_rng.cuh).  q, k, v, out are addressed in place in the reference's
// (len, batch, embed) layout (row strides from the descriptor: q/k/v may be column slices of one packed projection), through
// 4-D tensor maps (element-in-panel, row, 32-channel panel, batch) whose boxes land as 64B-swizzled [panel][128 rows][64 B]
// tiles -- the K-major operand of Q K^T and, read transposed (MN-major), the operand of P V, dS^T Q, P^T dO and dS K alike.
//
//   forward   CTA = (128 queries, head, batch); K/V tiles of 128 keys stream through a 2-stage ring.  Per key tile:
//             S = Q K^T (tcgen05, TMEM) -> one thread per query row: online softmax in fp32 (two passes over the TMEM tile:
//             max, then exp2 / sum), P (bf16) back into TMEM as the A operand of P V; the tile's P V lands in its own TMEM
//             columns and is folded into the row's output in REGISTERS (O = O * alpha + PV) -- no TMEM rescale pass.
//             Two CTAs per SM (256 TMEM columns, 80 KB of shared memory each) overlap one's softmax with the other's MMAs.
//   backward  two kernels, both recompute S and dP = dO V^T per 128 x 128 block and form P = exp2(s - lse),
//             dS = P o (dP - delta) * scale in registers -> bf16 tiles in shared memory:
//               mode dKdV: CTA = (128 keys, head, batch), query tiles stream;  dV += P^T dO,  dK += dS^T Q   (TMEM)
//               mode dQ  : CTA = (128 queries, head, batch), key tiles stream; dQ += dS K                    (TMEM)
//             delta = rowsum(dO o O) comes from a small pre-pass.  No atomics: deterministic.
#include <algorithm>
#include <cstdio>
#include <mutex>

#include "dropout_rng.cuh"
#include "tc_window.cuh"
#include "winattn_tc.h"

namespace mmn { namespace tc {

constexpr float kMLog2e = 1.4426950408889634f;
constexpr float kMLn2 = 0.6931471805599453f;
// 12 warps: 8 compute warps (two warpgroups), then a warpgroup holding the TMA producer (warp 8) and the MMA issuer (warp 9).
// Launched at 168 registers per thread; the compute warpgroups take 216 (a thread holds a whole row of logits), the third 72.
constexpr int kMThreads = 384;
constexpr int kMRegCompute = 216, kMRegAux = 72;   // 256 x 216 + 128 x 72 = 384 x 168: the launch allocation is the pool
constexpr int kMStagesF = 4;                   // forward: K / V ring
constexpr int kMStagesB = 4;                   // backward: streamed-tile ring
constexpr int kMComputeWarpsB = 16, kMThreadsB = (kMComputeWarpsB + 2) * 32;   // backward: + TMA producer + MMA issuer
constexpr float kMRescaleTau = 8.f;            // forward: the running maximum is only raised when it grows by more than 2^tau

struct MhaParams {
  CUtensorMap q, k, v, dout;                   // 4-D maps (32, rows, E / 32, batch); box (32, 128, D / 32, 1)
  int T, S, B, nH;
  int mask_kind, mask_diag;
  float scale;
  const float* mask;                           // (T, S) additive, MMN_MASK_TENSOR
  __nv_bfloat16* out; long long o_st, o_sb;    // forward output rows (t, b): out + t * o_st + b * o_sb + h * D
  float* lse;                                  // (B * nH, T) natural-log log-sum-exp
  DropoutCfg drop;                             // attention dropout (dropout_rng.cuh); thr == 0: none
  const unsigned long long* rng;               // null, or device {seed, offset} replacing drop's stream (dropout_at_entry)
  const float* rowdata; int Tpad;              // backward: (B * nH, Tpad / 2, 4) per query pair {-lse2, -lse2, -delta scale, -delta scale}
  __nv_bfloat16 *dq, *dk, *dv;                 // backward outputs
  long long dq_st, dq_sb, dk_st, dk_sb, dv_st, dv_sb;
};

// number of key tiles a query tile starting at t0 can see / first query tile that sees key tile j (FUTURE mask:
// key s is visible to query t iff s - t < diag)
__device__ __forceinline__ int visible_key_tiles(const MhaParams& P, int t0) {
  const int nkt = (P.S + 127) >> 7;
  if (P.mask_kind != MMN_MASK_FUTURE) return nkt;
  const long long last = (long long)t0 + 127 + P.mask_diag - 1;          // largest visible key index of the tile's last row
  if (last < 0) return 0;
  return (int)min((long long)nkt, (last >> 7) + 1);
}
__device__ __forceinline__ int first_query_tile(const MhaParams& P, int s0) {
  if (P.mask_kind != MMN_MASK_FUTURE) return 0;
  const long long t_min = (long long)s0 - P.mask_diag + 1;               // smallest t with s0 - t < diag
  return t_min <= 0 ? 0 : (int)(t_min >> 7);
}

// additive mask term (log2 domain) for logit (t, s); -inf outside the valid / visible range
__device__ __forceinline__ float mask_term(const MhaParams& P, int t, int s) {
  if (s >= P.S) return -INFINITY;
  if (P.mask_kind == MMN_MASK_FUTURE) return (s - t >= P.mask_diag) ? -INFINITY : 0.f;
  if (P.mask_kind == MMN_MASK_TENSOR) return t < P.T ? __ldg(P.mask + (long long)t * P.S + s) * kMLog2e : 0.f;
  return 0.f;
}
__device__ __forceinline__ bool tile_needs_mask(const MhaParams& P, int t0, int s0) {
  if (s0 + 128 > P.S || P.mask_kind == MMN_MASK_TENSOR) return true;
  if (P.mask_kind == MMN_MASK_FUTURE) return (s0 + 127) - t0 >= P.mask_diag;   // some (t, s) of the block is masked
  return false;
}

__device__ __forceinline__ float fmax3(float a, float b, float c) {       // sm_100: one FMNMX3
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

// exp2 of an fp32 pair WITHOUT the special-function unit: round-to-nearest split x = i + f through the 1.5 * 2^23 magic
// add, a cubic for 2^f on [-0.5, 0.5] (relative error <= 7.5e-5, fifty times below the bf16 rounding the probabilities get
// as MMA operands), and i added into the exponent field.  MUFU (16 lanes per clock and SM) is what bounds these kernels:
// 128 x 128 exponentials per block are 1024 cycles of it.  MMN_MHA_POLY_FWD / _BWD of every 8 pairs take this route on the FMA pipe
// (packed fp32x2 arithmetic) instead, so both pipes work on the exponentials at once.
#ifndef MMN_MHA_POLY_FWD
#define MMN_MHA_POLY_FWD 3
#endif
#ifndef MMN_MHA_POLY_BWD
#define MMN_MHA_POLY_BWD 0
#endif
__device__ __forceinline__ void exp2_poly_pair(uint64_t x2, float& e0, float& e1) {
  float x0, x1;
  upk2(x2, x0, x1);
  const uint64_t xc = pk2(fmaxf(x0, -126.f), fmaxf(x1, -126.f));          // also catches -inf (masked logits)
  const uint64_t t2 = add2(xc, pk2(12582912.f, 12582912.f));              // low mantissa bits = round(x)
  const uint64_t r2 = add2(t2, pk2(-12582912.f, -12582912.f));
  const uint64_t f2 = fma2(r2, pk2(-1.f, -1.f), xc);
  uint64_t p2 = fma2(f2, pk2(0.0551716685f, 0.0551716685f), pk2(0.2426111251f, 0.2426111251f));
  p2 = fma2(p2, f2, pk2(0.6932609677f, 0.6932609677f));
  p2 = fma2(p2, f2, pk2(0.9999280572f, 0.9999280572f));
  float p0, p1, t0, t1;
  upk2(p2, p0, p1);
  upk2(t2, t0, t1);
  e0 = __uint_as_float(__float_as_uint(p0) + (__float_as_uint(t0) << 23));
  e1 = __uint_as_float(__float_as_uint(p1) + (__float_as_uint(t1) << 23));
}
// exp2 of the pair x2; `e` is the pair's (compile-time) index: which unit computes it
template <int POLY_OF8>
__device__ __forceinline__ void exp2_pair(uint64_t x2, int e, float& e0, float& e1) {
  if ((e & 7) < POLY_OF8) {
    exp2_poly_pair(x2, e0, e1);
  } else {
    upk2(x2, e0, e1);
    e0 = fast_exp2(e0); e1 = fast_exp2(e1);
  }
}

// ------------------------------------------------------------------------------------------
// Forward
// ------------------------------------------------------------------------------------------
// CTA = (256 queries = two 128-row tiles, head, batch), one CTA per SM.  Compute warpgroup g owns query tile g: its own
// S / P / O columns in TMEM (S 128 | P 64 | O D, at column 256 g) and its own barriers, so the two tiles are two independent
// streams over the SAME K / V tiles (loaded once for both: half the L2 -> SM traffic of one tile per CTA), and while one
// stream's threads are in their exp2 phase (MUFU-bound: 128 exp2 per row and key tile) the other's MMAs and bookkeeping run.
// Per key tile a thread (= one query row) loads its 128 logits into registers in ONE pass and hands the S buffer back at
// once -- Q K^T of the next key tile is issued while this one's exponentials are computed.  O accumulates in TMEM over all
// key tiles (the MMA's accumulate flag); it is rescaled only when a row's maximum grows by more than 2^tau since the last
// rescale (P then stays <= 2^tau, exact in fp32 / fine in bf16), which after the first key tiles practically never happens.
template <int D, bool DROP>
__global__ void __launch_bounds__(kMThreads, 1)
mha_fwd_tc_kernel(const __grid_constant__ MhaParams P) {
  constexpr int kTileB = D * 256;                       // 128 rows x D bf16
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sQ = smem;                                   // [2]
  uint8_t* sK = sQ + 2 * kTileB;                        // [kMStagesF]
  uint8_t* sV = sK + kMStagesF * kTileB;                // [kMStagesF]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + kMStagesF * kTileB);
  uint64_t* q_full = bars;
  uint64_t* full = bars + 1;                            // [kMStagesF]
  uint64_t* empty = full + kMStagesF;                   // [kMStagesF]
  uint64_t* s_full = empty + kMStagesF;                 // [2] S(j) of stream g is in TMEM
  uint64_t* s_free = s_full + 2;                        // [2] ... and in the rows' registers (4 warp arrivals)
  uint64_t* p_ready = s_full + 4;                       // [2] P(j) is in TMEM, O has been rescaled if it had to be (4 warp arrivals)
  uint64_t* pv_done = s_full + 6;                       // [2] P V(j) has completed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_full + 8);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int t0 = blockIdx.x * 256, h = blockIdx.y, b = blockIdx.z;
  const DropoutCfg drop = DROP ? dropout_at_entry(P.drop, P.rng) : P.drop;
  int n_g[2];
#pragma unroll
  for (int g = 0; g < 2; ++g) n_g[g] = t0 + g * 128 < P.T ? visible_key_tiles(P, t0 + g * 128) : 0;
  const int n_max = max(n_g[0], n_g[1]);
  const bool two = t0 + 128 < P.T;

  if (tid == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < kMStagesF; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int g = 0; g < 2; ++g) { mbar_init(&s_full[g], 1); mbar_init(&s_free[g], 4); mbar_init(&p_ready[g], 4); mbar_init(&pv_done[g], 1); }
    fence_barrier_init();
  }
  if (warp == 8 && lane == 0) { tma_prefetch_desc(&P.q); tma_prefetch_desc(&P.k); tma_prefetch_desc(&P.v); }
  if (warp == 9) tmem_alloc<512>(tmem_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp >= 8) {
    setmaxnreg_dec<kMRegAux>();
    if (warp == 8) {
      if (elect_one() && n_max > 0) {
        mbar_arrive_expect_tx(q_full, (two ? 2 : 1) * kTileB);
        tma_load_4d(&P.q, q_full, sQ, 0, t0, h * (D / 32), b);
        if (two) tma_load_4d(&P.q, q_full, sQ + kTileB, 0, t0 + 128, h * (D / 32), b);
        for (int j = 0; j < n_max; ++j) {
          const int s = j % kMStagesF;
          mbar_wait(&empty[s], ((j / kMStagesF) & 1) ^ 1);
          mbar_arrive_expect_tx(&full[s], 2 * kTileB);
          tma_load_4d(&P.k, &full[s], sK + s * kTileB, 0, j * 128, h * (D / 32), b);
          tma_load_4d(&P.v, &full[s], sV + s * kTileB, 0, j * 128, h * (D / 32), b);
        }
      }
    } else if (warp == 9) {
      constexpr uint32_t idescS = umma_idesc_bf16(128, 128, 0, 0);
      constexpr uint32_t idescPV = umma_idesc_bf16(128, D, 0, 1);
      const uint64_t dK = umma_smem_desc(0, 0, 512, kSwz64);            // K-major tiles (Q, K)
      const uint64_t dVm = umma_smem_desc(0, 8192, 512, kSwz64);        // V read MN-major: channel panels 8 KB apart
      const uint32_t q0 = smem_u32(sQ) >> 4, k0 = smem_u32(sK) >> 4, v0 = smem_u32(sV) >> 4;
      auto issue_S = [&](int g, int j) {
        const int s = j % kMStagesF;
        if (elect_one()) {
#pragma unroll
          for (int ks = 0; ks < D / 16; ++ks) {
            const uint32_t o = (ks >> 1) * (8192 >> 4) + (ks & 1) * 2;
            umma_bf16_ss(tmem + g * 256, dK + (q0 + g * (kTileB >> 4) + o), dK + (k0 + s * (kTileB >> 4) + o), idescS, ks > 0 ? 1u : 0u);
          }
          umma_commit(&s_full[g]);
        }
        __syncwarp();
      };
      if (n_max > 0) {
        mbar_wait(q_full, 0);
        mbar_wait(&full[0], 0);
        tcgen05_fence_after();
#pragma unroll
        for (int g = 0; g < 2; ++g)
          if (n_g[g] > 0) issue_S(g, 0);
      }
      // Four queues served in turn, none blocking another: S_g(j + 1) goes out as soon as stream g's rows hold S_g(j) in
      // registers (s_free) and K(j + 1) has landed -- it then runs under the exponentials of tile j -- and P V_g(j) as
      // soon as P_g(j) is in TMEM.  (Waiting for P_g(j) before issuing S_g(j + 1) left the rows without logits for ~30 %
      // of their time.)  A K / V stage is released once both streams' P V of its tile have been issued.
      int ns[2] = {1, 1}, np[2] = {0, 0}, released = 0;
      uint32_t idle = 0;
      while (np[0] < n_g[0] || np[1] < n_g[1]) {
        bool progressed = false;
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          if (ns[g] < n_g[g]) {
            const int j = ns[g];                       // S_g(j): needs K(j) and the S buffer back from tile j - 1
            if (mbar_test(&full[j % kMStagesF], (j / kMStagesF) & 1) && mbar_test(&s_free[g], (j - 1) & 1)) {
              tcgen05_fence_after();
              issue_S(g, j);
              ++ns[g];
              progressed = true;
            }
          }
          if (np[g] < n_g[g] && np[g] < ns[g] && mbar_test(&p_ready[g], np[g] & 1)) {
            const int j = np[g], s = j % kMStagesF;
            tcgen05_fence_after();
            if (elect_one()) {
              const uint32_t tP = tmem + g * 256 + 128, tO = tmem + g * 256 + 192;
#pragma unroll
              for (int ks = 0; ks < 8; ++ks)          // 16 keys = 8 TMEM columns of P per step
                umma_bf16_ts(tO, tP + ks * 8, dVm + (v0 + s * (kTileB >> 4) + ks * 64), idescPV, (j > 0 || ks > 0) ? 1u : 0u);
              umma_commit(&pv_done[g]);
            }
            __syncwarp();
            ++np[g];
            progressed = true;
          }
        }
        // tile `released` is done with once every stream that sees it has had its P V issued (S of that tile went out before)
        while (released < n_max && (np[0] > released || released >= n_g[0]) && (np[1] > released || released >= n_g[1])) {
          if (elect_one()) umma_commit(&empty[released % kMStagesF]);
          __syncwarp();
          ++released;
        }
        if (progressed) idle = 0;
        else if (++idle > (1u << 26)) __trap();       // a broken pipeline becomes a CUDA error, not a hang
      }
    }
  } else {
    // ============================== softmax: warpgroup = query tile, thread = query row ==============================
    setmaxnreg_inc<kMRegCompute>();
    const int g = warp >> 2, r = tid & 127;
    const int tg0 = t0 + g * 128, t = tg0 + r;
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t tS = tmem + g * 256 + lane_base, tP = tS + 128, tO = tS + 192;
    const int n_tiles = n_g[g];
    const float sc = P.scale * kMLog2e;
    float m_use = -INFINITY, l = 0.f;
    for (int j = 0; j < n_tiles; ++j) {
      const int s0 = j * 128;
      const bool masked = tile_needs_mask(P, tg0, s0);
      mbar_wait(&s_full[g], j & 1);
      tcgen05_fence_after();
      uint32_t v[128];
      {
        uint32_t (*v32)[32] = reinterpret_cast<uint32_t (*)[32]>(v);
        tmem_ld_32x32b_x32(tS, v32[0]); tmem_ld_32x32b_x32(tS + 32, v32[1]);
        tmem_ld_32x32b_x32(tS + 64, v32[2]); tmem_ld_32x32b_x32(tS + 96, v32[3]);
        tmem_ld_wait();
      }
      tcgen05_fence_before();
      mbar_arrive_warp(&s_free[g]);
      float a_mul = sc;                               // logit (log2 domain) = v * a_mul
      if (masked) {                                   // the diagonal / ragged tiles of a row block, outside the main path
        if (P.mask_kind == MMN_MASK_TENSOR) {         // an additive mask tensor: fold scale and mask into v
#pragma unroll
          for (int e = 0; e < 128; ++e) v[e] = __float_as_uint(fmaf(__uint_as_float(v[e]), sc, mask_term(P, t, s0 + e)));
          a_mul = 1.f;
        } else {
          // future mask and / or the ragged last key tile: the row sees the keys e < e_lim of this tile.  One compare and
          // one select per logit (the general form above is ~25 instructions per logit: a diagonal tile cost 3.5 tiles).
          int e_lim = P.S - s0;
          if (P.mask_kind == MMN_MASK_FUTURE) e_lim = min(e_lim, t + P.mask_diag - s0);
#pragma unroll
          for (int e = 0; e < 128; ++e) v[e] = e < e_lim ? v[e] : 0xff800000u;      // -inf survives the positive scale
        }
      }
      // row maximum: a tree of three-input maxima (the scale is positive, so it commutes with the maximum)
      float mx;
      {
        float m3[43];
#pragma unroll
        for (int e = 0; e < 42; ++e) m3[e] = fmax3(__uint_as_float(v[3 * e]), __uint_as_float(v[3 * e + 1]), __uint_as_float(v[3 * e + 2]));
        m3[42] = fmaxf(__uint_as_float(v[126]), __uint_as_float(v[127]));
#pragma unroll
        for (int e = 0; e < 14; ++e) m3[e] = fmax3(m3[3 * e], m3[3 * e + 1], m3[3 * e + 2]);
        m3[14] = m3[42];
#pragma unroll
        for (int e = 0; e < 5; ++e) m3[e] = fmax3(m3[3 * e], m3[3 * e + 1], m3[3 * e + 2]);
        mx = fmaxf(fmax3(m3[0], m3[1], m3[2]), fmaxf(m3[3], m3[4]));
      }
      const float m_new = fmaxf(m_use, mx * a_mul);
      bool pv_waited = false;
      if (__any_sync(0xffffffffu, m_new > m_use + kMRescaleTau)) {
        // raise the maximum of every row of this warp (rows that would not have had to are rescaled for free)
        const float alpha = m_new == -INFINITY ? 1.f : fast_exp2(m_use - m_new);     // m_use = -inf: 0
        l *= alpha;
        m_use = m_new;
        if (j > 0) {                                  // O holds P V of tiles < j: wait for the last of them, rescale in place
          mbar_wait(&pv_done[g], (j - 1) & 1);
          tcgen05_fence_after();
          pv_waited = true;
#pragma unroll
          for (int c = 0; c < D / 16; ++c) {
            uint32_t o[16];
            tmem_ld_32x32b_x16(tO + c * 16, o);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 16; ++e) o[e] = __float_as_uint(__uint_as_float(o[e]) * alpha);
            tmem_st_32x32b_x16(tO + c * 16, o);
          }
        }
      }
      const float m_eff = m_use == -INFINITY ? 0.f : m_use;
      // P = exp2(v * a_mul - m) -> bf16 pairs, row sum
      const uint64_t a2 = pk2(a_mul, a_mul), nm2 = pk2(-m_eff, -m_eff);
      uint64_t rs2[2] = {0ull, 0ull};
      uint32_t pk[64];
#pragma unroll
      for (int e = 0; e < 64; ++e) {
        float x0, x1;
        exp2_pair<MMN_MHA_POLY_FWD>(fma2(pk2u(v[2 * e], v[2 * e + 1]), a2, nm2), e, x0, x1);
        rs2[e & 1] = add2(rs2[e & 1], pk2(x0, x1));
        if (DROP) {                                   // dropped probabilities leave the row sum untouched, not P V; 1 / (1 - p) is folded into 1 / l
          const uint4 rr = dropout_block(drop, b * P.nH + h, t >> 1, (s0 >> 1) + e);
          if (!dropout_keep_word((t & 1) ? rr.z : rr.x, drop.thr)) x0 = 0.f;
          if (!dropout_keep_word((t & 1) ? rr.w : rr.y, drop.thr)) x1 = 0.f;
        }
        pk[e] = pack_bf16x2(x0, x1);
      }
      if (j > 0 && !pv_waited) {                      // P V(j - 1) has read the P buffer
        mbar_wait(&pv_done[g], (j - 1) & 1);
        tcgen05_fence_after();
      }
      {
        uint32_t (*p16)[16] = reinterpret_cast<uint32_t (*)[16]>(pk);
        tmem_st_32x32b_x16(tP, p16[0]); tmem_st_32x32b_x16(tP + 16, p16[1]);
        tmem_st_32x32b_x16(tP + 32, p16[2]); tmem_st_32x32b_x16(tP + 48, p16[3]);
      }
      tmem_st_wait();
      tcgen05_fence_before();
      mbar_arrive_warp(&p_ready[g]);
      float r0, r1, r2, r3;
      upk2(rs2[0], r0, r1); upk2(rs2[1], r2, r3);
      l += (r0 + r1) + (r2 + r3);
    }
    // ---- epilogue: O / l -> bf16 rows, lse
    if (n_tiles > 0) {
      mbar_wait(&pv_done[g], (n_tiles - 1) & 1);
      tcgen05_fence_after();
    }
    const float inv = l > 0.f ? __frcp_rn(l) * (DROP ? drop.inv_keep : 1.f) : 0.f;
    uint4* dst = reinterpret_cast<uint4*>(P.out + (long long)t * P.o_st + (long long)b * P.o_sb + h * D);
#pragma unroll
    for (int c = 0; c < D / 32; ++c) {
      uint32_t o[32];
      if (n_tiles > 0) {
        tmem_ld_32x32b_x32(tO + c * 32, o);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int e = 0; e < 32; ++e) o[e] = 0u;
      }
      if (t < P.T) {
#pragma unroll
        for (int e = 0; e < 4; ++e)
          dst[c * 4 + e] = make_uint4(pack_bf16x2(__uint_as_float(o[8 * e]) * inv, __uint_as_float(o[8 * e + 1]) * inv),
                                      pack_bf16x2(__uint_as_float(o[8 * e + 2]) * inv, __uint_as_float(o[8 * e + 3]) * inv),
                                      pack_bf16x2(__uint_as_float(o[8 * e + 4]) * inv, __uint_as_float(o[8 * e + 5]) * inv),
                                      pack_bf16x2(__uint_as_float(o[8 * e + 6]) * inv, __uint_as_float(o[8 * e + 7]) * inv));
      }
    }
    if (t < P.T) P.lse[((long long)b * P.nH + h) * P.T + t] = l > 0.f ? (m_use + __log2f(l)) * kMLn2 : -INFINITY;
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 9) tmem_dealloc<512>(tmem);
}

// ------------------------------------------------------------------------------------------
// Backward
// ------------------------------------------------------------------------------------------
// Pre-pass: per query row (b, h, t) the two numbers the backward kernels need, already in the form their inner loop uses
// and interleaved per PAIR of queries -- rowdata[(b, h)][t / 2] = {-lse2(t), -lse2(t + 1), -delta(t) scale, -delta(t + 1) scale}
// with lse2 = lse log2(e) and delta = sum_e dO[t, b, h D + e] * O[t, b, h D + e] -- so that the dK/dV kernel gets the 128
// queries of a streamed tile as ONE 1 KB bulk copy that lands with the tile.  Rows are padded to Tpad = a multiple of 128 per
// (b, h) with {-inf, 0} (P = 0, dS = 0); a fully masked row (lse = -inf) gets -inf as well.
// D / 8 threads per row, 16 bytes each, channels fastest: a warp reads 512 contiguous bytes of a (t, b) row.
template <int D>
__global__ void mha_rowdata_kernel(const __nv_bfloat16* __restrict__ o, long long o_st, long long o_sb, const __nv_bfloat16* __restrict__ dout,
                                   long long do_st, long long do_sb, const float* __restrict__ lse, int T, int Tpad, int B, int nH,
                                   float scale, float* __restrict__ rowdata) {
  constexpr int G = D / 8;                              // threads per row
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;       // (((t, b), h), c)
  const long long row = idx / G;
  const int c = (int)(idx - row * G);
  const bool live = row < (long long)Tpad * B * nH;
  const int h = live ? (int)(row % nH) : 0;
  const long long tb = live ? row / nH : 0;
  const int b = (int)(tb % B), t = (int)(tb / B);
  float s = 0.f;
  if (live && t < T) {
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(o + (long long)t * o_st + (long long)b * o_sb + h * D) + c);
    const uint4 g = __ldg(reinterpret_cast<const uint4*>(dout + (long long)t * do_st + (long long)b * do_sb + h * D) + c);
    const uint32_t ua[4] = {a.x, a.y, a.z, a.w}, ug[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
    for (int k = 0; k < 4; ++k)
      s += __uint_as_float(ua[k] << 16) * __uint_as_float(ug[k] << 16) + __uint_as_float(ua[k] & 0xffff0000u) * __uint_as_float(ug[k] & 0xffff0000u);
  }
#pragma unroll
  for (int m = G / 2; m > 0; m >>= 1) s += __shfl_xor_sync(0xffffffffu, s, m);
  if (live && c == 0) {
    const long long bh = (long long)b * nH + h;
    float nl = -INFINITY, nds = 0.f;
    if (t < T) {
      const float l = __ldg(lse + bh * T + t);
      nl = l == -INFINITY ? -INFINITY : -l * kMLog2e;
      nds = -s * scale;
    }
    float* dst = rowdata + (bh * (Tpad >> 1) + (t >> 1)) * 4 + (t & 1);
    dst[0] = nl;
    dst[2] = nds;
  }
}

// MODE 0: dK, dV (CTA = key tile, query tiles stream).  MODE 1: dQ (CTA = query tile, key tiles stream).
//
// Per 128 x 128 block both kernels recompute the logits and dP with the CTA's RESIDENT rows along M (TMEM lanes) and the
// STREAMED rows along N (TMEM columns):
//   mode 0   S^T = K Q^T, dP^T = V dO^T   (lane = key, column = query);   dV += P^T dO,  dK += dS^T Q
//   mode 1   S   = Q K^T, dP   = dO V^T   (lane = query, column = key);   dQ += dS K
// so that P / dS, written by the thread that owns the lane, are already the A operand (M x K, K along the columns) of the
// gradient MMAs and go back into TENSOR MEMORY as bf16 pairs (tcgen05.st), never through shared memory.  (With P and dS as
// shared-memory tiles the kernels were bound by shared-memory bandwidth: an M128 N64 K16 MMA with both operands in shared
// memory reads 6 KB per 32 tensor cycles, 192 B/clk of the SM's 128, on top of 64 KB of P / dS stores per block.)
//
// Sixteen compute warps: warps w, w + 4, w + 8, w + 12 share the TMEM lane quadrant 32 (w % 4) and take one 32-column
// panel of the block each.  A thread loads its 32 logits and 32 dP values into registers in one go and hands the S / dP
// buffer back: the MMA warp issues S and dP of the next block at once (they run under this block's exponentials), then
// this block's gradient MMAs when P / dS are in TMEM.  lse and delta belong to the query: the thread's own row in mode 1;
// in mode 0 the streamed tile's 128 query pairs, which arrive in shared memory WITH the tile (one 1 KB bulk copy of the
// pre-pass's row data on the tile's barrier: no staging through registers, no CTA-wide barrier per block).
// (Tried and dropped: two independent groups of eight warps, each on its own 64 streamed rows of the block with M128 N64
// MMAs, so that one group's exponentials overlap the other's TMEM traffic -- 7 % SLOWER: with both operands in shared memory
// an N64 MMA reads 6 KB per 32 tensor cycles, 192 B/clk against the SM's 128 B/clk, and per block the operand reads of the
// seven GEMMs plus the TMA writes already add up to ~1000 shared-memory cycles, as many as the tensor and MUFU pipes need.)
// TMEM columns: S 0 | dP 128 | accumulators 256 (dV or dQ), 256 + D (dK) | P 384 | dS 448.   576 threads x 96 registers.
// PERSISTENT: one CTA per SM walks the (resident tile, head, batch) items with stride gridDim.x.  All pipelines run on
// across item boundaries -- the streamed-tile ring, the S / dP and P / dS hand-offs (running step counter g), the resident
// tiles (double-buffered: the next item's K / V or Q / dO land while this item streams) -- so the only per-item cost left is
// the accumulator read-out, and that overlaps the next item's first S / dP MMAs and loads (the gradient MMAs of the next
// item wait for acc_free).  One CTA per item paid TMEM allocation, barrier setup, the resident loads' latency and the
// drain of every item in the open: ~15 % at 16 streamed tiles per item.
struct BwdItem { int o0, h, b, n_begin, n_tiles; };
template <int MODE>
__device__ __forceinline__ BwdItem bwd_item(const MhaParams& P, int w) {
  const int n_ot = ((MODE == 0 ? P.S : P.T) + 127) >> 7;
  BwdItem it;
  const int hb = w / n_ot;
  int ot = w % n_ot;
  // With the future mask an item's work grows (mode 1) or shrinks (mode 0) with its tile index, and a CTA's stride over w
  // visits only a few residues of it: every other (head, batch) runs its tiles in reverse, so heavy and light items mix.
  if (hb & 1) ot = n_ot - 1 - ot;
  it.o0 = ot * 128; it.h = hb % P.nH; it.b = hb / P.nH;
  int n_end;
  if (MODE == 0) { it.n_begin = first_query_tile(P, it.o0); n_end = (P.T + 127) >> 7; }
  else { it.n_begin = 0; n_end = visible_key_tiles(P, it.o0); }
  it.n_tiles = max(0, n_end - it.n_begin);
  return it;
}

template <int D, int MODE, bool DROP>
__global__ void __launch_bounds__(kMThreadsB, 1)
mha_bwd_tc_kernel(const __grid_constant__ MhaParams P) {
  constexpr int kTileB = D * 256;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sR = smem;                                   // [2][2] resident, double-buffered over items: K | V (mode 0) / Q | dO (mode 1)
  uint8_t* sS0 = sR + 4 * kTileB;                       // [kMStagesB] streamed: Q (mode 0) / K (mode 1)
  uint8_t* sS1 = sS0 + kMStagesB * kTileB;              // [kMStagesB] streamed: dO (mode 0) / V (mode 1)
  float4* sRow = reinterpret_cast<float4*>(sS1 + kMStagesB * kTileB);   // mode 0: [kMStagesB][64] row data of the streamed queries
  uint64_t* bars = reinterpret_cast<uint64_t*>(sRow + kMStagesB * 64);
  uint64_t* r_full = bars;                              // [2]
  uint64_t* r_empty = bars + 2;                         // [2] the item's S / dP MMAs have all read the resident tiles
  uint64_t* full = bars + 4;                            // [kMStagesB]
  uint64_t* empty = full + kMStagesB;                   // [kMStagesB]
  uint64_t* s_full = empty + kMStagesB;                 // S and dP in TMEM
  uint64_t* sdp_free = s_full + 1;                      // ... and in the threads' registers (one arrival per compute warp)
  uint64_t* ps_ready = s_full + 2;                      // P / dS in TMEM (one arrival per compute warp)
  uint64_t* ps_free = s_full + 3;                       // the gradient MMAs have read them
  uint64_t* acc_done = s_full + 4;                      // the item's last gradient MMAs have completed
  uint64_t* acc_free = s_full + 5;                      // ... and the accumulators are in the epilogue warps' registers
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_full + 6);
  constexpr int kEpiWarpsB = MODE == 0 ? 8 : 4;         // warps that read accumulators: dV, dK (mode 0) / dQ (mode 1)

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int total = (((MODE == 0 ? P.S : P.T) + 127) >> 7) * P.nH * P.B;
  const DropoutCfg drop = DROP ? dropout_at_entry(P.drop, P.rng) : P.drop;

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) { mbar_init(&r_full[i], 1); mbar_init(&r_empty[i], 1); }
    for (int s = 0; s < kMStagesB; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(s_full, 1); mbar_init(sdp_free, kMComputeWarpsB); mbar_init(ps_ready, kMComputeWarpsB); mbar_init(ps_free, 1);
    mbar_init(acc_done, 1); mbar_init(acc_free, kEpiWarpsB);
    fence_barrier_init();
  }
  if (warp == kMComputeWarpsB && lane == 0) { tma_prefetch_desc(&P.q); tma_prefetch_desc(&P.k); tma_prefetch_desc(&P.v); tma_prefetch_desc(&P.dout); }
  if (warp == kMComputeWarpsB + 1) tmem_alloc<512>(tmem_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tA0 = tmem + 256, tA1 = tmem + 256 + D, tP = tmem + 384, tdS = tmem + 448;

  if (warp >= kMComputeWarpsB) {
    if (warp == kMComputeWarpsB) {
      // ============================== TMA producer ==============================
      if (elect_one()) {
        int g = 0, ri = 0;                              // streamed tiles / items with work so far (this CTA)
        for (int w = blockIdx.x; w < total; w += gridDim.x) {
          const BwdItem it = bwd_item<MODE>(P, w);
          if (it.n_tiles == 0) continue;
          const int rb = ri & 1;
          mbar_wait(&r_empty[rb], ((ri >> 1) & 1) ^ 1);
          mbar_arrive_expect_tx(&r_full[rb], 2 * kTileB);
          tma_load_4d(MODE == 0 ? &P.k : &P.q, &r_full[rb], sR + rb * 2 * kTileB, 0, it.o0, it.h * (D / 32), it.b);
          tma_load_4d(MODE == 0 ? &P.v : &P.dout, &r_full[rb], sR + rb * 2 * kTileB + kTileB, 0, it.o0, it.h * (D / 32), it.b);
          const float4* rowdata = reinterpret_cast<const float4*>(P.rowdata) + ((long long)it.b * P.nH + it.h) * (P.Tpad >> 1);
          for (int n = 0; n < it.n_tiles; ++n, ++g) {
            const int s = g % kMStagesB, row0 = (it.n_begin + n) * 128;
            mbar_wait(&empty[s], ((g / kMStagesB) & 1) ^ 1);
            mbar_arrive_expect_tx(&full[s], 2 * kTileB + (MODE == 0 ? 1024 : 0));
            tma_load_4d(MODE == 0 ? &P.q : &P.k, &full[s], sS0 + s * kTileB, 0, row0, it.h * (D / 32), it.b);
            tma_load_4d(MODE == 0 ? &P.dout : &P.v, &full[s], sS1 + s * kTileB, 0, row0, it.h * (D / 32), it.b);
            if (MODE == 0) bulk_load_1d(sRow + s * 64, rowdata + (row0 >> 1), 1024, &full[s]);
          }
          ++ri;
        }
      }
    } else {
      // ============================== MMA issuer ==============================
      constexpr uint32_t idescS = umma_idesc_bf16(128, 128, 0, 0);      // A = resident tile, B = streamed tile, both K-major
      constexpr uint32_t idescG = umma_idesc_bf16(128, D, 0, 1);        // A = P / dS (TMEM), B = streamed tile read MN-major
      const uint64_t dKm = umma_smem_desc(0, 0, 512, kSwz64);           // K-major
      const uint64_t dMn = umma_smem_desc(0, 8192, 512, kSwz64);        // MN-major, 32-wide panels 8 KB (128 rows) apart
      const uint32_t rbase = smem_u32(sR) >> 4, s0b = smem_u32(sS0) >> 4, s1b = smem_u32(sS1) >> 4;
      const uint32_t tS = tmem, tdP = tmem + 128;
      // gradient MMAs of step pg (deferred by one step so that the next S / dP run first); first / last: of their item
      int pg = -1, p_ri = 0;
      bool p_first = false, p_last = false;
      auto issue_grad = [&]() {
        const int s = pg % kMStagesB;
        mbar_wait(ps_ready, pg & 1);
        if (p_first && p_ri > 0) mbar_wait(acc_free, (p_ri - 1) & 1);   // the previous item's accumulators have been read out
        tcgen05_fence_after();
        if (elect_one()) {
          const uint32_t acc = p_first ? 0u : 1u;
#pragma unroll
          for (int ks = 0; ks < 8; ++ks) {                               // 16 streamed rows = 8 TMEM columns of P / dS per step
            if (MODE == 0) {
              umma_bf16_ts(tA0, tP + ks * 8, dMn + (s1b + s * (kTileB >> 4) + ks * 64), idescG, acc | (ks > 0));    // dV += P^T dO
              umma_bf16_ts(tA1, tdS + ks * 8, dMn + (s0b + s * (kTileB >> 4) + ks * 64), idescG, acc | (ks > 0));   // dK += dS^T Q
            } else {
              umma_bf16_ts(tA0, tdS + ks * 8, dMn + (s0b + s * (kTileB >> 4) + ks * 64), idescG, acc | (ks > 0));   // dQ += dS K
            }
          }
          umma_commit(ps_free);
          umma_commit(&empty[s]);
          if (p_last) umma_commit(acc_done);
        }
        __syncwarp();
        pg = -1;
      };
      int g = 0, ri = 0;
      for (int w = blockIdx.x; w < total; w += gridDim.x) {
        const BwdItem it = bwd_item<MODE>(P, w);
        if (it.n_tiles == 0) continue;
        const int rb = ri & 1;
        const uint32_t r0 = rbase + rb * (2 * kTileB >> 4), r1 = r0 + (kTileB >> 4);
        mbar_wait(&r_full[rb], (ri >> 1) & 1);
        for (int n = 0; n < it.n_tiles; ++n, ++g) {
          const int s = g % kMStagesB;
          mbar_wait(&full[s], (g / kMStagesB) & 1);
          if (g > 0) mbar_wait(sdp_free, (g - 1) & 1);                   // S, dP of the previous step are in registers
          tcgen05_fence_after();
          if (elect_one()) {
#pragma unroll
            for (int ks = 0; ks < D / 16; ++ks) {
              const uint32_t o = (ks >> 1) * (8192 >> 4) + (ks & 1) * 2;
              umma_bf16_ss(tS, dKm + (r0 + o), dKm + (s0b + s * (kTileB >> 4) + o), idescS, ks > 0 ? 1u : 0u);      // S(^T) = R0 S0^T
            }
#pragma unroll
            for (int ks = 0; ks < D / 16; ++ks) {
              const uint32_t o = (ks >> 1) * (8192 >> 4) + (ks & 1) * 2;
              umma_bf16_ss(tdP, dKm + (r1 + o), dKm + (s1b + s * (kTileB >> 4) + o), idescS, ks > 0 ? 1u : 0u);     // dP(^T) = R1 S1^T
            }
            umma_commit(s_full);
            if (n == it.n_tiles - 1) umma_commit(&r_empty[rb]);          // the resident buffer can take the item after next
          }
          __syncwarp();
          if (pg >= 0) issue_grad();
          pg = g; p_ri = ri; p_first = n == 0; p_last = n == it.n_tiles - 1;
        }
        ++ri;
      }
      if (pg >= 0) issue_grad();
    }
  } else {
    // ============================== P / dS: thread = (resident row, one 32-column panel of the block) ==============================
    const int r = tid & 127, col0 = (warp >> 2) * 32;   // lane = resident row; streamed columns col0 .. col0 + 31
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t tS = tmem + lane_base + col0, tdP = tS + 128;
    const float sc = P.scale * kMLog2e;
    const int which = warp >> 2;                        // epilogue: warps 0-3 dV / dQ, warps 4-7 dK
    int g = 0, ri = 0;
    for (int w = blockIdx.x; w < total; w += gridDim.x) {
      const BwdItem itm = bwd_item<MODE>(P, w);
      const int o0 = itm.o0, h = itm.h, b = itm.b, n_begin = itm.n_begin, n_tiles = itm.n_tiles;
      const long long item = (long long)b * P.nH + h;
      float nl_own = -INFINITY, nds_own = 0.f;          // mode 1: the thread's own query
      if (MODE == 1 && n_tiles > 0) {
        const float* rd = reinterpret_cast<const float*>(reinterpret_cast<const float4*>(P.rowdata) + item * (P.Tpad >> 1) + ((o0 + r) >> 1)) + (r & 1);
        nl_own = __ldg(rd); nds_own = __ldg(rd + 2);
      }
      for (int n = 0; n < n_tiles; ++n, ++g) {
        const int t0 = MODE == 0 ? (n_begin + n) * 128 : o0, s0 = MODE == 0 ? o0 : (n_begin + n) * 128;
        const float4* row = sRow + (g % kMStagesB) * 64 + (col0 >> 1);
        const bool masked = tile_needs_mask(P, t0, s0);
        if (MODE == 0) mbar_wait(&full[g % kMStagesB], (g / kMStagesB) & 1);   // the row data came with the tile (long complete: one test)
        mbar_wait(s_full, g & 1);
        tcgen05_fence_after();
        uint32_t vs[32], vd[32];
        tmem_ld_32x32b_x32(tS, vs);
        tmem_ld_32x32b_x32(tdP, vd);
        tmem_ld_wait();
        tcgen05_fence_before();
        mbar_arrive_warp(sdp_free);
        // P = exp2(s sc - lse), dS = P (dP - delta) scale  ->  bf16 pairs
        float a_mul = sc;                             // logit (log2 domain) = vs * a_mul
        if (masked) {                                 // diagonal / ragged blocks, kept out of the main path
          if (P.mask_kind == MMN_MASK_TENSOR) {       // an additive mask tensor: fold scale and mask into vs
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              const int col = col0 + e;
              const float mt = MODE == 0 ? mask_term(P, t0 + col, s0 + r) : mask_term(P, t0 + r, s0 + col);
              vs[e] = __float_as_uint(fmaf(__uint_as_float(vs[e]), sc, mt));
            }
            a_mul = 1.f;
          } else if (MODE == 0) {
            // lane = key s, columns = queries: the key is seen by the queries t > s - diag, i.e. columns e >= e_min; a key
            // beyond S by none (queries beyond T carry -inf in their row data)
            const int sk = s0 + r;
            int e_min = P.mask_kind == MMN_MASK_FUTURE ? sk - P.mask_diag + 1 - t0 - col0 : 0;
            if (sk >= P.S) e_min = 32;
#pragma unroll
            for (int e = 0; e < 32; ++e) vs[e] = e >= e_min ? vs[e] : 0xff800000u;
          } else {
            // lane = query t, columns = keys: the row sees the keys e < e_lim of this panel
            int e_lim = P.S - s0 - col0;
            if (P.mask_kind == MMN_MASK_FUTURE) e_lim = min(e_lim, t0 + r + P.mask_diag - s0 - col0);
#pragma unroll
            for (int e = 0; e < 32; ++e) vs[e] = e < e_lim ? vs[e] : 0xff800000u;
          }
        }
        const float scd = DROP ? P.scale * drop.inv_keep : P.scale;
        const uint64_t a2 = pk2(a_mul, a_mul), sc2 = pk2(scd, scd);
        uint32_t pp[16], dd[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          uint64_t nl2, nds2;
          if (MODE == 0) {
            const float4 rw = row[e];                 // the pair's queries (broadcast read)
            nl2 = pk2(rw.x, rw.y); nds2 = pk2(rw.z, rw.w);
          } else {
            nl2 = pk2(nl_own, nl_own); nds2 = pk2(nds_own, nds_own);
          }
          float x0, x1;
          exp2_pair<MMN_MHA_POLY_BWD>(fma2(pk2u(vs[2 * e], vs[2 * e + 1]), a2, nl2), e, x0, x1);
          if (DROP) {
            // the forward's mask: dP of a dropped probability is 0, of a kept one dP / (1 - p) (sc2 carries the factor); P^T dO
            // uses the dropped P (its 1 / (1 - p) is applied to dV in the epilogue)
            bool k0, k1;
            if (MODE == 0) {                          // lane = key, the pair = two queries of one block row pair
              const uint4 rr = dropout_block(drop, (int)item, ((t0 + col0) >> 1) + e, (s0 + r) >> 1);
              const bool odd = (s0 + r) & 1;
              k0 = dropout_keep_word(odd ? rr.y : rr.x, drop.thr); k1 = dropout_keep_word(odd ? rr.w : rr.z, drop.thr);
            } else {                                  // lane = query, the pair = two keys
              const uint4 rr = dropout_block(drop, (int)item, (t0 + r) >> 1, ((s0 + col0) >> 1) + e);
              const bool odd = (t0 + r) & 1;
              k0 = dropout_keep_word(odd ? rr.z : rr.x, drop.thr); k1 = dropout_keep_word(odd ? rr.w : rr.y, drop.thr);
            }
            if (!k0) vd[2 * e] = 0u;
            if (!k1) vd[2 * e + 1] = 0u;
            pp[e] = pack_bf16x2(k0 ? x0 : 0.f, k1 ? x1 : 0.f);
          } else {
            pp[e] = pack_bf16x2(x0, x1);
          }
          dd[e] = pack_bf16x2(mul2(pk2(x0, x1), fma2(pk2u(vd[2 * e], vd[2 * e + 1]), sc2, nds2)));
        }
        if (g > 0) {                                  // the gradient MMAs of the previous step have read P / dS
          mbar_wait(ps_free, (g - 1) & 1);
          tcgen05_fence_after();
        }
        tmem_st_32x32b_x16(tdS + lane_base + (col0 >> 1), dd);
        if (MODE == 0) tmem_st_32x32b_x16(tP + lane_base + (col0 >> 1), pp);
        tmem_st_wait();
        tcgen05_fence_before();
        mbar_arrive_warp(ps_ready);
      }
      // ---- epilogue of the item: the accumulators -> bf16 rows (warps 0-3: dV / dQ, warps 4-7: dK); the other warps go on
      if (which < (MODE == 0 ? 2 : 1)) {
        const int orow = o0 + r;
        const int limit = MODE == 0 ? P.S : P.T;
        __nv_bfloat16* base = MODE == 0 ? (which == 0 ? P.dv : P.dk) : P.dq;
        const long long st = MODE == 0 ? (which == 0 ? P.dv_st : P.dk_st) : P.dq_st, sb = MODE == 0 ? (which == 0 ? P.dv_sb : P.dk_sb) : P.dq_sb;
        uint32_t v[D];
        if (n_tiles > 0) {
          mbar_wait(acc_done, ri & 1);
          tcgen05_fence_after();
          uint32_t (*v32)[32] = reinterpret_cast<uint32_t (*)[32]>(v);
#pragma unroll
          for (int c = 0; c < D / 32; ++c) tmem_ld_32x32b_x32((which == 0 ? tA0 : tA1) + lane_base + c * 32, v32[c]);
          tmem_ld_wait();
          tcgen05_fence_before();
          mbar_arrive_warp(acc_free);                 // the next item's gradient MMAs may overwrite the accumulators
        } else {
#pragma unroll
          for (int e = 0; e < D; ++e) v[e] = 0u;
        }
        if (DROP && MODE == 0 && which == 0) {         // dV = (P_drop / (1 - p))^T dO
#pragma unroll
          for (int e = 0; e < D; ++e) v[e] = __float_as_uint(__uint_as_float(v[e]) * drop.inv_keep);
        }
        if (orow < limit) {
          uint4* dst = reinterpret_cast<uint4*>(base + (long long)orow * st + (long long)b * sb + h * D);
#pragma unroll
          for (int e = 0; e < D / 8; ++e)
            dst[e] = make_uint4(pack_bf16x2(__uint_as_float(v[8 * e]), __uint_as_float(v[8 * e + 1])),
                                pack_bf16x2(__uint_as_float(v[8 * e + 2]), __uint_as_float(v[8 * e + 3])),
                                pack_bf16x2(__uint_as_float(v[8 * e + 4]), __uint_as_float(v[8 * e + 5])),
                                pack_bf16x2(__uint_as_float(v[8 * e + 6]), __uint_as_float(v[8 * e + 7])));
        }
      }
      if (n_tiles > 0) ++ri;
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == kMComputeWarpsB + 1) tmem_dealloc<512>(tmem);
}

// ------------------------------------------------------------------------------------------
// Host side
// ------------------------------------------------------------------------------------------
static bool row_map(CUtensorMap* out, const void* ptr, int len, int batch, int embed, long long st, long long sb, int D) {
  EncodeTiledFn enc = encode_fn();
  if (!enc) return false;
  cuuint64_t dims[4] = {32, (cuuint64_t)len, (cuuint64_t)(embed / 32), (cuuint64_t)batch};
  cuuint64_t strides[3] = {(cuuint64_t)st * 2, 64, (cuuint64_t)sb * 2};
  cuuint32_t box[4] = {32, 128, (cuuint32_t)(D / 32), 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  return enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static bool aligned(const void* p, long long st, long long sb) {
  return reinterpret_cast<uintptr_t>(p) % 16 == 0 && st % 8 == 0 && sb % 8 == 0;
}

const char* mha_why_not(const mmn_mha_desc* d, bool backward) {
  if (d->io_dtype != MMN_DT_BF16) return "io dtype is not bf16";
  if (d->head_dim != 32 && d->head_dim != 64) return "head_dim is not 32 or 64";
  if (d->q_stride_t % 8 || d->q_stride_b % 8 || d->k_stride_t % 8 || d->k_stride_b % 8 || d->v_stride_t % 8 || d->v_stride_b % 8 ||
      d->o_stride_t % 8 || d->o_stride_b % 8)
    return "row strides not 16-byte aligned";
  if (backward && (d->do_stride_t % 8 || d->do_stride_b % 8 || d->dq_stride_t % 8 || d->dq_stride_b % 8 || d->dk_stride_t % 8 ||
                   d->dk_stride_b % 8 || d->dv_stride_t % 8 || d->dv_stride_b % 8))
    return "gradient row strides not 16-byte aligned";
  if (d->batch > 65535 || d->num_heads > 65535) return "batch or head count beyond the grid limits";
  if ((long long)((std::max(d->tgt_len, d->src_len) + 127) / 128) * d->num_heads * d->batch > 0x7fffffffLL) return "too many tiles";
  if (!encode_fn()) return "cuTensorMapEncodeTiled unavailable";
  return nullptr;
}

static void fill_common(MhaParams& P, const mmn_mha_desc* d, const float* mask) {
  P.T = d->tgt_len; P.S = d->src_len; P.B = d->batch; P.nH = d->num_heads;
  P.mask_kind = d->mask_kind; P.mask_diag = d->mask_diagonal; P.scale = d->scale; P.mask = mask;
  P.drop = make_dropout(d->dropout_p, d->seed, d->offset);
  P.rng = reinterpret_cast<const unsigned long long*>(d->rng);
}

template <int D, bool DROP>
static int mha_fwd_launch(const MhaParams& P, cudaStream_t st) {
  constexpr size_t smem = 1024 + (size_t)(2 + 2 * kMStagesF) * D * 256 + 24 * 8 + 16;
  static std::once_flag once;
  std::call_once(once, [] { cudaFuncSetAttribute(mha_fwd_tc_kernel<D, DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); });
  dim3 grid((P.T + 255) / 256, P.nH, P.B);
  mha_fwd_tc_kernel<D, DROP><<<grid, kMThreads, smem, st>>>(P);
  return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

int mha_fwd(const mmn_mha_desc* d, const void* q, const void* k, const void* v, const float* mask, void* out, float* lse, cudaStream_t st,
            char* err, size_t errlen, int* launches) {
  MhaParams P{};
  fill_common(P, d, mask);
  const int E = d->num_heads * d->head_dim, D = d->head_dim;
  if (!aligned(q, d->q_stride_t, d->q_stride_b) || !aligned(k, d->k_stride_t, d->k_stride_b) || !aligned(v, d->v_stride_t, d->v_stride_b) ||
      !aligned(out, d->o_stride_t, d->o_stride_b) || !row_map(&P.q, q, P.T, P.B, E, d->q_stride_t, d->q_stride_b, D) ||
      !row_map(&P.k, k, P.S, P.B, E, d->k_stride_t, d->k_stride_b, D) || !row_map(&P.v, v, P.S, P.B, E, d->v_stride_t, d->v_stride_b, D)) {
    snprintf(err, errlen, "mha: cuTensorMapEncodeTiled failed (pointer alignment or strides)");
    return MMN_ERR_CUDA;
  }
  P.out = static_cast<__nv_bfloat16*>(out); P.o_st = d->o_stride_t; P.o_sb = d->o_stride_b; P.lse = lse;
  const bool drop = P.drop.thr != 0;
  const int rc = D == 32 ? (drop ? mha_fwd_launch<32, true>(P, st) : mha_fwd_launch<32, false>(P, st))
                         : (drop ? mha_fwd_launch<64, true>(P, st) : mha_fwd_launch<64, false>(P, st));
  if (rc) { snprintf(err, errlen, "mha_fwd_tc_kernel: %s", cudaGetErrorString(cudaGetLastError())); return MMN_ERR_CUDA; }
  ++*launches;
  return MMN_OK;
}

template <int D, int MODE, bool DROP>
static int mha_bwd_launch(const MhaParams& P, cudaStream_t st) {
  constexpr size_t smem = 1024 + (size_t)(4 + 2 * kMStagesB) * D * 256 + kMStagesB * 64 * 16 + (2 * kMStagesB + 10) * 8 + 16;
  static std::once_flag once;
  std::call_once(once, [] { cudaFuncSetAttribute(mha_bwd_tc_kernel<D, MODE, DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); });
  const long long total = (long long)(((MODE == 0 ? P.S : P.T) + 127) / 128) * P.nH * P.B;
  const int grid = (int)std::min<long long>(total, num_sms_cached());      // persistent: one CTA per SM
  mha_bwd_tc_kernel<D, MODE, DROP><<<grid, kMThreadsB, smem, st>>>(P);
  return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

int mha_bwd(const mmn_mha_desc* d, const void* q, const void* k, const void* v, const float* mask, const void* out, const float* lse,
            const void* dout, void* dq, void* dk, void* dv, float* workspace, cudaStream_t st, char* err, size_t errlen, int* launches) {
  MhaParams P{};
  fill_common(P, d, mask);
  const int E = d->num_heads * d->head_dim, D = d->head_dim;
  if (!out) { snprintf(err, errlen, "mha backward (tcgen05) needs the forward output"); return MMN_ERR_INVALID; }
  if (!aligned(q, d->q_stride_t, d->q_stride_b) || !aligned(k, d->k_stride_t, d->k_stride_b) || !aligned(v, d->v_stride_t, d->v_stride_b) ||
      !aligned(out, d->o_stride_t, d->o_stride_b) || !aligned(dout, d->do_stride_t, d->do_stride_b) || !aligned(dq, d->dq_stride_t, d->dq_stride_b) ||
      !aligned(dk, d->dk_stride_t, d->dk_stride_b) || !aligned(dv, d->dv_stride_t, d->dv_stride_b) ||
      !row_map(&P.q, q, P.T, P.B, E, d->q_stride_t, d->q_stride_b, D) || !row_map(&P.k, k, P.S, P.B, E, d->k_stride_t, d->k_stride_b, D) ||
      !row_map(&P.v, v, P.S, P.B, E, d->v_stride_t, d->v_stride_b, D) || !row_map(&P.dout, dout, P.T, P.B, E, d->do_stride_t, d->do_stride_b, D)) {
    snprintf(err, errlen, "mha: cuTensorMapEncodeTiled failed (pointer alignment or strides)");
    return MMN_ERR_CUDA;
  }
  P.lse = const_cast<float*>(lse);
  P.rowdata = workspace;
  P.Tpad = (P.T + 127) / 128 * 128;
  P.dq = static_cast<__nv_bfloat16*>(dq); P.dk = static_cast<__nv_bfloat16*>(dk); P.dv = static_cast<__nv_bfloat16*>(dv);
  P.dq_st = d->dq_stride_t; P.dq_sb = d->dq_stride_b; P.dk_st = d->dk_stride_t; P.dk_sb = d->dk_stride_b;
  P.dv_st = d->dv_stride_t; P.dv_sb = d->dv_stride_b;
  const long long n = (long long)P.B * P.nH * P.Tpad * (D / 8);
  const unsigned blocks = (unsigned)((n + 255) / 256);
  if (D == 32)
    mha_rowdata_kernel<32><<<blocks, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(out), d->o_stride_t, d->o_stride_b,
                                                   static_cast<const __nv_bfloat16*>(dout), d->do_stride_t, d->do_stride_b, lse, P.T, P.Tpad,
                                                   P.B, P.nH, P.scale, workspace);
  else
    mha_rowdata_kernel<64><<<blocks, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(out), d->o_stride_t, d->o_stride_b,
                                                   static_cast<const __nv_bfloat16*>(dout), d->do_stride_t, d->do_stride_b, lse, P.T, P.Tpad,
                                                   P.B, P.nH, P.scale, workspace);
  if (cudaGetLastError() != cudaSuccess) { snprintf(err, errlen, "mha_rowdata_kernel launch failed"); return MMN_ERR_CUDA; }
  ++*launches;
  const bool drop = P.drop.thr != 0;
  int rc = D == 32 ? (drop ? mha_bwd_launch<32, 0, true>(P, st) : mha_bwd_launch<32, 0, false>(P, st))
                   : (drop ? mha_bwd_launch<64, 0, true>(P, st) : mha_bwd_launch<64, 0, false>(P, st));
  if (!rc) {
    ++*launches;
    rc = D == 32 ? (drop ? mha_bwd_launch<32, 1, true>(P, st) : mha_bwd_launch<32, 1, false>(P, st))
                 : (drop ? mha_bwd_launch<64, 1, true>(P, st) : mha_bwd_launch<64, 1, false>(P, st));
  }
  if (rc) { snprintf(err, errlen, "mha_bwd_tc_kernel: %s", cudaGetErrorString(cudaGetLastError())); return MMN_ERR_CUDA; }
  ++*launches;
  return MMN_OK;
}

}}  // namespace mmn::tc
