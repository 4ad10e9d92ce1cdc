// winattn_tc_qkv_fwd.cuh -- self-attention window forward with the qkv projection fused in (tcgen05.mma + TMEM + TMA):
//
//   qkv = x W_qkv^T + b_qkv        fp32 accumulate, fp32 bias, rounded to bf16 and written to global (the backward reads it)
//   out, lse, records              exactly what winattn_fwd_tc_kernel computes from that bf16 qkv
//
// Shape: C = 96 = 3 heads x 32, 64-token windows (fwd_why_not's shapes), y = None.  The separate projection wrote
// qkv (3C per token) and the attention read it straight back; here x (C per token) is read once and qkv only written.
//
// A work item is a PAIR of windows of one wrap class (tc_sched.cuh, ClassQueue, one queue for all heads), now across all
// three heads: sub-item n = (pair n / 3, head n % 3), and softmax group g = head g.  One CTA per SM, 512 threads:
//
//   warp 12     TMA producer: schedule, pair descriptors, the pair's x tile (128 rows x 96 channels = three 64B-swizzled
//               32-channel panels) through the wrap-class box plans over x (B, D, H, W, C).  2-stage ring.
//   warp 13     MMA issuer, three queues served in turn:
//                 projection  D[g] = [x tile] W_g^T, M128 N96 K96 (q_g | k_g | v_g) into group g's columns 0..95, once
//                             PV of the group's previous sub-item has completed (those columns held its S and P);
//                 S           M128 N128 K32: [Q0;Q1] x [K0;K1]^T, both windows' queries against both windows' keys;
//                             each row reads only its own window's 64 columns (no zero block: 8 KB less shared memory
//                             per group than the [Q0;0],[0;Q1] product of the unfused kernel, at the same MMA cost);
//                 PV          as in the unfused kernel, A = P from TMEM columns 0..63 of the group.
//   warps 0-11  softmax groups: one thread per row.  Drain the projection (bias, bf16, swizzled rows of the group's
//               Q, K, V operand tiles; 1/||q||, 1/||k|| from the rounded values in registers), then the unfused kernel's
//               softmax (softmax_row) and epilogue (o_row_to_smem); o is staged in the group's Q tile (dead after S).
//   warp 14     TMA store of o; a staging tile goes back to its group as soon as its stores have read it.
//   warp 15     TMA store of the Q, K, V tiles to global qkv through the q/k/v box plans (the layout the backward reads).
//
// Shared memory (bytes): W_qkv head-major [3 heads][3 K panels][96 rows][64] 55296 | x ring 2 x 24576 | per group
// Q | K | V tiles 3 x 24576 | class tables 3 x 64 x 64 fp32 (float4-swizzled rows, no padding) 49152 | 1/||k|| 3 x 512 |
// position / region LUTs 1024 | descriptor ring | barriers.  TMEM: group g owns columns 160 g .. 160 g + 159: S (and the
// projection, and P in 0..63) in 0..127, O in 128..159; 480 of 512.  Registers by setmaxnreg as in the unfused kernel.
#pragma once

#include "winattn_tc_fwd.cuh"

namespace mmn { namespace tc {

constexpr int kQkvHeads = kGroupsF;                 // one softmax group per head
constexpr int kQkvC = kQkvHeads * kD;               // 96
constexpr int kXPanel = 128 * 64;                   // one 32-channel panel of a pair's x tile
constexpr int kXStage = (kQkvC / 32) * kXPanel;     // 24 KB
constexpr int kXStages = 2;
constexpr int kWPanel = 96 * 64;                    // q_h | k_h | v_h rows of one 32-channel K panel
constexpr int kWHead = (kQkvC / 32) * kWPanel;
constexpr int kWBytes = kQkvHeads * kWHead;         // 54 KB
constexpr int kOpTile = 128 * 64;                   // the pair's Q, K or V tile of one head
constexpr int kOpSet = 3 * kOpTile;
constexpr int kQkvBars = 2 * kXStages + 8 * kGroupsF;
constexpr size_t kQkvSmemBytes = 1024 /*align slack*/ + kWBytes + kXStages * kXStage + kGroupsF * kOpSet + kGroupsF * kN * kN * 4 +
                                 kGroupsF * 128 * 4 + 1024 + ItemRing<kItemRing>::kBytes + 16 + kQkvBars * 8 + 8;
static_assert(kQkvSmemBytes <= 227 * 1024, "fused qkv forward: shared memory over the 227 KB a block may use");
static_assert(kGroupsF * kTmemGroup <= kTmemColsF && 96 <= 128, "fused qkv forward: TMEM columns");

struct QkvFwdParams {
  CUtensorMap x[3][8];                // x, one map set per 32-channel panel (base x + 32 p)
  CUtensorMap q[8], k[8], v[8], o[8];
  WinShape S;
  Sched sc;
  int mask_windows;
  float scale;
  const __nv_bfloat16* w;             // (3C, C)
  const float* b;                     // (3C) or null
  const float* bias;
  const float* head_scale;
  const float* mask;
  float* lse;                         // as FwdParams
  long long slab;
  int* work;
};

__device__ __forceinline__ void tmem_st_zero_x32(uint32_t taddr) {
  const uint32_t z = 0u;
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, "
      "%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(z)
      : "memory");
}

template <bool COS, int MASK>
__global__ void __launch_bounds__(kFwdThreads, 1)
winattn_qkv_fwd_tc_kernel(const __grid_constant__ QkvFwdParams P) {
  constexpr int G = kGroupsF;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sW = smem;
  uint8_t* sX = sW + kWBytes;                             // [kXStages] x tiles
  uint8_t* sOp = sX + kXStages * kXStage;                 // [G] Q | K | V (Q doubles as the o staging tile)
  float* sTbl = reinterpret_cast<float*>(sOp + G * kOpSet); // [G][64][64], float4 j4 of row i at j4 ^ (i & 7)
  float* sRk = sTbl + G * kN * kN;                        // [G][128] per-key 1/||k||
  uint8_t* sPos = reinterpret_cast<uint8_t*>(sRk + G * 128);
  uint8_t* sRid = sPos + 512;
  const ItemRing<kItemRing> ring{reinterpret_cast<int4*>(sRid + 512)};      // pair descriptors (tc_sched.cuh)
  int* sEnd = reinterpret_cast<int*>(sRid + 512 + ring.kBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(sEnd + 4);
  uint64_t* x_full = bars;                                // [kXStages] TMA -> MMA
  uint64_t* x_empty = x_full + kXStages;                  // [kXStages] the pair's last projection -> TMA
  uint64_t* proj_full = x_empty + kXStages;               // [G] projection in TMEM (commit + the MMA thread's arrival)
  uint64_t* tiles_full = proj_full + G;                   // [G] Q, K, V tiles written (one arrival per warp)
  uint64_t* s_full = tiles_full + G;
  uint64_t* p_full = s_full + G;
  uint64_t* o_full = p_full + G;
  uint64_t* qkv_free = o_full + G;                        // [G] Q, K, V tiles read out by the qkv stores
  uint64_t* so_ready = qkv_free + G;
  uint64_t* so_free = so_ready + G;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(so_free + G);

  const WinShape& S = P.S;
  const Sched& sc = P.sc;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  // ---- one-time setup: W_qkv into shared memory, head-major, as K-major 64B-swizzled panels of 96 rows; the x ring
  // zeroed (rows of a pair's missing second window project stale but finite data, which P = 0 then cancels)
  for (int e = tid; e < kWBytes / 16; e += kFwdThreads) {
    const int c = e & 3, j = (e >> 2) % 96, hp = (e >> 2) / 96;      // hp = head * 3 + panel
    const int hh = hp / 3, p = hp - hh * 3;
    const int row = (j >> 5) * kQkvC + hh * kD + (j & 31);
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(P.w + (size_t)row * kQkvC + p * 32 + c * 8));
    *reinterpret_cast<uint4*>(sW + hp * kWPanel + j * 64 + ((c ^ ((j >> 1) & 3)) << 4)) = v;
  }
  for (int i = tid; i < (kXStages * kXStage) / 16; i += kFwdThreads) reinterpret_cast<uint4*>(sX)[i] = make_uint4(0, 0, 0, 0);
  fill_class_luts(S, sPos, sRid, tid, kFwdThreads);
  if (tid == 0) {
    for (int g = 0; g < G; ++g) sEnd[g] = 0x7fffffff;
    for (int s = 0; s < kXStages; ++s) { mbar_init(&x_full[s], 1); mbar_init(&x_empty[s], 1); }
    for (int g = 0; g < G; ++g) {
      mbar_init(&proj_full[g], 2); mbar_init(&tiles_full[g], kGroupThreads / 32); mbar_init(&s_full[g], 1);
      mbar_init(&p_full[g], kGroupThreads / 32); mbar_init(&o_full[g], 1); mbar_init(&qkv_free[g], 1);
      mbar_init(&so_ready[g], kGroupThreads / 32); mbar_init(&so_free[g], 1);
    }
    fence_barrier_init();
  }
  if (warp == kProducerWarp && lane == 0)
    for (int i = 0; i < 8; ++i) { tma_prefetch_desc(&P.x[0][i]); tma_prefetch_desc(&P.x[1][i]); tma_prefetch_desc(&P.x[2][i]); }
  if (warp == kProducerWarpKV && lane == 0)
    for (int i = 0; i < 8; ++i) { tma_prefetch_desc(&P.q[i]); tma_prefetch_desc(&P.k[i]); tma_prefetch_desc(&P.v[i]); }
  if (warp == kStoreWarp && lane == 0)
    for (int i = 0; i < 8; ++i) tma_prefetch_desc(&P.o[i]);
  if (warp == kMmaWarp) tmem_alloc<kTmemColsF>(tmem_slot);
  fence_proxy_async_smem();            // W and the zeroed ring must be visible to the tensor-core (async) proxy
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp >= kProducerWarp) {
    setmaxnreg_dec<kRegAuxF>();
    if (warp == kProducerWarp) {
      // ============================== TMA producer: schedule, pair descriptors, x tiles ==============================
      const BoxLayout<3> lay{{P.x[0], P.x[1], P.x[2]}, {0, kXPanel, 2 * kXPanel}, {kWinBytes, kWinBytes, kWinBytes}};
      BoxPlan<3> plan;
      // ring depth (kItemRing): entry n + 16 is written once x stage (n + 16) % 2 is free, i.e. after the projections of
      // pair n + 14, which waited for PV of every sub-item of pair n + 13: every group, and both store warps (one item
      // behind their groups), are past pair n.
      auto load_pair = [=, &P, &S, &plan](int n, const RingItem& it) {
        const int stage = n % kXStages, phase = (n / kXStages) & 1;
        if (it.cls != plan.cls) plan.build(S, it.cls, lane, lay);
        mbar_wait(&x_empty[stage], phase ^ 1);
        if (lane == 0) {
          ring.publish(n, it);                                          // published by the arrival below
          mbar_arrive_expect_tx(&x_full[stage], it.nvalid * 3 * kWinBytes);
        }
        __syncwarp();
        plan.issue<true>(S, it.ws[0], it.ws[1], it.nvalid, 0, sX + stage * kXStage, &x_full[stage], lane);
      };
      const int chunk = max(1, min(kChunkF, sc.n_items / ((int)gridDim.x * 8)));
      const int n = walk_queue(S, sc, sched_range_begin(sc, blockIdx.x, gridDim.x), P.work, chunk, lane, load_pair);
      const int stage = n % kXStages, phase = (n / kXStages) & 1;      // end marker
      mbar_wait(&x_empty[stage], phase ^ 1);
      if (lane == 0) {
        ring.publish_end(n);
        mbar_arrive(&x_full[stage]);
      }
      __syncwarp();
    } else if (warp == kMmaWarp) {
      // ============================== MMA issuer ==============================
      constexpr uint32_t idescX = umma_idesc_bf16(128, 96, 0, 0);    // x (K-major) x W_h (K-major)
      constexpr uint32_t idescS = umma_idesc_bf16(128, 128, 0, 0);   // [Q0;Q1] x [K0;K1] (both K-major)
      constexpr uint32_t idescO = umma_idesc_bf16(128, 32, 0, 1);    // P (TMEM) x V (MN-major)
      const uint64_t dK = umma_smem_desc(0, 0, 512, kSwz64);
      const uint64_t dV = umma_smem_desc(0, 8192, 512, kSwz64);
      const uint32_t x0 = smem_u32(sX) >> 4, w0 = smem_u32(sW) >> 4, op0 = smem_u32(sOp) >> 4;
      // projection nj needs the pair's x tile and PV(nj - G) complete (it overwrites that sub-item's S and P columns);
      // S ns needs the group's tiles; PV np needs P.  Each test below checks a phase that cannot yet have been overtaken.
      int total = 0x7fffffff;                                        // sub-items of this CTA: known at the end marker
      int nj = 0, ns = 0, np = 0;
      uint32_t idle = 0;
      while (np < total) {
        bool progressed = false;
        if (total == 0x7fffffff && nj < np + G) {
          const int pr = nj / G, h = nj - pr * G, xs = pr % kXStages;
          if ((h != 0 || mbar_test(&x_full[xs], (pr / kXStages) & 1)) && (nj < G || mbar_test(&o_full[h], (pr - 1) & 1))) {
            progressed = true;
            if (h == 0 && ring.read(pr).end()) {
              total = nj;
            } else {
              tcgen05_fence_after();
              if (elect_one()) {
                const uint64_t ax = dK + (x0 + xs * (kXStage >> 4)), bw = dK + (w0 + h * (kWHead >> 4));
#pragma unroll
                for (int ks = 0; ks < 6; ++ks)
                  umma_bf16_ss(tmem + h * kTmemGroup, ax + ((ks >> 1) * (kXPanel >> 4) + (ks & 1) * 2),
                               bw + ((ks >> 1) * (kWPanel >> 4) + (ks & 1) * 2), idescX, ks);
                umma_commit(&proj_full[h]);
                if (h == G - 1) umma_commit(&x_empty[xs]);
                mbar_arrive(&proj_full[h]);          // releases the pair descriptor this thread acquired through x_full
              }
              __syncwarp();
              ++nj;
            }
          }
        }
        if (ns < nj) {
          const int g = ns % G;
          if (mbar_test(&tiles_full[g], (ns / G) & 1)) {
            progressed = true;
            tcgen05_fence_after();
            if (elect_one()) {
              const uint64_t aq = dK + (op0 + g * (kOpSet >> 4)), bk = aq + (kOpTile >> 4);
              umma_bf16_ss(tmem + g * kTmemGroup, aq, bk, idescS, 0);
              umma_bf16_ss(tmem + g * kTmemGroup, aq + 2, bk + 2, idescS, 1);
              umma_commit(&s_full[g]);
            }
            __syncwarp();
            ++ns;
          }
        }
        if (np < ns) {
          const int g = np % G;
          if (mbar_test(&p_full[g], (np / G) & 1)) {
            progressed = true;
            tcgen05_fence_after();
            if (elect_one()) {
              const uint32_t tP = tmem + g * kTmemGroup, tO = tP + 128;
              const uint64_t bv = dV + (op0 + g * (kOpSet >> 4) + ((2 * kOpTile) >> 4));
#pragma unroll
              for (int ks = 0; ks < 8; ++ks) umma_bf16_ts(tO, tP + ks * 8, bv + ks * (1024 >> 4), idescO, ks);
              umma_commit(&o_full[g]);
            }
            __syncwarp();
            ++np;
          }
        }
        if (progressed) idle = 0;
        else if (++idle > (1u << 24)) __trap();    // a broken pipeline becomes a CUDA error, not a hang
      }
      // end markers, once every group has handed over P of its last sub-item (so none of them can miss a phase)
      if (elect_one())
        for (int g = 0; g < G; ++g) { mbar_arrive(&proj_full[g]); mbar_arrive(&proj_full[g]); }
      __syncwarp();
    } else if (warp == kStoreWarp) {
      // ============================== TMA store of o ==============================
      // Unlike the unfused kernel's store warp, a tile goes back to its group as soon as its stores have read it: the
      // group waits for it before draining its next projection (the tile is its Q tile), at the head of its chain, and
      // handing it back one item late made every group wait for the next group's epilogue.
      const BoxLayout<1> lay{{P.o}, {0}, {kWinBytes}};
      BoxPlan<1> plan;
      int n = 0;
      for (;; ++n) {
        const int g = n % G, kk = n / G;
        mbar_wait(&so_ready[g], kk & 1);
        if (kk >= *reinterpret_cast<volatile int*>(&sEnd[g])) break;
        const RingItem it = ring.read(kk);
        if (it.cls != plan.cls) plan.build(S, it.cls, lane, lay);
        plan.issue<false>(S, it.ws[0], it.ws[1], it.nvalid, g * kD, sOp + g * kOpSet, nullptr, lane);
        tma_store_commit();
        tma_store_wait_read<0>();
        __syncwarp();
        if (lane == 0) mbar_arrive(&so_free[g]);
      }
      tma_store_wait_all<0>();
    } else {
      // ============================== TMA store of the Q, K, V tiles to qkv ==============================
      const BoxLayout<3> lay{{P.q, P.k, P.v}, {0, kOpTile, 2 * kOpTile}, {kWinBytes, kWinBytes, kWinBytes}};
      BoxPlan<3> plan;
      for (int n = 0;; ++n) {
        const int g = n % G, kk = n / G;
        mbar_wait(&tiles_full[g], kk & 1);
        const RingItem it = ring.read(kk);
        if (it.end()) break;                         // group 0's farewell: every earlier sub-item is stored
        if (it.cls != plan.cls) plan.build(S, it.cls, lane, lay);
        plan.issue<false>(S, it.ws[0], it.ws[1], it.nvalid, g * kD, sOp + g * kOpSet, nullptr, lane);
        tma_store_commit();
        tma_store_wait_read<0>();
        __syncwarp();
        if (lane == 0) mbar_arrive(&qkv_free[g]);
      }
      tma_store_wait_all<0>();
    }
  } else {
    // ============================== softmax groups: group g = head g, one thread per row of the pair ==============================
    setmaxnreg_inc<kRegSoftmaxF>();
    const int g = warp >> 2, h = g;
    const int r = tid & 127;
    const int slot = r >> 6, i = r & 63;
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t tG = tmem + lane_base + g * kTmemGroup;
    const float hscale = COS ? __ldg(P.head_scale + h) * kLog2e : P.scale * kLog2e;
    float* tbl = sTbl + g * kN * kN;
    float* rkbuf = sRk + g * 128;
    uint8_t* tiles = sOp + g * kOpSet;
    const int rsw = (r >> 1) & 3;
    const float* bias_h = P.bias ? P.bias + (size_t)h * kN * kN : nullptr;

    int cls_loaded = -1;
    int kk = 0;
    for (;; ++kk) {
      mbar_wait(&proj_full[g], kk & 1);
      const RingItem it = ring.read(kk);
      if (it.end()) break;
      tcgen05_fence_after();
      const int cls = it.cls, gw = slot ? it.win[1] : it.win[0];
      const bool valid = slot < it.nvalid;
      if (cls != cls_loaded) {
        named_bar_sync(1 + g, kGroupThreads);
        build_class_table(tbl, kN, bias_h, sPos + cls * 64, sRid + cls * 64, MASK == MMN_MASK_SHIFT && cls != 0, r, kGroupThreads, 7);
        cls_loaded = cls;
      }
      const int ipos = sPos[cls * 64 + i];
      const int gwh = gw * kQkvHeads + h;

      // ---- drain the projection: + bias, bf16, swizzled rows of the Q, K, V tiles; norms from the rounded values
      mbar_wait(&so_free[g], (kk & 1) ^ 1);            // o of the group's previous sub-item has left the Q tile
      float ssq = 0.f, ssk = 0.f;
#pragma unroll
      for (int t = 0; t < 3; ++t) {
        uint32_t raw[32];
        tmem_ld_32x32b_x32(tG + t * 32, raw);
        tmem_ld_wait();
        uint32_t u[16];
        if (P.b) {
          const float4* bp = reinterpret_cast<const float4*>(P.b + t * kQkvC + h * kD);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b4 = __ldg(bp + j);
            u[2 * j] = pack_bf16x2(__uint_as_float(raw[4 * j]) + b4.x, __uint_as_float(raw[4 * j + 1]) + b4.y);
            u[2 * j + 1] = pack_bf16x2(__uint_as_float(raw[4 * j + 2]) + b4.z, __uint_as_float(raw[4 * j + 3]) + b4.w);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) u[j] = pack_bf16x2(__uint_as_float(raw[2 * j]), __uint_as_float(raw[2 * j + 1]));
        }
        uint8_t* row = tiles + t * kOpTile + r * 64;
#pragma unroll
        for (int c = 0; c < 4; ++c)
          *reinterpret_cast<uint4*>(row + ((c ^ rsw) << 4)) = make_uint4(u[4 * c], u[4 * c + 1], u[4 * c + 2], u[4 * c + 3]);
        if (COS && t == 0) ssq = sumsq_bf16x32(u);
        if (COS && t == 1) ssk = sumsq_bf16x32(u);
      }
      tcgen05_fence_before();
      fence_proxy_async_smem();                        // tiles visible to the MMA and the TMA stores
      mbar_arrive_warp(&tiles_full[g]);
      float a_i = hscale;
      if (COS) {
        const float rq = rsqrtf(fmaxf(ssq, 1e-24f)), rkk = rsqrtf(fmaxf(ssk, 1e-24f));
        a_i *= rq;
        rkbuf[r] = rkk;                                // single buffer: every thread read the last one before o_full
        if (valid) {
          float* rec = P.lse + P.slab + (long long)gwh * (3 * kN) + i;
          rec[0] = rq;
          rec[kN] = rkk;
        }
      }
      named_bar_sync(1 + g, kGroupThreads);            // rk (and a rebuilt table) visible to the group

      // ---- logits of this row's 64 keys: its own window's block of the N128 product
      mbar_wait(&s_full[g], kk & 1);
      tcgen05_fence_after();
      uint64_t s2[32];
      {
        uint32_t raw0[32], raw1[32];
        tmem_ld_32x32b_x32(tG + slot * 64, raw0);
        tmem_ld_32x32b_x32(tG + slot * 64 + 32, raw1);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) { s2[j] = pk2u(raw0[2 * j], raw0[2 * j + 1]); s2[16 + j] = pk2u(raw1[2 * j], raw1[2 * j + 1]); }
      }
      uint32_t pp[32];
      float mx, l;
      softmax_row<COS, MASK, 7>(s2, tbl + i * kN, i, rkbuf + slot * 64,
                                (MASK == MMN_MASK_TENSOR) ? P.mask + ((size_t)(gw % P.mask_windows) * kN + ipos) * kN : nullptr,
                                a_i, valid, pp, mx, l);
      // P over columns 0..63 as [P0 0] / [0 P1]: the projection overwrote the zero halves
      tmem_st_32x32b_x32(tG + slot * 32, pp);
      tmem_st_zero_x32(tG + (slot ^ 1) * 32);
      tmem_st_wait();
      tcgen05_fence_before();
      mbar_arrive_warp(&p_full[g]);

      const float lse2 = mx + __log2f(l), inv_l = __frcp_rn(l);
      if (valid) {
        P.lse[(long long)gwh * kN + ipos] = lse2 * kLn2;
        P.lse[P.slab + (long long)gwh * (3 * kN) + 2 * kN + i] = lse2;
      }

      // ---- O / l -> bf16 -> the Q tile (once the qkv stores have read it) -> o store warp
      mbar_wait(&o_full[g], kk & 1);
      tcgen05_fence_after();
      uint32_t oraw[32];
      tmem_ld_32x32b_x32(tG + 128, oraw);
      tmem_ld_wait();
      tcgen05_fence_before();
      mbar_wait(&qkv_free[g], kk & 1);
      o_row_to_smem(oraw, inv_l, tiles + r * 64, r);
      fence_proxy_async_smem();
      mbar_arrive_warp(&so_ready[g]);
    }
    // farewells: to the qkv store warp (its next tiles_full phase, whose descriptor is the end marker) and to the o
    // store warp (sEnd, once it has taken the last tile: two so_ready phases completing back to back would alias)
    mbar_arrive_warp(&tiles_full[g]);
    if (kk > 0) mbar_wait(&so_free[g], (kk - 1) & 1);
    if (r == 0) sEnd[g] = kk;
    mbar_arrive_warp(&so_ready[g]);
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc<kTmemColsF>(tmem);
}

// ------------------------------------------------------------------------------------------
// Host side
// ------------------------------------------------------------------------------------------
const char* qkv_fwd_why_not(const mmn_winattn_desc* d, int in_channels) {
  if (d->num_heads != kQkvHeads || d->head_dim != kD) return "the fused qkv kernel is built for 3 heads of 32 channels (C = 96)";
  if (in_channels != kQkvC) return "input channels differ from the attention width";
  return fwd_why_not(d);
}

int winattn_qkv_fwd(const mmn_winattn_desc* d, const void* x, const void* w, const float* b, const float* bias, const float* head_scale,
                    const float* mask, void* qkv, void* out, float* lse, void* workspace, cudaStream_t st, char* err, size_t errlen) {
  QkvFwdParams P;
  P.S = shape_from(d);
  P.sc = make_sched(P.S, d->batch);
  const char* xb = static_cast<const char*>(x);
  char* qb = static_cast<char*>(qkv);
  bool ok = reinterpret_cast<uintptr_t>(w) % 16 == 0;
  for (int p = 0; p < 3; ++p) ok = ok && make_window_maps(P.x[p], xb + p * kD * 2, kQkvC, d->batch, kD, P.S);
  ok = ok && make_window_maps(P.q, qb, 3 * kQkvC, d->batch, kQkvC, P.S) &&
       make_window_maps(P.k, qb + kQkvC * 2, 3 * kQkvC, d->batch, kQkvC, P.S) &&
       make_window_maps(P.v, qb + 2 * kQkvC * 2, 3 * kQkvC, d->batch, kQkvC, P.S) &&
       make_window_maps(P.o, out, kQkvC, d->batch, kQkvC, P.S);
  if (!ok) return tensor_map_failed(err, errlen);
  P.mask_windows = d->mask_windows > 0 ? d->mask_windows : 1;
  P.scale = d->scale;
  P.w = static_cast<const __nv_bfloat16*>(w); P.b = b;
  P.bias = bias; P.head_scale = head_scale; P.mask = mask; P.lse = lse;
  P.slab = (long long)P.S.n_windows * d->num_heads * kN;
  P.work = arm_work_counters(workspace, st, err, errlen);
  if (!P.work) return MMN_ERR_CUDA;

  // [cosine][mask kind]
  static void (*const kernels[6])(QkvFwdParams) = {
      winattn_qkv_fwd_tc_kernel<false, MMN_MASK_NONE>, winattn_qkv_fwd_tc_kernel<false, MMN_MASK_SHIFT>, winattn_qkv_fwd_tc_kernel<false, MMN_MASK_TENSOR>,
      winattn_qkv_fwd_tc_kernel<true, MMN_MASK_NONE>, winattn_qkv_fwd_tc_kernel<true, MMN_MASK_SHIFT>, winattn_qkv_fwd_tc_kernel<true, MMN_MASK_TENSOR>};
  int grid = num_sms_cached();
  if (grid > P.sc.n_items) grid = P.sc.n_items;
  return launch_variant(kernels, (d->score_kind == MMN_SCORE_COSINE ? 3 : 0) + d->mask_kind, kQkvSmemBytes, grid, kFwdThreads, P, st,
                        "winattn_qkv_fwd_tc_kernel", err, errlen);
}

}}  // namespace mmn::tc
