// winattn_tc_fwd.cuh -- shifted-window attention forward on the Blackwell tensor cores
// (tcgen05.mma + TMEM accumulators + TMA), bf16 in / bf16 out, fp32 softmax.
//
// Tuned shape: 64-token windows (4x4x4, 8x8, or 64 pre-windowed tokens), head_dim 32.
// A work item is a PAIR of windows of one wrap class x one head (tc_sched.cuh): 128 query rows
// = the 128 TMEM lanes.  A CTA serves one head and claims items at run time (ClassQueue).  512 threads,
// one CTA per SM, warp-specialised, THREE items in flight (softmax groups 0-2 take items n % 3):
//
//   warps 0-11  three softmax groups of four warps: ONE thread per query row, all 64 keys of its window.
//               tcgen05.ld the logits, multiply by the cosine normalisation x logit scale (or q scale), add
//               the per-class table (relative position bias + shift mask, pre-permuted to the tile's token
//               order, log2 domain), exp2 softmax in fp32 on register pairs, P (bf16) straight back into TMEM
//               (tcgen05.st) as the A operand of the second MMA; then O / l -> bf16 -> 64B-swizzled staging
//               tile.  No cross-thread exchange except the per-key norms (one named barrier per group and item).
//               Also writes lse and the per-window record (norms, log2 lse) the backward kernel reads back.
//   warp 12     TMA producer: schedule (atomic claims), item descriptors (shared-memory ring) and the Q tiles,
//               gathered straight out of the un-windowed, un-shifted (B,D,H,W,3C) tensor with 5-D tensor maps:
//               the cyclic shift is a coordinate offset, a window that wraps around the volume edge is fetched
//               as its 2/4/8 contiguous pieces (tc_window.cuh).  5-stage ring.
//   warp 15     TMA producer for the K and V tiles of the same items (follows the descriptor ring).
//   warp 13     MMA issuer: S = Q K^T as ONE M128 N64 K64 product per pair -- the two windows are
//               stacked along M and their channels along K, the cross terms multiply a shared
//               zero block ([Q0;0] x K0^T + [0;Q1] x K1^T), so the accumulator holds exactly the two
//               64x64 diagonal blocks in 64 TMEM columns; O = P V (M128 N32 K128, A = [P0 0; 0 P1] from TMEM).
//               Per group: S 64 + P 64 + O 32 TMEM columns.  Polls its two queues (S, PV) without blocking.
//   warp 14     TMA store: staging tile -> global through the same boxes (= window_reverse + roll back); a tile
//               goes back to its group one item late.
// Registers by setmaxnreg: softmax 136, the four single warps 104.
#pragma once

#include <cstdio>
#include <cstdlib>
#include <mutex>

#include "tc_sched.cuh"
#include "winattn_tc.h"
#include "zero_fill.h"

namespace mmn { namespace tc {

constexpr int kStagesF = 5;
constexpr int kWinBytes = 64 * 64;                 // one window's (64 tokens x 32 ch) bf16 tile
constexpr int kTile = 2 * kWinBytes;               // a pair's tile
constexpr int kQRegion = 3 * kWinBytes;            // Q0 | zero block | Q1
constexpr int kStageBytesF = kQRegion + 2 * kTile; // + K0 K1 + V0 V1
constexpr int kGroupThreads = 128;
constexpr int kGroupsF = 3;                        // softmax groups = items in flight
constexpr int kProducerWarp = 4 * kGroupsF, kMmaWarp = kProducerWarp + 1, kStoreWarp = kProducerWarp + 2, kProducerWarpKV = kProducerWarp + 3;
constexpr int kFwdThreads = 32 * (kProducerWarp + 4);   // 4 warpgroups: 3 softmax groups + {Q producer, MMA, store, K/V producer}
constexpr int kRegSoftmaxF = 136, kRegAuxF = 104;  // setmaxnreg: 384 * 136 + 128 * 104 = 512 * 128
constexpr int kTblLd = 68;                         // padded row of the shared table (conflict-free float4 rows)
constexpr int kTmemColsF = 512;                    // group g: S at 160 g (64 columns), P at 160 g + 64 (64), O at 160 g + 128 (32)
constexpr int kTmemGroup = 160;
constexpr int kItemRing = 16;                      // item descriptors published by the TMA producer (see the ring-depth note there)
constexpr int kChunkF = 16;                        // most items a CTA claims per atomic
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

// Debug tracing: buf[(role*32 + item - item0)*16 + ev] = clock64() of CTA `cta`; buf[kTraceCtaOfs + 2*cta + {0,1}] =
// globaltimer at the start / end of every CTA (load balance).  Which CTA and which 32 items: MMN_TC_TRACE_CTA / _ITEM0.
constexpr int kTraceCtaOfs = 5 * 32 * 16;
constexpr int kTraceWords = kTraceCtaOfs + 2 * 1024;
struct TraceCfg { long long* buf; int cta; int item0; };
__device__ __forceinline__ long long global_ns() { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }

struct FwdParams {
  CUtensorMap q[8], k[8], v[8], o[8];   // one box shape per wrap class
  WinShape S;
  Sched sc;
  int nH, per_head;
  int mask_windows;
  float scale;
  const float* bias;
  const float* head_scale;
  const float* mask;
  float* lse;         // (B*nW, nH, 64) log-sum-exp by window position, then one record per window and head for the backward
  long long slab;     //   kernel, (B*nW, nH, 3, 64) in the tile's (piece-major) row order: 1/max(||q||,eps) | 1/max(||k||,eps) |
                      //   log2-domain lse (one 768-byte bulk copy per window there); slab = B*nW*nH*64
  int* work;          // dynamic schedule counters (tc_sched.cuh: ClassQueue): this launch's own, zeroed before it
  TraceCfg trace;     // debug: per-phase clock64 stamps of one CTA (MMN_TC_TRACE=<file>), else buf == null
};

// trace[(role*32 + item)*16 + ev]; roles: 0 group A warp 0, 1 group B warp 4, 2 producer, 3 MMA, 4 store
__device__ __forceinline__ void trace_stamp(const TraceCfg& t, int role, int item, int ev) {
  if (t.buf && (int)blockIdx.x == t.cta && (threadIdx.x & 31) == 0 && (unsigned)(item - t.item0) < 32u)
    t.buf[(role * 32 + item - t.item0) * 16 + ev] = clock64();
}
__device__ __forceinline__ void trace_cta_time(const TraceCfg& t, int which) {
  if (t.buf && threadIdx.x == 0 && blockIdx.x < 1024) t.buf[kTraceCtaOfs + 2 * blockIdx.x + which] = global_ns();
}
// Both kernels: the stamps are compiled in only with -DMMN_TC_TRACING (tools/build_variant.sh trace winattn_tc -DMMN_TC_TRACING,
// then MMN_LIB=<that build> tools/trace_{fwd,bwd}.py); they cost the backward 20 % and the forward 7 %.  (Round 1's forward
// kept them in production because its never-taken branches happened to stop ptxas from interleaving the softmax phases;
// with the current phase structure the build without them is the faster one: 0.182 -> 0.170 ms at BASELINE cfg2.)
__device__ __forceinline__ void trace_ev(const TraceCfg& trace, int role, int item, int ev) {
#ifdef MMN_TC_TRACING
  trace_stamp(trace, role, item, ev);
#endif
}
__device__ __forceinline__ void trace_evf(const TraceCfg& trace, int role, int item, int ev) { trace_ev(trace, role, item, ev); }

// sum of squares of 32 bf16 values packed in pairs (u[j] = elements 2j, 2j + 1), in one fixed order: one chain of
// (low, high) pairs per 8-element chunk, chunks added pairwise.  The fused qkv kernel computes its norms from registers
// with it and gets the same bits as row_sumsq over the stored row.
__device__ __forceinline__ float sumsq_bf16x32(const uint32_t (&u)[16]) {
  uint64_t ss[4] = {0ull, 0ull, 0ull, 0ull};
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const uint64_t x = pk2u(u[4 * c + e] << 16, u[4 * c + e] & 0xffff0000u);
      ss[c] = fma2(x, x, ss[c]);
    }
  float lo, hi;
  upk2(add2(add2(ss[0], ss[1]), add2(ss[2], ss[3])), lo, hi);
  return lo + hi;
}

// sum of squares of one 64-byte bf16 row.  `row` = the row's index in its tile: chunk c is read at its
// swizzled place, which also spreads the lanes of a warp over all banks (plain order is a 4-way conflict).
__device__ __forceinline__ float row_sumsq(const uint8_t* rowp, int row) {
  const int sw = (row >> 1) & 3;
  uint32_t u[16];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const uint4 a = *reinterpret_cast<const uint4*>(rowp + ((c ^ sw) << 4));
    u[4 * c] = a.x; u[4 * c + 1] = a.y; u[4 * c + 2] = a.z; u[4 * c + 3] = a.w;
  }
  return sumsq_bf16x32(u);
}

// One query row's softmax over its window's 64 keys, shared by both forward kernels.  s2: the row's logits as fp32
// pairs (overwritten); trow: its row of the class table (float4 j4 stored at j4 ^ (row & TSWZ)); krow: the 64 keys'
// 1/||k|| (COS); mrow: its mask row (MMN_MASK_TENSOR).  Out: P = exp2(s - max) as bf16 pairs (zero for an invalid
// slot), the max and the sum.
template <bool COS, int MASK, int TSWZ>
__device__ __forceinline__ void softmax_row(uint64_t (&s2)[32], const float* trow_f, int row, const float* krow_f, const float* mrow,
                                            float a_i, bool valid, uint32_t (&pp)[32], float& mx, float& l) {
  {
    const float4* trow = reinterpret_cast<const float4*>(trow_f);
    const float4* krow = reinterpret_cast<const float4*>(krow_f);
    const uint64_t a2 = pk2(a_i, a_i);
#pragma unroll
    for (int j4 = 0; j4 < 16; ++j4) {
      float4 tt = trow[j4 ^ (row & TSWZ)];
      if (MASK == MMN_MASK_TENSOR) {
        const float4 mm = __ldg(reinterpret_cast<const float4*>(mrow) + j4);
        tt.x = fmaf(mm.x, kLog2e, tt.x); tt.y = fmaf(mm.y, kLog2e, tt.y); tt.z = fmaf(mm.z, kLog2e, tt.z); tt.w = fmaf(mm.w, kLog2e, tt.w);
      }
      if (COS) {
        const float4 kv = krow[j4];
        s2[j4 * 2 + 0] = fma2(s2[j4 * 2 + 0], mul2(pk2(kv.x, kv.y), a2), pk2(tt.x, tt.y));
        s2[j4 * 2 + 1] = fma2(s2[j4 * 2 + 1], mul2(pk2(kv.z, kv.w), a2), pk2(tt.z, tt.w));
      } else {
        s2[j4 * 2 + 0] = fma2(s2[j4 * 2 + 0], a2, pk2(tt.x, tt.y));
        s2[j4 * 2 + 1] = fma2(s2[j4 * 2 + 1], a2, pk2(tt.z, tt.w));
      }
    }
  }
  {
    float m8[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) upk2(s2[j], m8[2 * j], m8[2 * j + 1]);
#pragma unroll
    for (int j = 4; j < 32; j += 2) {                // FMNMX3: two new values per instruction
      float a, b, c, d;
      upk2(s2[j], a, b); upk2(s2[j + 1], c, d);
      const int ch = (j >> 1) & 7;
      m8[ch] = fmaxf(fmaxf(m8[ch], a), b);
      m8[(ch + 4) & 7] = fmaxf(fmaxf(m8[(ch + 4) & 7], c), d);
    }
    mx = fmaxf(fmaxf(fmaxf(m8[0], m8[1]), fmaxf(m8[2], m8[3])), fmaxf(fmaxf(m8[4], m8[5]), fmaxf(m8[6], m8[7])));
  }
  {
    const uint64_t nmx2 = pk2(-mx, -mx);
    uint64_t l2[4] = {0ull, 0ull, 0ull, 0ull};
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      float a, b;
      upk2(add2(s2[j], nmx2), a, b);
      a = fast_exp2(a); b = fast_exp2(b);
      l2[j & 3] = add2(l2[j & 3], pk2(a, b));
      pp[j] = valid ? pack_bf16x2(a, b) : 0u;
    }
    float la, lb;
    upk2(add2(add2(l2[0], l2[1]), add2(l2[2], l2[3])), la, lb);
    l = la + lb;
  }
}

// O / l -> bf16 -> row r of a 64B-swizzled (128 x 32) staging tile
__device__ __forceinline__ void o_row_to_smem(const uint32_t (&oraw)[32], float inv_l, uint8_t* obuf, int r) {
  const uint64_t inv2 = pk2(inv_l, inv_l);
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint4 v4 = make_uint4(pack_bf16x2(mul2(pk2u(oraw[c * 8 + 0], oraw[c * 8 + 1]), inv2)), pack_bf16x2(mul2(pk2u(oraw[c * 8 + 2], oraw[c * 8 + 3]), inv2)),
                          pack_bf16x2(mul2(pk2u(oraw[c * 8 + 4], oraw[c * 8 + 5]), inv2)), pack_bf16x2(mul2(pk2u(oraw[c * 8 + 6], oraw[c * 8 + 7]), inv2)));
    *reinterpret_cast<uint4*>(obuf + ((c ^ ((r >> 1) & 3)) << 4)) = v4;
  }
}

// COS: cosine attention (else scaled dot product); MASK: MMN_MASK_NONE / _SHIFT / _TENSOR.
template <bool COS, int MASK>
__global__ void __launch_bounds__(kFwdThreads, 1)
winattn_fwd_tc_kernel(const __grid_constant__ FwdParams P) {
  constexpr int G = kGroupsF;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // swizzle atoms need 1024-B alignment
  uint8_t* sStage = smem;                                 // kStagesF x (Q0|Z|Q1 | K0 K1 | V0 V1)
  uint8_t* sO = sStage + kStagesF * kStageBytesF;         // [G] output staging tile
  float* sTbl = reinterpret_cast<float*>(sO + G * kTile); // [G][64][kTblLd]
  float* sRk = sTbl + G * kN * kTblLd;                    // [G][2][128] per-key 1/||k|| (double-buffered over the group's items)
  uint8_t* sPos = reinterpret_cast<uint8_t*>(sRk + G * 256);  // [8 wrap classes][64]: tile row -> window position
  uint8_t* sRid = sPos + 512;                             // [8 wrap classes][64]: window position -> shift-mask region id
  const ItemRing<kItemRing> ring{reinterpret_cast<int4*>(sRid + 512)};      // item descriptors (tc_sched.cuh)
  int* sEnd = reinterpret_cast<int*>(sRid + 512 + ring.kBytes);   // [G] items group g has produced when it left its loop (else INT_MAX)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sEnd + 4);
  uint64_t* full = bars;                                  // [kStagesF] TMA -> MMA, softmax
  uint64_t* empty = bars + kStagesF;                      // [kStagesF] MMA -> TMA
  uint64_t* s_full = bars + 2 * kStagesF;                 // [G] S in TMEM
  uint64_t* p_full = s_full + G;                          // [G] P in TMEM (one arrival per warp)
  uint64_t* o_full = s_full + 2 * G;                      // [G] O in TMEM
  uint64_t* so_ready = s_full + 3 * G;                    // [G] staging tile written (one arrival per warp)
  uint64_t* so_free = s_full + 4 * G;                     // [G] staging tile drained by the store warp
  uint64_t* desc_ready = s_full + 5 * G;                  // [kStagesF] item descriptor published (Q producer -> K/V producer)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(desc_ready + kStagesF);

  const WinShape& S = P.S;
  const Sched& sc = P.sc;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int h = blockIdx.x % P.nH;

  // ---- one-time setup: zero the operand tiles (zero blocks stay zero for the whole kernel; the rest must
  // not hold NaN bit patterns, because cross terms multiply stale tiles by the zero blocks)
  for (int i = tid; i < (kStagesF * kStageBytesF) / 16; i += kFwdThreads)
    reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  fill_class_luts(S, sPos, sRid, tid, kFwdThreads);
  if (tid == 0) {
    for (int g = 0; g < G; ++g) sEnd[g] = 0x7fffffff;
    for (int s = 0; s < kStagesF; ++s) { mbar_init(&full[s], 2); mbar_init(&empty[s], 1); mbar_init(&desc_ready[s], 1); }
    for (int g = 0; g < G; ++g) {
      mbar_init(&s_full[g], 1); mbar_init(&p_full[g], kGroupThreads / 32); mbar_init(&o_full[g], 1);
      mbar_init(&so_ready[g], kGroupThreads / 32); mbar_init(&so_free[g], 1);
    }
    fence_barrier_init();
  }
  if (warp == kProducerWarp && lane == 0)
    for (int i = 0; i < 8; ++i) tma_prefetch_desc(&P.q[i]);
  if (warp == kProducerWarpKV && lane == 0)
    for (int i = 0; i < 8; ++i) { tma_prefetch_desc(&P.k[i]); tma_prefetch_desc(&P.v[i]); }
  if (warp == kStoreWarp && lane == 0)
    for (int i = 0; i < 8; ++i) tma_prefetch_desc(&P.o[i]);
  if (warp == kMmaWarp) tmem_alloc<kTmemColsF>(tmem_slot);
  fence_proxy_async_smem();            // zeroed tiles must be visible to the tensor-core (async) proxy
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *tmem_slot;
  trace_cta_time(P.trace, 0);

  if (warp >= kProducerWarp) {
    setmaxnreg_dec<kRegAuxF>();
    if (warp == kProducerWarp) {
      // ============================== TMA producer (schedule, descriptors, Q tiles) ==============================
      // every lane runs the loop; lane l issues boxes l, l + 32 of the item (BoxPlan).  The K and V tiles of the same items
      // are issued by a second warp that follows the descriptor ring (one warp issuing all six boxes of an item, ~65
      // cycles per box plus the cursor arithmetic, was what bounded the kernel).
      const BoxLayout<1> lay{{P.q}, {0}, {2 * kWinBytes}};
      BoxPlan<1> plan;
      // Dynamic schedule (tc_sched.cuh: ClassQueue): chunks of kChunkF items of this head, home class first.
      // Every other warp learns its items from the descriptor ring (published by the full[] arrival).  Ring
      // depth: entry n + 16 is written only once stage (n + 16) % kStagesF is free, i.e. after PV(n + 11) has completed,
      // so its group has long finished item n + 8 and with it waited for the store of item n + 5 (so_free): every
      // consumer of entry n, the store warp included, has read it.
      auto load_item = [=, &P, &S, &plan](int n, const RingItem& it) {
        const int stage = n % kStagesF, phase = (n / kStagesF) & 1;
        if (it.cls != plan.cls) plan.build(S, it.cls, lane, lay);
        trace_evf(P.trace, 2, n, 0);
        mbar_wait(&empty[stage], phase ^ 1);
        trace_evf(P.trace, 2, n, 1);
        if (lane == 0) {
          ring.publish(n, it);                                          // published by the arrivals below
          mbar_arrive(&desc_ready[stage]);
          mbar_arrive_expect_tx(&full[stage], it.nvalid * kWinBytes);
        }
        __syncwarp();
        plan.issue<true>(S, it.ws[0], it.ws[1], it.nvalid, h * kD, sStage + stage * kStageBytesF, &full[stage], lane);
        trace_evf(P.trace, 2, n, 2);
      };
      // claims of up to kChunkF items (each costs the producer a seek with integer divisions), an eighth of a CTA's share at most
      const int chunk = max(1, min(kChunkF, sc.n_items / (P.per_head * 8)));
      int n = walk_queue(S, sc, sched_range_begin(sc, blockIdx.x / P.nH, P.per_head), P.work + h * 8, chunk, lane, load_item);
      // one end marker per softmax group (the MMA warp stops at the first)
      for (int e = 0; e < G; ++e, ++n) {
        const int stage = n % kStagesF, phase = (n / kStagesF) & 1;
        mbar_wait(&empty[stage], phase ^ 1);
        if (lane == 0) {
          ring.publish_end(n);
          mbar_arrive(&desc_ready[stage]);
          mbar_arrive(&full[stage]);
        }
        __syncwarp();
      }
    } else if (warp == kMmaWarp) {
      // ============================== MMA issuer ==============================
      constexpr uint32_t idescS = umma_idesc_bf16(128, 64, 0, 0);    // [Q0;0],[0;Q1] (K-major) x K0,K1 (K-major)
      constexpr uint32_t idescO = umma_idesc_bf16(128, 32, 0, 1);    // P (TMEM: [P0 0; 0 P1], K-major) x V (MN-major)
      // descriptors: everything but the 14-bit start-address field is loop-invariant, and adding (bytes >> 4)
      // to a descriptor moves its start address -- one add per operand instead of rebuilding it
      const uint64_t dQK = umma_smem_desc(0, 0, 512, kSwz64);        // Q / K tiles, K-major
      const uint64_t dV = umma_smem_desc(0, 8192, 512, kSwz64);      // V tile, MN-major
      const uint32_t stage0 = smem_u32(sStage) >> 4;
      // Two queues served in turn, neither blocking the other: S(ns) needs item ns's tiles (full[]) and its group's S
      // buffer back (true once PV(ns - G) has been issued: the group wrote P after reading S); PV(np) needs P(np).
      // A warp that waited for the tiles of S(n + G) right after PV(n) held up PV(n + 1) whenever the loads ran late.
      int total = 0x7fffffff;                                        // items of this CTA: known once the end marker shows up
      int ns = 0, np = 0;
      uint32_t idle = 0;
      while (np < total) {
        bool progressed = false;
        if (total == 0x7fffffff && ns < np + G) {
          const int stage = ns % kStagesF, phase = (ns / kStagesF) & 1;
          if (mbar_test(&full[stage], phase)) {
            progressed = true;
            if (ring.read(ns).end()) {
              total = ns;
            } else {
              tcgen05_fence_after();
              if (elect_one()) {
                const uint64_t aq = dQK + (stage0 + stage * (kStageBytesF >> 4)), bk = aq + (kQRegion >> 4);
                const uint32_t tS = tmem + (ns % G) * kTmemGroup;
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)      // ks 0,1: window 0's channels; ks 2,3: window 1's
                  umma_bf16_ss(tS, aq + ((ks >> 1) * (kWinBytes >> 4) + (ks & 1) * 2), bk + ((ks >> 1) * (kWinBytes >> 4) + (ks & 1) * 2), idescS, ks);
                umma_commit(&s_full[ns % G]);
              }
              __syncwarp();
              ++ns;
            }
          }
        }
        if (np < ns) {
          const int g = np % G, kk = np / G, stage = np % kStagesF;
          if (mbar_test(&p_full[g], kk & 1)) {     // the group has read S(np) out and written P(np)
            progressed = true;
            trace_evf(P.trace, 3, np, 1);
            tcgen05_fence_after();
            if (elect_one()) {
              const uint32_t tP = tmem + g * kTmemGroup + 64, tO = tmem + g * kTmemGroup + 128;
              const uint64_t bv = dV + (stage0 + stage * (kStageBytesF >> 4) + ((kQRegion + kTile) >> 4));
#pragma unroll
              for (int ks = 0; ks < 8; ++ks)      // 16 keys (8 TMEM columns of P) per step; ks < 4: window 0's keys
                umma_bf16_ts(tO, tP + ks * 8, bv + ks * (1024 >> 4), idescO, ks);
              umma_commit(&o_full[g]);
              umma_commit(&empty[stage]);
            }
            __syncwarp();
            trace_evf(P.trace, 3, np, 2);
            ++np;
          }
        }
        if (progressed) idle = 0;
        else if (++idle > (1u << 24)) __trap();    // a broken pipeline becomes a CUDA error, not a hang
      }
    } else if (warp == kStoreWarp) {
      // ============================== TMA store ==============================
      const BoxLayout<1> lay{{P.o}, {0}, {kWinBytes}};
      BoxPlan<1> plan;
      // A tile goes back to its group one item late: the stores of item n are issued, then the warp waits only for the
      // bulk group before (item n - 1) to have been read out of shared memory -- the read latency of one item's stores
      // hides under the next item's issue.
      int n = 0;
      for (;; ++n) {
        const int g = n % G, kk = n / G;
        trace_evf(P.trace, 4, n, 0);
        mbar_wait(&so_ready[g], kk & 1);
        if (kk >= *reinterpret_cast<volatile int*>(&sEnd[g])) break;   // the group left its loop: that arrival was its farewell
        trace_evf(P.trace, 4, n, 1);
        const RingItem it = ring.read(n);
        if (it.cls != plan.cls) plan.build(S, it.cls, lane, lay);
        plan.issue<false>(S, it.ws[0], it.ws[1], it.nvalid, h * kD, sO + g * kTile, nullptr, lane);
        tma_store_commit();
        tma_store_wait_read<1>();          // per thread: its boxes of item n - 1 have been read
        __syncwarp();
        if (lane == 0 && n > 0) mbar_arrive(&so_free[(n - 1) % G]);
        trace_evf(P.trace, 4, n, 2);
      }
      tma_store_wait_read<0>();
      __syncwarp();
      if (lane == 0 && n > 0) mbar_arrive(&so_free[(n - 1) % G]);
      tma_store_wait_all<0>();
    } else {
      // ============================== TMA producer (K and V tiles) ==============================
      const BoxLayout<2> lay{{P.k, P.v}, {kQRegion, kQRegion + kTile}, {kWinBytes, kWinBytes}};
      BoxPlan<2> plan;
      int ends = 0;
      for (int n = 0; ends < G; ++n) {
        const int stage = n % kStagesF, phase = (n / kStagesF) & 1;
        mbar_wait(&desc_ready[stage], phase);             // the Q producer has waited for the stage and published the item
        const RingItem it = ring.read(n);
        if (it.end()) {                                   // end marker: complete the phase for its readers
          if (lane == 0) mbar_arrive(&full[stage]);
          __syncwarp();
          ++ends;
          continue;
        }
        if (it.cls != plan.cls) plan.build(S, it.cls, lane, lay);
        if (lane == 0) mbar_arrive_expect_tx(&full[stage], it.nvalid * 2 * kWinBytes);
        __syncwarp();
        plan.issue<true>(S, it.ws[0], it.ws[1], it.nvalid, h * kD, sStage + stage * kStageBytesF, &full[stage], lane);
      }
    }
  } else {
    // ============================== softmax / epilogue: group g = warp / 4, one thread per query row ==============================
    setmaxnreg_inc<kRegSoftmaxF>();
    const int g = warp >> 2;
    const int r = tid & 127;
    const int slot = r >> 6, i = r & 63;
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t tS = tmem + lane_base + g * kTmemGroup, tP = tS + 64 + slot * 32, tO = tS + 128;
    const float hscale = COS ? __ldg(P.head_scale + h) * kLog2e : P.scale * kLog2e;
    float* tbl = sTbl + g * kN * kTblLd;
    uint8_t* obuf = sO + g * kTile + r * 64;                          // this thread's staging row
    const float* bias_h = P.bias ? P.bias + (size_t)h * kN * kN : nullptr;
    const int trole = (warp & 3) == 0 && g < 2 ? g : -1;
#define TR(item, ev) do { if (trole >= 0) trace_evf(P.trace, trole, item, ev); } while (0)

    // P lives in TMEM as the A operand of the second MMA: row = lane, two bf16 per column, K = the pair's 128 keys.
    // A row of window 0 is [P0_i | 0], a row of window 1 [0 | P1_i]: the zero halves are written once, here.
    {
      uint32_t z[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) z[j] = 0u;
      tmem_st_32x32b_x32(tS + 64, z);
      tmem_st_32x32b_x32(tS + 96, z);
      tmem_st_wait();
    }

    int cls_loaded = -1;
    int kk = 0;
    for (int n = g;; n += G, ++kk) {
      const int stage = n % kStagesF, phase = (n / kStagesF) & 1;
      TR(n, 0);
      mbar_wait(&full[stage], phase);
      const RingItem it = ring.read(n);                 // written by the producer before it armed full[stage]
      if (it.end()) break;
      const int cls = it.cls, gw = slot ? it.win[1] : it.win[0];
      const bool valid = slot < it.nvalid;
      if (cls != cls_loaded) {                          // rare: a CTA sees few classes (ClassQueue)
        named_bar_sync(1 + g, kGroupThreads);           // everyone is done reading the old table
        build_class_table(tbl, kTblLd, bias_h, sPos + cls * 64, sRid + cls * 64, MASK == MMN_MASK_SHIFT && cls != 0, r, kGroupThreads);
        cls_loaded = cls;
      }
      const int ipos = sPos[cls * 64 + i];              // window position of this thread's query row
      const int gwh = gw * P.nH + h;
      const uint8_t* base = sStage + stage * kStageBytesF;
      float* rkbuf = sRk + (g * 2 + (kk & 1)) * 128;
      TR(n, 1);
      float a_i = hscale;
      if (COS) {
        const float ssq = row_sumsq(base + slot * 2 * kWinBytes + i * 64, i);
        const float ssk = row_sumsq(base + kQRegion + r * 64, i);
        const float rq = rsqrtf(fmaxf(ssq, 1e-24f)), rkk = rsqrtf(fmaxf(ssk, 1e-24f));
        a_i *= rq;                                       // 1 / max(||q||, 1e-12) x logit scale x log2(e)
        rkbuf[r] = rkk;
        if (valid) {                                     // kept for the backward kernel (it reads them with one bulk copy per window)
          float* rec = P.lse + P.slab + (long long)gwh * (3 * kN) + i;    // [window][head][1/|q| | 1/|k| | lse log2][64 tile rows]
          rec[0] = rq;
          rec[kN] = rkk;
        }
      }
      named_bar_sync(1 + g, kGroupThreads);             // rk (and a rebuilt table) visible to the group
      TR(n, 2);

      // ---- logits of this row's 64 keys
      mbar_wait(&s_full[g], kk & 1);
      tcgen05_fence_after();
      TR(n, 3);
      uint64_t s2[32];                                   // this row's 64 logits as fp32 pairs
      {
        uint32_t raw0[32], raw1[32];
        tmem_ld_32x32b_x32(tS, raw0);
        tmem_ld_32x32b_x32(tS + 32, raw1);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) { s2[j] = pk2u(raw0[2 * j], raw0[2 * j + 1]); s2[16 + j] = pk2u(raw1[2 * j], raw1[2 * j + 1]); }
      }
      TR(n, 4);
      uint32_t pp[32];
      float mx, l;
      softmax_row<COS, MASK, 0>(s2, tbl + i * kTblLd, i, rkbuf + slot * 64,
                                (MASK == MMN_MASK_TENSOR) ? P.mask + ((size_t)(gw % P.mask_windows) * kN + ipos) * kN : nullptr,
                                a_i, valid, pp, mx, l);
      TR(n, 5);
      tmem_st_32x32b_x32(tP, pp);
      tmem_st_wait();
      tcgen05_fence_before();
      mbar_arrive_warp(&p_full[g]);
      TR(n, 6);

      // ---- while the second MMA runs: log-sum-exp out
      const float lse2 = mx + __log2f(l), inv_l = __frcp_rn(l);
      if (valid) {
        P.lse[(long long)gwh * kN + ipos] = lse2 * kLn2;
        P.lse[P.slab + (long long)gwh * (3 * kN) + 2 * kN + i] = lse2;
      }

      // ---- O / l -> bf16 -> staging tile -> store warp
      mbar_wait(&o_full[g], kk & 1);
      tcgen05_fence_after();
      TR(n, 7);
      uint32_t oraw[32];
      tmem_ld_32x32b_x32(tO, oraw);
      tmem_ld_wait();
      tcgen05_fence_before();
      mbar_wait(&so_free[g], (kk & 1) ^ 1);              // the store warp has drained this group's staging tile
      o_row_to_smem(oraw, inv_l, obuf, r);
      fence_proxy_async_smem();
      mbar_arrive_warp(&so_ready[g]);
      TR(n, 8);
    }
    // farewell to the store warp: this group has produced kk tiles.  The store warp must have taken the last one
    // first -- two so_ready phases completing back to back would alias in its parity wait.
    if (kk > 0) mbar_wait(&so_free[g], (kk - 1) & 1);
    if (r == 0) sEnd[g] = kk;
    mbar_arrive_warp(&so_ready[g]);
#undef TR
  }

  tcgen05_fence_before();
  __syncthreads();
  trace_cta_time(P.trace, 1);
  if (warp == kMmaWarp) tmem_dealloc<kTmemColsF>(tmem);
}

constexpr size_t kFwdSmemBytes = 1024 /*align slack*/ + kStagesF * kStageBytesF + kGroupsF * kTile + kGroupsF * kN * kTblLd * 4 +
                                 kGroupsF * 256 * 4 + 1024 + ItemRing<kItemRing>::kBytes + 16 + (3 * kStagesF + 5 * kGroupsF + 1) * 8;

// ------------------------------------------------------------------------------------------
// Host side
// ------------------------------------------------------------------------------------------
const char* fwd_why_not(const mmn_winattn_desc* d) {
  if (d->io_dtype != MMN_DT_BF16) return "io dtype is not bf16";
  if (d->head_dim != kD) return "head_dim != 32";
  if (d->num_heads * 8 > kWorkDone) return "more than 63 heads";
  if (d->dropout_p > 0.f) return "attention dropout is only implemented in the generic path";
  WinShape g = shape_from(d);
  if (g.win[0] * g.win[1] * g.win[2] != kN) return "window does not hold 64 tokens";
  for (int a = 0; a < 3; ++a)
    if (g.shift[a] != 0 && (2 * g.shift[a] != g.win[a] || g.nwin[a] < 2)) return "shift is neither 0 nor window/2";
  // a mask tensor is addressed by window position; tiles of wrapped windows hold their tokens piece-major, and the kernels
  // read mask rows in tile order -- correct only while no window wraps (the modules pass tensors for pre-windowed calls only)
  if (d->mask_kind == MMN_MASK_TENSOR && (g.shift[0] | g.shift[1] | g.shift[2])) return "mask tensor together with a cyclic shift";
  if (d->q_row_stride % 8 || d->k_row_stride % 8 || d->v_row_stride % 8 || d->o_row_stride % 8) return "row stride not 16-byte aligned";
  if (!encode_fn()) return "cuTensorMapEncodeTiled unavailable";
  return nullptr;
}

inline void dump_trace(long long* dev, const char* path, cudaStream_t st) {
  static long long host[kTraceWords];
  cudaStreamSynchronize(st);
  cudaMemcpy(host, dev, sizeof(host), cudaMemcpyDeviceToHost);
  cudaFree(dev);
  if (FILE* f = fopen(path, "w")) {
    for (int role = 0; role < 5; ++role)
      for (int item = 0; item < 32; ++item) {
        fprintf(f, "%d %d", role, item);
        for (int ev = 0; ev < 16; ++ev) fprintf(f, " %lld", host[(role * 32 + item) * 16 + ev]);
        fprintf(f, "\n");
      }
    for (int cta = 0; cta < 1024; ++cta)
      if (host[kTraceCtaOfs + 2 * cta]) fprintf(f, "cta %d %lld %lld\n", cta, host[kTraceCtaOfs + 2 * cta], host[kTraceCtaOfs + 2 * cta + 1]);
    fclose(f);
  }
}
inline TraceCfg trace_setup(const char* path, cudaStream_t st) {
  TraceCfg t{nullptr, 0, 0};
  if (path && *path) {
    cudaMalloc(&t.buf, kTraceWords * sizeof(long long));
    cudaMemsetAsync(t.buf, 0, kTraceWords * sizeof(long long), st);
    const char* cta = getenv("MMN_TC_TRACE_CTA");        // which CTA to trace (default 0)
    const char* it0 = getenv("MMN_TC_TRACE_ITEM0");      // first of the 32 traced items (default 0)
    t.cta = cta ? atoi(cta) : 0;
    t.item0 = it0 ? atoi(it0) : 0;
  }
  return t;
}

// Work counters of the dynamic schedule (tc_sched.cuh: ClassQueue): kWorkSlotInts ints that belong to ONE launch -- the
// caller's `workspace` -- zeroed on the launch's stream right before the kernel (by a one-block kernel: zero_fill.h).  Nothing
// is shared between launches, so launches on different streams, captured graphs replayed side by side and any number
// of launches in flight are independent by construction.
inline int* arm_work_counters(void* workspace, cudaStream_t st, char* err, size_t errlen) {
  if (!workspace || reinterpret_cast<uintptr_t>(workspace) % 4) { snprintf(err, errlen, "workspace missing or misaligned"); return nullptr; }
  if (mmn::zero_words_async(workspace, kWorkSlotInts, st) != cudaSuccess) {       // a kernel, not a memset node: zero_fill.h
    snprintf(err, errlen, "zeroing the work counters: %s", cudaGetErrorString(cudaGetLastError()));
    return nullptr;
  }
  return static_cast<int*>(workspace);
}

inline int tensor_map_failed(char* err, size_t errlen) {
  snprintf(err, errlen, "cuTensorMapEncodeTiled failed (pointer alignment or strides)");
  return MMN_ERR_CUDA;
}

// Launches kernels[variant] of a table of one kernel's template instantiations and reports a launch error under `name`.  The
// first launch through a table raises the dynamic shared-memory limit of all its variants to `smem` (one table per
// parameter type: the flag is per instantiation of this template).
template <class Params, int N>
inline int launch_variant(void (*const (&kernels)[N])(Params), int variant, size_t smem, int grid, int threads, const Params& P,
                          cudaStream_t st, const char* name, char* err, size_t errlen) {
  static std::once_flag once;
  std::call_once(once, [&] {
    for (auto kern : kernels) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  });
  kernels[variant]<<<grid, threads, smem, st>>>(P);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    snprintf(err, errlen, "%s: %s", name, cudaGetErrorString(e));
    return MMN_ERR_CUDA;
  }
  return MMN_OK;
}

int winattn_fwd(const mmn_winattn_desc* d, const void* q, const void* k, const void* v, const float* bias, const float* head_scale,
                const float* mask, void* out, float* lse, void* workspace, cudaStream_t st, char* err, size_t errlen) {
  FwdParams P;
  P.S = shape_from(d);
  P.sc = make_sched(P.S, d->batch);
  const int C = d->num_heads * d->head_dim;
  if (!make_window_maps(P.q, q, d->q_row_stride, d->batch, C, P.S) || !make_window_maps(P.k, k, d->k_row_stride, d->batch, C, P.S) ||
      !make_window_maps(P.v, v, d->v_row_stride, d->batch, C, P.S) || !make_window_maps(P.o, out, d->o_row_stride, d->batch, C, P.S))
    return tensor_map_failed(err, errlen);
  P.nH = d->num_heads;
  P.mask_windows = d->mask_windows > 0 ? d->mask_windows : 1;
  P.scale = d->scale;
  P.bias = bias; P.head_scale = head_scale; P.mask = mask; P.lse = lse;
  P.slab = (long long)P.S.n_windows * d->num_heads * kN;
  P.work = arm_work_counters(workspace, st, err, errlen);
  if (!P.work) return MMN_ERR_CUDA;
  const char* trace_path = getenv("MMN_TC_TRACE");
  P.trace = trace_setup(trace_path, st);

  // [cosine][mask kind]
  static void (*const kernels[6])(FwdParams) = {winattn_fwd_tc_kernel<false, MMN_MASK_NONE>, winattn_fwd_tc_kernel<false, MMN_MASK_SHIFT>,
                                                winattn_fwd_tc_kernel<false, MMN_MASK_TENSOR>, winattn_fwd_tc_kernel<true, MMN_MASK_NONE>,
                                                winattn_fwd_tc_kernel<true, MMN_MASK_SHIFT>, winattn_fwd_tc_kernel<true, MMN_MASK_TENSOR>};
  int per_head = num_sms_cached() / P.nH;        // CTAs per head (each CTA keeps one head's table resident)
  if (per_head < 1) per_head = 1;
  if (per_head > P.sc.n_items) per_head = P.sc.n_items;
  P.per_head = per_head;
  const int rc = launch_variant(kernels, (d->score_kind == MMN_SCORE_COSINE ? 3 : 0) + d->mask_kind, kFwdSmemBytes, per_head * P.nH,
                                kFwdThreads, P, st, "winattn_fwd_tc_kernel", err, errlen);
  if (rc != MMN_OK) return rc;
  if (P.trace.buf) dump_trace(P.trace.buf, trace_path, st);      // debug only: synchronous dump of CTA 0's timeline
  return MMN_OK;
}

}}  // namespace mmn::tc
