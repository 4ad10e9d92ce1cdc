// winattn_tc_bwd.cuh -- shifted-window attention backward on the Blackwell tensor cores.
//
// Same tiling and schedule as the forward (winattn_tc_fwd.cuh, tc_sched.cuh): a work item is a
// pair of 64-token windows of one wrap class x one head, operands gathered by TMA straight out of
// the un-windowed tensors, gradients scattered back through the same boxes.  Per item, with
// P = exp(S - lse) recomputed:
//   S  = Q K^T, dP = dO V^T        (M128 N64 K64 each: windows stacked along M, channels along K
//                                    against a shared zero block; S/dP double-buffered in TMEM so the
//                                    next item's are ready when the softmax warps finish this one)
//   dS = P o (dP - rowsum(P o dP)),  dS' = dS o c,  c_ij = d s_ij / d (q_i . k_j)
//   dV = P^T dO, dQ~ = dS' K, dK~ = dS'^T Q   (M128 N32 K128; one bf16 dS' tile serves both)
// Cosine attention differentiates through x / max(||x||, eps) in the epilogue:
// dq = dQ~ - q^ (q^ . dQ~) (likewise dk), exact because c already carries 1/||q|| 1/||k|| x logit scale.
// rowsum(P o dP) is computed in-tile, so `out` is never read.
//
// 768 threads, one CTA per SM (the kernel is latency-bound: 4 softmax warps per scheduler hide what 2 cannot):
//   warps 0-15   softmax: FOUR threads per query row (16 keys each).  Descriptor, lse and the q / k norms of an
//                item arrive in shared memory with its stage (producer ring + the forward kernel's per-window
//                record), so the loop carries no per-item state and issues no global load.  dbias accumulates
//                in registers in the item's tile order and leaves through the table buffer when the wrap
//                class changes (a CTA sees few classes: ClassQueue).
//   warps 16-19  epilogue: one thread per row; takes its q / k rows and norms out of the stage and hands the stage
//                back, then dQ~/dK~/dV out of TMEM -> normalisation Jacobian -> bf16 staging tiles.
//   warp 20 TMA producer (schedule, descriptor ring, tiles, records), warp 21 MMA issuer, warp 22 TMA store,
//   warp 23 column sums of dq, dk, dv (= projection bias gradients) read from the staging tiles.
//   (A 25th warp -- a second producer as in the forward -- does not launch: 800 threads x 80 registers are refused.)
// Shared memory: 3 stages (Q0|Z|Q1, K, V, dO0|Z|dO1), P double-buffered and dS' around one shared zero block,
// three staging tiles, the class table, the records.
// Register budget by warpgroup (setmaxnreg): softmax 80 (= launch), epilogue 104, the rest 56: 512*80 + 128*104 + 128*56 = 768*80.
#pragma once

#include "winattn_tc_fwd.cuh"

namespace mmn { namespace tc {

constexpr int kStagesB = 3;
constexpr int kStageBytesB = 2 * kQRegion + 2 * kTile;   // Q0|Z|Q1, K0 K1, V0 V1, dO0|Z|dO1
constexpr int kOffK = kQRegion, kOffV = kQRegion + kTile, kOffDO = kQRegion + 2 * kTile;
constexpr int kKeysPerThread = 16;                          // four softmax threads per query row
constexpr int kSoftmaxThreadsB = 4 * 128, kEpiThreads = 128;
constexpr int kEpiWarp0 = kSoftmaxThreadsB / 32, kProducerWarpB = kEpiWarp0 + 4, kMmaWarpB = kEpiWarp0 + 5, kStoreWarpB = kEpiWarp0 + 6;
constexpr int kColsumWarpB = kEpiWarp0 + 7;
constexpr int kBwdThreads = kSoftmaxThreadsB + 256;
// register budget by warpgroup (setmaxnreg only moves registers inside the CTA's launch allocation of 80):
//   softmax 80, epilogue 104, the rest 56     (512*80 + 128*104 + 128*56 = 768*80)
constexpr int kRegEpi = 104, kRegAux = 56;
constexpr int kChunkB = 1;            // items a CTA claims per atomic
constexpr int kItemRingB = 8;         // descriptor ring: entry n + 8 is written once the epilogue has handed back item n + 5's stage
constexpr int kPDBytes = 7 * 8192;    // P0[2] | dS'0 | Z | dS'1 | P1[2]
constexpr int kBwdTmemCols = 512;     // S[b] at 128 b, dP[b] at 128 b + 64; dV|dQ~|dK~ [b] at 256 + 96 b

struct BwdParams {
  CUtensorMap q[8], k[8], v[8], dout[8], dq[8], dk[8], dv[8];
  WinShape S;
  Sched sc;
  int nH, per_head;
  int mask_windows;
  float scale;
  const float* bias;
  const float* head_scale;
  const float* mask;
  const float* lse;     // written by the forward kernel: lse (B*nW, nH, 64), then the norms (B*nW, nH, 2, 64) in tile row order
  long long slab;       // B*nW*nH*64
  float* dbias;         // (nH, 64, 64) accumulated, may be null
  float* dhead_scale;   // (nH) accumulated, may be null
  float* dcolsum;       // (3, nH*32) accumulated column sums of dq, dk, dv (= projection bias grads), may be null
  int* work;            // dynamic schedule counters (winattn_tc_fwd.cuh: arm_work_counters)
  float* part;          // deterministic kernels: per-CTA partial sums, kDetSlotFloats per CTA (winattn_bwd_det_reduce)
  TraceCfg trace;       // debug: clock64 stamps of one CTA (MMN_TC_TRACE_BWD=<file>)
};


// Deterministic kernels (DET): CTA k of head h walks the static cost-balanced item range k of the head instead of the
// run-time queue, and its dbias / dcolsum / dhead_scale sums go to a slot of the workspace that only it writes, in program
// order; winattn_bwd_det_reduce then adds the slots of a head in CTA order.  Every slot entry that is read is written:
// the dbias region by the first flush (or zeros when the CTA had no item), the others once at the end.
constexpr int kDetColsum = kN * kN, kDetHscale = kN * kN + 3 * kD, kDetSlotFloats = kN * kN + 3 * kD + 4;

template <bool COS, int MASK, bool DET>
__global__ void __launch_bounds__(kBwdThreads, 1)
winattn_bwd_tc_kernel(const __grid_constant__ BwdParams P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sStage = smem;                                 // kStagesB x kStageBytesB
  // P (double-buffered over items) and dS' around ONE shared zero block, 8 KB each:
  //   P0[0] | P0[1] | dS'0 | Z | dS'1 | P1[0] | P1[1]
  // dS' is read K-major (dQ~) and MN-major (dK~) and needs Z adjacent on both sides; P is only read MN-major (dV), where
  // the second 64-row atom of the operand sits one leading-dimension offset away -- any distance -- so its zero half can be
  // the same Z.  With P double-buffered the softmax warps write P(n + 1) while the gradient MMAs of item n still run
  // (they were waiting ~1000 cycles per item for them); the second buffer costs 8 KB, not 24.
  uint8_t* sPD = sStage + kStagesB * kStageBytesB;
  uint8_t* sDS = sPD + 2 * 8192;                          // dS'0 | Z | dS'1
  uint8_t* sOut = sPD + kPDBytes;                         // dQ | dK | dV staging, 3 x kTile
  float* sTbl = reinterpret_cast<float*>(sOut + 3 * kTile);   // [64][kTblLd]
  float* sRec = sTbl + kN * kTblLd;                       // [kStagesB][2 slots][1/|q| | 1/|k| | lse log2][64 tile rows]: the forward kernel's
                                                          //   per-window records, bulk-copied with the stage
  float* sDelta = sRec + kStagesB * 2 * 3 * kN;           // [4][128] partial deltas
  float* sRed = sDelta + 512;                             // 16 floats: dhead_scale per softmax warp
  uint8_t* sPos = reinterpret_cast<uint8_t*>(sRed + 16);  // [8][64]
  uint8_t* sRid = sPos + 512;                             // [8][64] window position -> shift-mask region id
  const ItemRing<kItemRingB> ring{reinterpret_cast<int4*>(sRid + 512)};      // item descriptors (tc_sched.cuh)
  int* sEnd = reinterpret_cast<int*>(sRid + 512 + ring.kBytes);  // [0] items of this CTA once the epilogue warps know (else INT_MAX)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sEnd + 4);
  uint64_t* full = bars;                                  // [kStagesB]
  uint64_t* empty = bars + kStagesB;                      // [kStagesB] (one arrival per warp: epilogue threads)
  uint64_t* sdp_full = bars + 2 * kStagesB;               // [2]
  uint64_t* sdp_empty = sdp_full + 2;                     // [2] one arrival per warp
  uint64_t* pds_full = sdp_full + 4;                      // one arrival per warp
  uint64_t* out_full = sdp_full + 5;                      // [2]
  uint64_t* out_empty = sdp_full + 7;                     // [2] one arrival per warp
  uint64_t* so_ready = sdp_full + 9;                      // [3] one per staging tile (dq, dk, dv), one arrival per warp
  uint64_t* so_free = sdp_full + 12;                      // [3]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sdp_full + 15);

  const WinShape& S = P.S;
  const Sched& sc = P.sc;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int h = blockIdx.x % P.nH;
  float* const det_slot = DET ? P.part + (size_t)(h * P.per_head + blockIdx.x / P.nH) * kDetSlotFloats : nullptr;

  // ---- one-time setup
  for (int i = tid; i < (kStagesB * kStageBytesB + kPDBytes) / 16; i += kBwdThreads)
    reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  fill_class_luts(S, sPos, sRid, tid, kBwdThreads);
  for (int i = tid; i < kStagesB * 2 * 3 * kN; i += kBwdThreads) sRec[i] = 0.f;
  if (tid == 0) {
    sEnd[0] = 0x7fffffff;
    for (int s = 0; s < kStagesB; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], kEpiThreads / 32); }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&sdp_full[b], 1); mbar_init(&sdp_empty[b], kSoftmaxThreadsB / 32);
      mbar_init(&out_full[b], 1); mbar_init(&out_empty[b], kEpiThreads / 32);
    }
    mbar_init(pds_full, kSoftmaxThreadsB / 32);
    for (int t = 0; t < 3; ++t) { mbar_init(&so_ready[t], kEpiThreads / 32); mbar_init(&so_free[t], P.dcolsum ? 2 : 1); }
    fence_barrier_init();
  }
  if (warp == kProducerWarpB && lane == 0)
    for (int i = 0; i < 8; ++i) { tma_prefetch_desc(&P.q[i]); tma_prefetch_desc(&P.k[i]); tma_prefetch_desc(&P.v[i]); tma_prefetch_desc(&P.dout[i]); }
  if (warp == kStoreWarpB && lane == 0)
    for (int i = 0; i < 8; ++i) { tma_prefetch_desc(&P.dq[i]); tma_prefetch_desc(&P.dk[i]); tma_prefetch_desc(&P.dv[i]); }
  if (warp == kMmaWarpB) tmem_alloc<kBwdTmemCols>(tmem_slot);
  fence_proxy_async_smem();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *tmem_slot;
  trace_cta_time(P.trace, 0);

  if (warp >= kProducerWarpB) {
    setmaxnreg_dec<kRegAux>();
    if (warp == kProducerWarpB) {
      // ============================== TMA producer (schedule, descriptor ring, tiles, records) ==============================
      // every lane runs the loop; lane l issues boxes l, l + 32 of the item (BoxPlan: which map, piece offset and
      // shared-memory offset a lane's boxes have depends only on the wrap class)
      const BoxLayout<4> lay{{P.q, P.dout, P.k, P.v}, {0, kOffDO, kOffK, kOffV}, {2 * kWinBytes, 2 * kWinBytes, kWinBytes, kWinBytes}};
      BoxPlan<4> plan;
      // Dynamic schedule (see the forward kernel's producer): chunks of kChunkB items of this head's class-sorted list
      // through an atomic counter; every other warp follows the descriptor ring.  One end marker.
      // (An L2 prefetch of item n + 1's boxes issued right after item n's loads made the kernel 33 % SLOWER, 0.46 -> 0.61 ms:
      // the extra boxes queue in the SM's TMA unit in front of the next loads and the gradient stores.)
      // One item: descriptor (published by the arrival on full[stage]), tiles, and per slot (lane = slot) the window's
      // record of norms and lse, already in tile row order.  The same in both schedules.
      auto load_item = [=, &P, &S, &plan](int n, const RingItem& it) {
        const int stage = n % kStagesB, phase = (n / kStagesB) & 1;
        if (it.cls != plan.cls) plan.build(S, it.cls, lane, lay);
        trace_ev(P.trace, 2, n, 0);
        mbar_wait(&empty[stage], phase ^ 1);
        trace_ev(P.trace, 2, n, 1);
        if (lane == 0) {
          ring.publish(n, it);
          mbar_arrive_expect_tx(&full[stage], it.nvalid * (4 * kWinBytes + 3 * kN * 4));
        }
        __syncwarp();
        plan.issue<true>(S, it.ws[0], it.ws[1], it.nvalid, h * kD, sStage + stage * kStageBytesB, &full[stage], lane);
        if (lane < it.nvalid)
          bulk_load_1d(sRec + (stage * 2 + lane) * (3 * kN), P.lse + P.slab + ((long long)(lane ? it.win[1] : it.win[0]) * P.nH + h) * (3 * kN),
                       3 * kN * 4, &full[stage]);
        trace_ev(P.trace, 2, n, 2);
      };
      const int k = blockIdx.x / P.nH;
      int n;
      if (DET) {
        const int begin = sched_range_begin(sc, k, P.per_head);
        n = walk_range(S, sc, begin, sched_range_begin(sc, k + 1, P.per_head) - begin, 0, load_item);
      } else {
        n = walk_queue(S, sc, sched_range_begin(sc, k, P.per_head), P.work + h * 8, kChunkB, lane, load_item);
      }
      {   // end marker
        const int stage = n % kStagesB, phase = (n / kStagesB) & 1;
        mbar_wait(&empty[stage], phase ^ 1);
        if (lane == 0) {
          ring.publish_end(n);
          mbar_arrive(&full[stage]);
        }
        __syncwarp();
      }
    } else if (warp == kMmaWarpB) {
      // ============================== MMA issuer ==============================
      constexpr uint32_t idescS = umma_idesc_bf16(128, 64, 0, 0);     // A K-major, B K-major
      constexpr uint32_t idescKM = umma_idesc_bf16(128, 32, 0, 1);    // A K-major (dS'),        B MN-major (K)
      constexpr uint32_t idescMM = umma_idesc_bf16(128, 32, 1, 1);    // A MN-major (P^T, dS'^T), B MN-major (dO, Q)
      // descriptors: everything but the 14-bit start-address field is loop-invariant, and adding (bytes >> 4)
      // to a descriptor moves its start address -- one add per operand instead of rebuilding it
      const uint64_t dKm = umma_smem_desc(0, 0, 512, kSwz64);         // Q, K, V, dO tiles read K-major
      const uint64_t dMn = umma_smem_desc(0, 8192, 512, kSwz64);      // K, Q, dO tiles read MN-major
      const uint64_t dPk = umma_smem_desc(0, 0, 1024, kSwz128);       // dS' read K-major
      const uint64_t dPm = umma_smem_desc(0, 8192, 1024, kSwz128);    // dS' read MN-major (transposed)
      const uint32_t stage0 = smem_u32(sStage) >> 4, pd0 = smem_u32(sPD) >> 4, ds0 = smem_u32(sDS) >> 4;
      constexpr uint32_t W16 = kWinBytes >> 4;
      int total = 0x7fffffff;                                         // items of this CTA: known once the end marker shows up
      auto issue_sdp = [&](int n) {
        const int stage = n % kStagesB, phase = (n / kStagesB) & 1, b = n & 1;
        mbar_wait(&full[stage], phase);
        if (ring.read(n).end()) { total = n; return; }
        mbar_wait(&sdp_empty[b], ((n >> 1) & 1) ^ 1);
        tcgen05_fence_after();
        trace_ev(P.trace, 3, n - 2, 4);
        if (elect_one()) {
          const uint64_t sb = dKm + (stage0 + stage * (kStageBytesB >> 4));
          const uint32_t tS = tmem + b * 128, tDP = tS + 64;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
            umma_bf16_ss(tS, sb + ((ks >> 1) * W16 + (ks & 1) * 2), sb + ((kOffK >> 4) + (ks >> 1) * W16 + (ks & 1) * 2), idescS, ks);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
            umma_bf16_ss(tDP, sb + ((kOffDO >> 4) + (ks >> 1) * W16 + (ks & 1) * 2), sb + ((kOffV >> 4) + (ks >> 1) * W16 + (ks & 1) * 2), idescS, ks);
          umma_commit(&sdp_full[b]);
        }
        __syncwarp();
        trace_ev(P.trace, 3, n - 2, 5);
      };
      issue_sdp(0);
      if (total > 1) issue_sdp(1);
      for (int n = 0; n < total; ++n) {
        const int stage = n % kStagesB, b = n & 1;
        trace_ev(P.trace, 3, n, 0);
        mbar_wait(pds_full, n & 1);
        mbar_wait(&out_empty[b], ((n >> 1) & 1) ^ 1);
        trace_ev(P.trace, 3, n, 1);
        tcgen05_fence_after();
        if (elect_one()) {
          const uint64_t sbm = dMn + (stage0 + stage * (kStageBytesB >> 4));
          const uint64_t adk = dPk + ds0, adm = dPm + ds0;
          // P buffer b, read MN-major: window 0's steps start in P0[b] with the zero block one LBO above, window 1's start
          // in the zero block with P1[b] one LBO above
          const uint64_t ap0 = umma_smem_desc(0, 3 * 8192 - b * 8192, 1024, kSwz128) + (pd0 + b * (8192 >> 4));
          const uint64_t ap1 = umma_smem_desc(0, 2 * 8192 + b * 8192, 1024, kSwz128) + (pd0 + ((3 * 8192) >> 4));
          const uint32_t tO = tmem + 256 + b * 96;
#pragma unroll
          for (int ks = 0; ks < 8; ++ks) {   // 16 queries (dV, dK~) or 16 keys (dQ~) per step; ks < 4: window 0
            const uint32_t wofs = (ks >> 2) * 2 * W16 + (ks & 3) * 64;     // 16 rows of window ks/4 inside a X0|Z|X1 region
            // dV[key][d] += P[query][key]^T dO[query][d]
            umma_bf16_ss(tO, (ks < 4 ? ap0 : ap1) + (ks & 3) * 128, sbm + ((kOffDO >> 4) + wofs), idescMM, ks);
            // dQ~[query][d] += dS'[query][key] K[key][d]
            umma_bf16_ss(tO + 32, adk + ((ks >> 2) * 512 + (ks & 3) * 2), sbm + ((kOffK >> 4) + ks * 64), idescKM, ks);
            // dK~[key][d] += dS'[query][key]^T Q[query][d]
            umma_bf16_ss(tO + 64, adm + ks * 128, sbm + wofs, idescMM, ks);
          }
          umma_commit(&out_full[b]);
        }
        __syncwarp();
        trace_ev(P.trace, 3, n, 2);
        if (total == 0x7fffffff) issue_sdp(n + 2);
        trace_ev(P.trace, 3, n, 3);
      }
      // farewell to the epilogue warps: an arrival on the out_full buffer item `total` would have used, once they have
      // taken item total - 2 from it (two phases completing back to back would alias in their parity wait)
      if (total >= 2) mbar_wait(&out_empty[total & 1], ((total - 2) >> 1) & 1);
      if (lane == 0) {
        sEnd[0] = total;
        mbar_arrive(&out_full[total & 1]);
      }
      __syncwarp();
    } else if (warp == kStoreWarpB) {
      // ============================== TMA store ==============================
      // The three staging tiles (dq, dk, dv) are handed over one by one, so the epilogue warps fill the next
      // tile while this one drains.  Each lane issues its share of a tile's boxes; a tile is returned to the
      // epilogue once the bulk group two behind has finished reading shared memory.
      const BoxLayout<1> lay{{P.dq}, {0}, {kWinBytes}};   // dq[8] | dk[8] | dv[8] are contiguous in BwdParams: tensor t's maps are 8 t further
      BoxPlan<1> plan;
      int grp = 0;
      bool done = false;
      for (int n = 0; !done; ++n) {
        RingItem it;
#pragma unroll
        for (int t = 0; t < 3; ++t, ++grp) {
          if (t == 0) trace_ev(P.trace, 4, n, 0);
          mbar_wait(&so_ready[t], n & 1);
          if (t == 0) {
            if (n >= *reinterpret_cast<volatile int*>(sEnd)) { done = true; break; }   // that arrival was the epilogue warps' farewell
            it = ring.read(n);
            if (it.cls != plan.cls) plan.build(S, it.cls, lane, lay);
            trace_ev(P.trace, 4, n, 1);
          }
          plan.issue<false>(S, it.ws[0], it.ws[1], it.nvalid, h * kD, sOut + t * kTile, nullptr, lane, 8 * t);
          tma_store_commit();
          tma_store_wait_read<2>();        // per thread: the group two behind (tile (t + 1) % 3) has been read out
          __syncwarp();
          if (lane == 0 && grp >= 2) mbar_arrive(&so_free[(t + 1) % 3]);
        }
        trace_ev(P.trace, 4, n, 2);
      }
      tma_store_wait_all<0>();
    } else if (warp == kColsumWarpB && P.dcolsum) {
      // ============================== column sums of dq, dk, dv (= q / k / v projection bias gradients) ==============================
      // One warp sums the bf16 staging tiles while the TMA store drains them: lane (r0, c) owns the 16-byte channel group
      // c of rows r0, r0 + 8, ...; 24 running fp32 sums per lane for the whole kernel, reduced across lanes once at the
      // end.  (In the epilogue warps this was a 32x32 transpose-reduce per tile: 40 % of their instructions.)  Rows of an
      // invalid slot are zero in the tile.  Sums are over the bf16-rounded gradients, i.e. exactly the column sums of the
      // dq/dk/dv tensors the kernel writes (what a bias gradient computed from them would be).
      const int cg = lane & 3, r0 = lane >> 2;
      float acc[3][8];
#pragma unroll
      for (int t = 0; t < 3; ++t)
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[t][e] = 0.f;
      bool done = false;
      for (int n = 0; !done; ++n) {
#pragma unroll
        for (int t = 0; t < 3; ++t) {
          mbar_wait(&so_ready[t], n & 1);
          if (t == 0 && n >= *reinterpret_cast<volatile int*>(sEnd)) { done = true; break; }
          const uint8_t* tile = sOut + t * kTile;
#pragma unroll 4
          for (int it = 0; it < 16; ++it) {
            const int row = r0 + 8 * it;
            const uint4 v = *reinterpret_cast<const uint4*>(tile + row * 64 + ((cg ^ ((row >> 1) & 3)) << 4));
            const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              acc[t][2 * e] += __uint_as_float(u[e] << 16);
              acc[t][2 * e + 1] += __uint_as_float(u[e] & 0xffff0000u);
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&so_free[t]);
        }
      }
      const int C = P.nH * kD;
#pragma unroll
      for (int t = 0; t < 3; ++t)
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float v = acc[t][e];
          v += __shfl_xor_sync(0xffffffffu, v, 4);
          v += __shfl_xor_sync(0xffffffffu, v, 8);
          v += __shfl_xor_sync(0xffffffffu, v, 16);
          if (lane < 4) {
            if (DET) det_slot[kDetColsum + t * kD + cg * 8 + e] = v;
            else atomicAdd(P.dcolsum + t * C + h * kD + cg * 8 + e, v);
          }
        }
    }
  } else if (warp >= kEpiWarp0) {
    // ============================== epilogue warpgroup: one thread per tile row ==============================
    const int r = tid - kEpiWarp0 * 32;
    const int slot = r >> 6, i = r & 63;
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const int rsw = (r >> 1) & 3;                       // 64B-swizzle phase of this thread's tile row
    setmaxnreg_inc<kRegEpi>();
    float dscale_acc = 0.f;                             // sum over rows of q_i . dQ~_i = sum_ij dS_ij (s_ij - bias_ij)
    const float inv_hscale = COS ? 1.f / __ldg(P.head_scale + h) : 1.f;
    int n = 0;
    for (;; ++n) {
      const int stage = n % kStagesB, b = n & 1;
      const uint8_t* base = sStage + stage * kStageBytesB;
      const uint32_t tO = tmem + lane_base + 256 + b * 96;
      if (warp == kEpiWarp0) trace_ev(P.trace, 1, n, 0);
      mbar_wait(&out_full[b], (n >> 1) & 1);
      if (n >= *reinterpret_cast<volatile int*>(sEnd)) break;      // that arrival was the MMA warp's farewell
      tcgen05_fence_after();
      const bool valid = slot < ring.read(n).nvalid;
      if (warp == kEpiWarp0) trace_ev(P.trace, 1, n, 1);

      // Everything this item still needs from its stage -- this thread's q and k rows and their norms (ring slot n % 3,
      // written by the softmax warps when they prepared the item) -- is taken into registers first, and the stage is
      // handed back to the producer at once: the refill (issue + TMA latency) then runs under the three tiles below
      // instead of after two of them, which is what the softmax warps were waiting for at the next-but-one item.
      uint4 xrow[2][4];
      float rinv2[2] = {1.f, 1.f};
      if (COS) {
        const uint8_t* qrow = base + slot * 2 * kWinBytes + i * 64;
        const uint8_t* krow_ = base + kOffK + r * 64;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          xrow[0][c] = *reinterpret_cast<const uint4*>(qrow + ((c ^ rsw) << 4));
          xrow[1][c] = *reinterpret_cast<const uint4*>(krow_ + ((c ^ rsw) << 4));
        }
        rinv2[0] = sRec[(stage * 2 + slot) * (3 * kN) + i];
        rinv2[1] = sRec[(stage * 2 + slot) * (3 * kN) + kN + i];
      }
      mbar_arrive_warp(&empty[stage]);

#pragma unroll
      for (int t = 0; t < 3; ++t) {                     // t = 0: dQ~ with the q row, 1: dK~ with the k row, 2: dV
        uint32_t g32[32];
        tmem_ld_32x32b_x32(tO + (t == 2 ? 0 : 32 + t * 32), g32);
        tmem_ld_wait();
        if (t == 2) {
          tcgen05_fence_before();
          mbar_arrive_warp(&out_empty[b]);                   // accumulators read out
        }
        uint32_t o[16];
        if (COS && t < 2) {
          // d/dx of x / max(||x||, eps) applied to G = dQ~ (which already carries 1/||x||): G - x^ (x^ . G)
          uint64_t x2[16];                              // the row's 32 channels as fp32 pairs
          uint64_t dot2[4] = {0ull, 0ull, 0ull, 0ull};
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const uint4 xq = xrow[t][c];
            const uint32_t u[4] = {xq.x, xq.y, xq.z, xq.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              x2[c * 4 + e] = pk2u(u[e] << 16, u[e] & 0xffff0000u);
              dot2[e] = fma2(x2[c * 4 + e], pk2u(g32[c * 8 + 2 * e], g32[c * 8 + 2 * e + 1]), dot2[e]);
            }
          }
          const float rinv = rinv2[t];                  // 1 / max(||x||, eps)
          float xga, xgb;
          upk2(add2(add2(dot2[0], dot2[1]), add2(dot2[2], dot2[3])), xga, xgb);
          const float xg = xga + xgb;
          if (t == 0 && valid) dscale_acc += xg;
          const float proj = rinv >= 1e12f ? 0.f : -xg * rinv * rinv;     // below eps the normalisation is x / eps: no projection
          const uint64_t proj2 = pk2(proj, proj);
#pragma unroll
          for (int c = 0; c < 16; ++c) {
            const uint64_t o2 = fma2(x2[c], proj2, pk2u(g32[2 * c], g32[2 * c + 1]));
            float o0, o1;
            upk2(o2, o0, o1);
            o[c] = pack_bf16x2(o0, o1);
          }
        } else {
#pragma unroll
          for (int c = 0; c < 16; ++c) o[c] = pack_bf16x2(__uint_as_float(g32[2 * c]), __uint_as_float(g32[2 * c + 1]));
        }
        mbar_wait(&so_free[t], (n & 1) ^ 1);            // the previous item's stores have drained this staging tile
        uint8_t* orow = sOut + t * kTile + r * 64;
#pragma unroll
        for (int c = 0; c < 4; ++c)
          *reinterpret_cast<uint4*>(orow + ((c ^ rsw) << 4)) =
              valid ? make_uint4(o[c * 4 + 0], o[c * 4 + 1], o[c * 4 + 2], o[c * 4 + 3]) : make_uint4(0, 0, 0, 0);
        fence_proxy_async_smem();
        mbar_arrive_warp(&so_ready[t]);
        if (warp == kEpiWarp0) trace_ev(P.trace, 1, n, 2 + t);
      }
    }
    // farewell to the store / column-sum warps through so_ready[0], once they have taken the last item's tile 0
    if (n > 0) mbar_wait(&so_free[0], (n - 1) & 1);
    mbar_arrive_warp(&so_ready[0]);
    if (COS && P.dhead_scale) {                          // d s_ij / d(logit scale) = cos_ij = (s_ij - bias_ij) / logit scale
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) dscale_acc += __shfl_xor_sync(0xffffffffu, dscale_acc, o);
      if (lane == 0) {
        if (DET) det_slot[kDetHscale + (warp - kEpiWarp0)] = dscale_acc * inv_hscale;
        else atomicAdd(P.dhead_scale + h, dscale_acc * inv_hscale);
      }
    }
  } else {
    // ============================== softmax (512 threads: 4 per row, 16 keys each; registers as launched) ==============================
    constexpr int KP = kKeysPerThread;
    const int r = tid & 127, qt = tid >> 7;             // tile row; which quarter of its 64 keys
    const int slot = r >> 6, i = r & 63;
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const float hscale = COS ? __ldg(P.head_scale + h) : P.scale;
    const float* bias_h = P.bias ? P.bias + (size_t)h * kN * kN : nullptr;
    float* const gdb_head = P.dbias ? P.dbias + (size_t)h * kN * kN : nullptr;
    uint8_t* prow0 = sPD + slot * (5 * 8192) + i * 128;     // this thread's row of P0[0] / P1[0]; buffer 1 is 8 KB further
    uint8_t* drow = sDS + slot * 16384 + i * 128;
    float dbacc[KP];                                    // dbias[tile row i][KP*qt + j] of the current wrap class
#pragma unroll
    for (int j = 0; j < KP; ++j) dbacc[j] = 0.f;
    const int trole = warp == 0 ? 0 : -1;
    bool det_flushed = false;                           // DET: this CTA's dbias slot has been written once
#define TRB(item, ev) do { if (trole >= 0) trace_ev(P.trace, trole, item, ev); } while (0)

    // dbias of a wrap class leaves the CTA through the (idle at that moment) table buffer: the two windows of the tile
    // are summed there, then the 64x64 sums go out as atomics with consecutive threads on consecutive columns, so a
    // warp's 32 atomics fall into one or two cache lines.  (One atomic per thread and register, rows 256 B apart, was
    // 8192 scattered L2 transactions per CTA and flush -- ~30 us when every CTA changes class at the same time.)
    // Called by all softmax threads; the caller has made sure nobody reads the table any more.
    auto flush_dbias = [&](int cls) {
      float4* mine = reinterpret_cast<float4*>(sTbl + i * kTblLd + qt * KP);
      if (slot == 0) {
#pragma unroll
        for (int j4 = 0; j4 < KP / 4; ++j4) mine[j4] = make_float4(dbacc[j4 * 4], dbacc[j4 * 4 + 1], dbacc[j4 * 4 + 2], dbacc[j4 * 4 + 3]);
      }
      named_bar_sync(3, kSoftmaxThreadsB);
      if (slot == 1) {
#pragma unroll
        for (int j4 = 0; j4 < KP / 4; ++j4) {
          float4 v = mine[j4];
          v.x += dbacc[j4 * 4]; v.y += dbacc[j4 * 4 + 1]; v.z += dbacc[j4 * 4 + 2]; v.w += dbacc[j4 * 4 + 3];
          mine[j4] = v;
        }
      }
#pragma unroll
      for (int j = 0; j < KP; ++j) dbacc[j] = 0.f;
      named_bar_sync(3, kSoftmaxThreadsB);
      const uint8_t* pos = sPos + cls * 64;
      for (int e = tid; e < kN * kN; e += kSoftmaxThreadsB) {
        const int ti = e >> 6, tj = e & 63;
        if (DET) {                                      // pos is a permutation: the flush covers the whole slot
          float* dst = det_slot + (int)pos[ti] * kN + pos[tj];
          *dst = (det_flushed ? *dst : 0.f) + sTbl[ti * kTblLd + tj];
        } else {
          atomicAdd(gdb_head + (int)pos[ti] * kN + pos[tj], sTbl[ti * kTblLd + tj]);
        }
      }
      det_flushed = true;
    };

    // Everything an item needs besides its logits -- descriptor, this row's lse, the q / k norms -- arrives in shared
    // memory with the item's stage (descriptor ring + the forward kernel's per-window record), so the loop carries no
    // per-item state in registers and issues no global load.
    int cls_loaded = -1;
    for (int n = 0;; ++n) {
      const int b = n & 1, stage = n % kStagesB;
      TRB(n, 0);
      mbar_wait(&full[stage], (n / kStagesB) & 1);
      const RingItem item = ring.read(n);               // written by the producer before it armed full[stage]
      if (item.end()) break;
      const int cls = item.cls;
      const bool valid = slot < item.nvalid;
      const float* rec = sRec + (stage * 2 + slot) * (3 * kN);
      const float lse2 = valid ? rec[2 * kN + i] : 0.f;
      if (cls != cls_loaded) {                          // rare: at most 8 times per CTA
        named_bar_sync(3, kSoftmaxThreadsB);            // everyone is done reading the old table
        if (gdb_head && cls_loaded >= 0) {
          flush_dbias(cls_loaded);
          named_bar_sync(3, kSoftmaxThreadsB);          // sums read out: the buffer can take the new table
        }
        build_class_table(sTbl, kTblLd, bias_h, sPos + cls * 64, sRid + cls * 64, MASK == MMN_MASK_SHIFT && cls != 0, tid, kSoftmaxThreadsB);
        cls_loaded = cls;
        named_bar_sync(3, kSoftmaxThreadsB);
      }
      TRB(n, 2);
      const float a_i = COS ? rec[i] * hscale : hscale;
      const float a_l2 = a_i * kLog2e;
      const float4* krow = reinterpret_cast<const float4*>(rec + kN + qt * KP);

      // ---- (b) additive terms of this thread's logits (table, mask, -lse), log2 domain
      float p[KP];
      {
        const float4* trow = reinterpret_cast<const float4*>(sTbl + i * kTblLd + qt * KP);
        const float* mrow = nullptr;
        if (MASK == MMN_MASK_TENSOR) {
          const int gw = slot ? item.win[1] : item.win[0], ipos = sPos[cls * 64 + i];
          mrow = P.mask + ((size_t)(gw % P.mask_windows) * kN + ipos) * kN + qt * KP;
        }
#pragma unroll
        for (int j4 = 0; j4 < KP / 4; ++j4) {
          float4 tt = trow[j4];
          if (MASK == MMN_MASK_TENSOR) {
            const float4 mm = __ldg(reinterpret_cast<const float4*>(mrow) + j4);
            tt.x = fmaf(mm.x, kLog2e, tt.x); tt.y = fmaf(mm.y, kLog2e, tt.y); tt.z = fmaf(mm.z, kLog2e, tt.z); tt.w = fmaf(mm.w, kLog2e, tt.w);
          }
          p[j4 * 4 + 0] = tt.x - lse2; p[j4 * 4 + 1] = tt.y - lse2; p[j4 * 4 + 2] = tt.z - lse2; p[j4 * 4 + 3] = tt.w - lse2;
        }
      }

      // ---- (c) S and dP from TMEM; P = exp(S - lse); partial delta and d(logit scale) sums
      TRB(n, 3);
      mbar_wait(&sdp_full[b], (n >> 1) & 1);
      tcgen05_fence_after();
      TRB(n, 4);
      float delta = 0.f;                                // sum_j p_j dp_j over this thread's keys
      {
        // dP is read twice (here for delta, after the barrier for dS) rather than kept in 16 registers across the
        // barrier and the next item's preparation: the softmax warps run at the 80-register limit, and the S/dP buffer
        // is not needed back before item n + 2's MMAs anyway (they are issued after this item's dS').
        uint32_t raw[KP], dpr[KP];
        tmem_ld_32x32b(tmem + lane_base + b * 128 + qt * KP, raw);
        tmem_ld_32x32b(tmem + lane_base + b * 128 + 64 + qt * KP, dpr);
        tmem_ld_wait();
#pragma unroll
        for (int j4 = 0; j4 < KP / 4; ++j4) {
          const float4 kk = COS ? krow[j4] : make_float4(1.f, 1.f, 1.f, 1.f);
          const float rk[4] = {kk.x, kk.y, kk.z, kk.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int j = j4 * 4 + e;
            const float pj = fast_exp2(fmaf(__uint_as_float(raw[j]), COS ? rk[e] * a_l2 : a_l2, p[j]));   // log2 domain: a_l2 = a_i log2(e)
            const float dpj = __uint_as_float(dpr[j]);
            delta = fmaf(pj, dpj, delta);
            p[j] = pj;
          }
        }
      }
      sDelta[qt * 128 + r] = delta;
      TRB(n, 5);
      // P (bf16) can go out before delta is known, into the buffer the gradient MMAs of item n - 2 have long left
      if (n > 1) mbar_wait(&out_full[b], ((n - 2) >> 1) & 1);
      uint8_t* prow = prow0 + b * 8192;
      TRB(n, 6);
#pragma unroll
      for (int c = 0; c < KP / 8; ++c) {
        uint4 v4 = make_uint4(pack_bf16x2(p[c * 8 + 0], p[c * 8 + 1]), pack_bf16x2(p[c * 8 + 2], p[c * 8 + 3]),
                              pack_bf16x2(p[c * 8 + 4], p[c * 8 + 5]), pack_bf16x2(p[c * 8 + 6], p[c * 8 + 7]));
        if (!valid) v4 = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4*>(prow + (((qt * (KP / 8) + c) ^ (i & 7)) << 4)) = v4;
      }
      named_bar_sync(2, kSoftmaxThreadsB);
      TRB(n, 7);
      delta = sDelta[r] + sDelta[128 + r];
      delta += sDelta[256 + r] + sDelta[384 + r];

      // ---- (d) dS = P o (dP - delta): dbias; dS' = dS o c into the MMA tile; d(logit scale)
      {
        uint32_t dpr[KP];
        tmem_ld_32x32b(tmem + lane_base + b * 128 + 64 + qt * KP, dpr);
        tmem_ld_wait();
        tcgen05_fence_before();
        mbar_arrive_warp(&sdp_empty[b]);
#pragma unroll
        for (int j = 0; j < KP; ++j) p[j] *= __uint_as_float(dpr[j]) - delta;
      }
      if (valid && gdb_head) {
#pragma unroll
        for (int j = 0; j < KP; ++j) dbacc[j] += p[j];
      }
      if (n > 0) mbar_wait(&out_full[b ^ 1], ((n - 1) >> 1) & 1);   // the previous item's dQ~ / dK~ MMAs have read dS'
#pragma unroll
      for (int c = 0; c < KP / 8; ++c) {
        float cj[8];
        if (COS) {
          const float4 k0 = krow[c * 2], k1 = krow[c * 2 + 1];
          cj[0] = k0.x * a_i; cj[1] = k0.y * a_i; cj[2] = k0.z * a_i; cj[3] = k0.w * a_i;
          cj[4] = k1.x * a_i; cj[5] = k1.y * a_i; cj[6] = k1.z * a_i; cj[7] = k1.w * a_i;
        } else {
#pragma unroll
          for (int e = 0; e < 8; ++e) cj[e] = a_i;
        }
        uint4 v4 = make_uint4(pack_bf16x2(p[c * 8 + 0] * cj[0], p[c * 8 + 1] * cj[1]), pack_bf16x2(p[c * 8 + 2] * cj[2], p[c * 8 + 3] * cj[3]),
                              pack_bf16x2(p[c * 8 + 4] * cj[4], p[c * 8 + 5] * cj[5]), pack_bf16x2(p[c * 8 + 6] * cj[6], p[c * 8 + 7] * cj[7]));
        if (!valid) v4 = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4*>(drow + (((qt * (KP / 8) + c) ^ (i & 7)) << 4)) = v4;
      }
      fence_proxy_async_smem();
      mbar_arrive_warp(pds_full);
      TRB(n, 8);
    }
#undef TRB

    // ---- cross-window reduction: dbias (registers)
    if (gdb_head && cls_loaded >= 0) {
      named_bar_sync(3, kSoftmaxThreadsB);              // everyone is done reading the table
      flush_dbias(cls_loaded);
    } else if (DET && gdb_head) {                       // no item: the slot still enters the reduction
      for (int e = tid; e < kN * kN; e += kSoftmaxThreadsB) det_slot[e] = 0.f;
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  trace_cta_time(P.trace, 1);
  if (warp == kMmaWarpB) tmem_dealloc<kBwdTmemCols>(tmem);
}

constexpr size_t kBwdSmemBytes = 1024 + kStagesB * kStageBytesB + kPDBytes + 3 * kTile + kN * kTblLd * 4 +
                                 (kStagesB * 2 * 3 * kN + 512 + 16) * 4 + 1024 + ItemRing<kItemRingB>::kBytes + 16 + 24 * 8;

// Deterministic mode, second launch: for each head, the per_head slots of its CTAs summed in CTA order and added into dbias,
// dcolsum and dhead_scale (each may be null).  Block = 128 slot entries (one float4 per lane) x 32 slices of the CTA range,
// as gemm_reduce_kernel: pure latency, at most ceil(per_head / 32) loads per thread; fixed summation order.
constexpr int kDetRedSlices = 32;
__global__ void __launch_bounds__(kDetRedSlices * 32)
winattn_bwd_det_reduce(const float* __restrict__ part, int per_head, int nH, float* __restrict__ dbias, float* __restrict__ dcolsum,
                       float* __restrict__ dhead_scale) {
  __shared__ float4 red[kDetRedSlices][32];
  const int lane = threadIdx.x & 31, sl = threadIdx.x >> 5, h = blockIdx.y;
  const int e = (blockIdx.x * 32 + lane) * 4;
  const float* base = part + (size_t)h * per_head * kDetSlotFloats;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (e < kDetSlotFloats) {
#pragma unroll 4
    for (int k = sl; k < per_head; k += kDetRedSlices) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(base + (size_t)k * kDetSlotFloats + e));
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
  }
  red[sl][lane] = acc;
  __syncthreads();
  if (sl < 4) {
    acc = red[8 * sl][lane];
#pragma unroll
    for (int k = 1; k < 8; ++k) { const float4 v = red[8 * sl + k][lane]; acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w; }
    red[8 * sl][lane] = acc;
  }
  __syncthreads();
  if (sl != 0 || e >= kDetSlotFloats) return;
#pragma unroll
  for (int k = 1; k < 4; ++k) { const float4 v = red[8 * k][lane]; acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w; }
  if (e < kDetColsum) {
    if (dbias) {
      float4* o = reinterpret_cast<float4*>(dbias + (size_t)h * kN * kN + e);
      float4 r = *o;
      r.x += acc.x; r.y += acc.y; r.z += acc.z; r.w += acc.w;
      *o = r;
    }
  } else if (e < kDetHscale) {
    if (dcolsum) {
      const int t = (e - kDetColsum) / kD, c = (e - kDetColsum) % kD;
      float* o = dcolsum + (size_t)t * nH * kD + h * kD + c;
      o[0] += acc.x; o[1] += acc.y; o[2] += acc.z; o[3] += acc.w;
    }
  } else if (dhead_scale) {                                      // the four epilogue warps' sums
    dhead_scale[h] += (acc.x + acc.y) + (acc.z + acc.w);
  }
}

// CTAs per head of the backward launch (one CTA per SM over all heads, at least one per head, at most one per item).
inline int bwd_ctas_per_head(const WinShape& S, const mmn_winattn_desc* d) {
  int per_head = num_sms_cached() / d->num_heads;
  if (per_head < 1) per_head = 1;
  const int n_items = make_sched(S, d->batch).n_items;
  return per_head > n_items ? n_items : per_head;
}

size_t bwd_det_workspace_bytes(const mmn_winattn_desc* d) {
  return (size_t)bwd_ctas_per_head(shape_from(d), d) * d->num_heads * kDetSlotFloats * sizeof(float);
}

const char* bwd_why_not(const mmn_winattn_desc* d) {
  const char* w = fwd_why_not(d);
  if (w) return w;
  if (d->do_row_stride % 8 || d->dq_row_stride % 8 || d->dk_row_stride % 8 || d->dv_row_stride % 8) return "gradient row stride not 16-byte aligned";
  return nullptr;
}

int winattn_bwd(const mmn_winattn_desc* d, const void* q, const void* k, const void* v, const float* bias, const float* head_scale,
                const float* mask, const void* /*out*/, const float* lse, const void* dout, void* dq, void* dk, void* dv, float* dbias,
                float* dhead_scale, float* dcolsum, float* workspace, cudaStream_t st, char* err, size_t errlen, int* launches) {
  BwdParams P;
  P.S = shape_from(d);
  P.sc = make_sched(P.S, d->batch);
  const int C = d->num_heads * d->head_dim;
  const int B = d->batch;
  if (!make_window_maps(P.q, q, d->q_row_stride, B, C, P.S) || !make_window_maps(P.k, k, d->k_row_stride, B, C, P.S) ||
      !make_window_maps(P.v, v, d->v_row_stride, B, C, P.S) || !make_window_maps(P.dout, dout, d->do_row_stride, B, C, P.S) ||
      !make_window_maps(P.dq, dq, d->dq_row_stride, B, C, P.S) || !make_window_maps(P.dk, dk, d->dk_row_stride, B, C, P.S) ||
      !make_window_maps(P.dv, dv, d->dv_row_stride, B, C, P.S))
    return tensor_map_failed(err, errlen);
  P.nH = d->num_heads;
  P.mask_windows = d->mask_windows > 0 ? d->mask_windows : 1;
  P.scale = d->scale;
  P.bias = bias; P.head_scale = head_scale; P.mask = mask; P.lse = lse;
  P.slab = (long long)P.S.n_windows * d->num_heads * kN;
  P.dbias = bias ? dbias : nullptr;
  P.dhead_scale = d->score_kind == MMN_SCORE_COSINE ? dhead_scale : nullptr;
  P.dcolsum = dcolsum;
  const bool det = d->deterministic != 0;
  P.work = nullptr;
  P.part = nullptr;
  if (det) {                                           // static schedule: no counters; the workspace holds the CTA slots
    if (!workspace || reinterpret_cast<uintptr_t>(workspace) % 16) { snprintf(err, errlen, "workspace missing or misaligned"); return MMN_ERR_CUDA; }
    P.part = workspace;
  } else {
    P.work = arm_work_counters(workspace, st, err, errlen);
    if (!P.work) return MMN_ERR_CUDA;
  }
  const char* trace_path = getenv("MMN_TC_TRACE_BWD");
  P.trace = trace_setup(trace_path, st);

  // [deterministic][cosine][mask kind]
  static void (*const kernels[12])(BwdParams) = {
      winattn_bwd_tc_kernel<false, MMN_MASK_NONE, false>, winattn_bwd_tc_kernel<false, MMN_MASK_SHIFT, false>, winattn_bwd_tc_kernel<false, MMN_MASK_TENSOR, false>,
      winattn_bwd_tc_kernel<true, MMN_MASK_NONE, false>, winattn_bwd_tc_kernel<true, MMN_MASK_SHIFT, false>, winattn_bwd_tc_kernel<true, MMN_MASK_TENSOR, false>,
      winattn_bwd_tc_kernel<false, MMN_MASK_NONE, true>, winattn_bwd_tc_kernel<false, MMN_MASK_SHIFT, true>, winattn_bwd_tc_kernel<false, MMN_MASK_TENSOR, true>,
      winattn_bwd_tc_kernel<true, MMN_MASK_NONE, true>, winattn_bwd_tc_kernel<true, MMN_MASK_SHIFT, true>, winattn_bwd_tc_kernel<true, MMN_MASK_TENSOR, true>};
  P.per_head = bwd_ctas_per_head(P.S, d);
  const int rc = launch_variant(kernels, (det ? 6 : 0) + (d->score_kind == MMN_SCORE_COSINE ? 3 : 0) + d->mask_kind, kBwdSmemBytes,
                                P.per_head * P.nH, kBwdThreads, P, st, "winattn_bwd_tc_kernel", err, errlen);
  if (rc != MMN_OK) return rc;
  ++*launches;
  if (det && (P.dbias || P.dhead_scale || P.dcolsum)) {
    winattn_bwd_det_reduce<<<dim3((kDetSlotFloats / 4 + 31) / 32, P.nH), kDetRedSlices * 32, 0, st>>>(P.part, P.per_head, P.nH, P.dbias,
                                                                                                    P.dcolsum, P.dhead_scale);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
      snprintf(err, errlen, "winattn_bwd_det_reduce: %s", cudaGetErrorString(e));
      return MMN_ERR_CUDA;
    }
    ++*launches;
  }
  if (P.trace.buf) dump_trace(P.trace.buf, trace_path, st);
  return MMN_OK;
}

}}  // namespace mmn::tc
