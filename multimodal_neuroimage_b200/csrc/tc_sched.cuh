// tc_sched.cuh -- work schedule of the tensor-core window-attention kernels.
//
// Windows are enumerated CLASS-SORTED: all windows that do not wrap around the volume edge first,
// then the seven wrap classes (tc_window.cuh: bit a of the class = the shifted window wraps along
// axis a, which happens exactly for the last window index of a shifted axis).  Inside a class the
// windows form a dense (batch, j0, j1, j2) lattice.  A work ITEM is a pair of consecutive windows
// of one class (the last item of an odd class has one window), so that everything that depends
// on the class -- TMA box shape, piece-major token permutation, shift mask -- is uniform over an
// item, and a CTA, which owns a contiguous (cost-weighted) range of items, sees a class change at
// most seven times.  That is what lets the kernels keep a per-class, pre-permuted, pre-masked
// bias table in shared memory and accumulate the bias gradient in registers without atomics.
#pragma once

#include "tc_window.cuh"

namespace mmn { namespace tc {

struct Sched {
  int cnt[8];        // windows per wrap class
  int dim[8][4];     // lattice extents (batch, j0, j1, j2) of the class
  int wt[8];         // relative cost of one item of the class (partitioning only)
  int n_items;       // sum over classes of ceil(cnt / 2)
  long long total_wt;
};

// Relative item cost by number of wrapped axes (partitioning only), tuned on B200 at BASELINE cfg2.  The same weights set the
// static per-CTA ranges of the deterministic backward, so they are part of what makes its sums reproducible.
constexpr int kSchedWeights[4] = {16, 18, 20, 22};

inline Sched make_sched(const WinShape& S, int batch) {
  Sched sc;
  sc.n_items = 0;
  sc.total_wt = 0;
  for (int c = 0; c < 8; ++c) {
    long long n = batch;
    sc.dim[c][0] = batch;
    for (int a = 0; a < 3; ++a) {
      const int bit = (c >> a) & 1;
      const int d = S.shift[a] ? (bit ? 1 : S.nwin[a] - 1) : (bit ? 0 : S.nwin[a]);
      sc.dim[c][1 + a] = d;
      n *= d;
    }
    sc.cnt[c] = (int)n;
    sc.wt[c] = kSchedWeights[__builtin_popcount(c)];
    sc.n_items += (sc.cnt[c] + 1) / 2;
    sc.total_wt += (long long)((sc.cnt[c] + 1) / 2) * sc.wt[c];
  }
  return sc;
}

// First item of the k-th of G cost-balanced contiguous ranges (k = G gives n_items).
__device__ __forceinline__ int sched_range_begin(const Sched& sc, int k, int G) {
  if (k >= G) return sc.n_items;
  long long target = sc.total_wt * k / G;
  int base = 0;
  for (int c = 0; c < 8; ++c) {
    const int np = (sc.cnt[c] + 1) >> 1;
    const long long cw = (long long)np * sc.wt[c];
    if (target < cw) return base + (int)(target / sc.wt[c]);
    target -= cw;
    base += np;
  }
  return sc.n_items;
}

struct ItemCursor {
  int cls, b, j0, j1, j2;
  int d0, d1, d2;    // lattice extents of the current class (cached: sc.dim[cls] is a dynamically indexed constant load)
  int left;          // windows of this class not yet consumed, including the current item's

  __device__ __forceinline__ void load_dims(const Sched& sc) {
    d0 = sc.dim[cls][1]; d1 = sc.dim[cls][2]; d2 = sc.dim[cls][3];
  }
  __device__ __forceinline__ void seek(const Sched& sc, int item) {
    cls = 0;
    while (cls < 8) {
      const int np = (sc.cnt[cls] + 1) >> 1;
      if (item < np) break;
      item -= np;
      ++cls;
    }
    if (cls == 8) { left = 0; b = j0 = j1 = j2 = 0; d0 = d1 = d2 = 1; return; }
    load_dims(sc);
    int w = 2 * item;
    left = sc.cnt[cls] - w;
    j2 = w % d2; w /= d2;
    j1 = w % d1; w /= d1;
    j0 = w % d0;
    b = w / d0;
  }
  __device__ __forceinline__ void step_window() {
    if (++j2 == d2) {
      j2 = 0;
      if (++j1 == d1) {
        j1 = 0;
        if (++j0 == d0) { j0 = 0; ++b; }
      }
    }
  }
  __device__ __forceinline__ void next_item(const Sched& sc) {
    if (left <= 2) {
      do { ++cls; } while (cls < 8 && sc.cnt[cls] == 0);
      b = j0 = j1 = j2 = 0;
      if (cls < 8) { left = sc.cnt[cls]; load_dims(sc); } else { left = 0; d0 = d1 = d2 = 1; }
    } else {
      step_window();
      step_window();
      left -= 2;
    }
  }
  __device__ __forceinline__ bool slot_valid(int slot) const { return slot == 0 || left >= 2; }
};

// ------------------------------------------------------------------------------------------
// Dynamic schedule.  Each head has one atomic counter per wrap class (work[cls] = next unclaimed item of the class).
// A CTA starts in its HOME class -- the class its cost-weighted static range would start in, so CTAs are spread over
// the classes in proportion to the work -- and claims chunks there; when a class runs dry it moves on to the next one
// (cyclically) and helps there.  Most CTAs therefore see one or two classes (a class change costs a table rebuild and,
// in the backward kernel, a dbias flush: ~3 us), yet all CTAs finish within one chunk of each other whatever the
// per-class item costs are.  The next claim is always in flight while the current chunk is processed.
// All lanes of the producer warp call next() together; lane 0 does the atomics.
// ------------------------------------------------------------------------------------------
constexpr int kWorkDone = 511, kWorkSlotInts = 512;   // counters of one launch: 63 heads x 8 classes (MMN_WINATTN_WORK_BYTES)
struct ClassQueue {
  int cls, pend, tried;
  // items per claim: the wrapped classes are small and their items cost up to 3x (2^k boxes per tile), so their chunks
  // shrink with the number of wrapped axes -- a late chunk of eight 3-axis items was a 30 us tail
  static __device__ __forceinline__ int chunk_of(int chunk, int c) { return max(1, chunk >> __popc(c)); }
  __device__ __forceinline__ void init(const Sched& sc, int home_item, int* work, int chunk, int lane) {
    cls = 0;
    while (cls < 7) {
      const int np = (sc.cnt[cls] + 1) >> 1;
      if (home_item < np) break;
      home_item -= np;
      ++cls;
    }
    tried = 0;
    pend = 0;
    if (lane == 0) pend = atomicAdd(work + cls, chunk_of(chunk, cls));
  }
  // first item (index in the class-sorted list) and length of the next chunk; false when every class is exhausted
  __device__ __forceinline__ bool next(const Sched& sc, int* work, int chunk, int lane, int& item0, int& m) {
    for (;;) {
      const int c0 = __shfl_sync(0xffffffffu, pend, 0);
      const int np = (sc.cnt[cls] + 1) >> 1;
      if (c0 < np) {
        int base = 0;
        for (int c = 0; c < cls; ++c) base += (sc.cnt[c] + 1) >> 1;
        item0 = base + c0;
        m = min(chunk_of(chunk, cls), np - c0);
        if (lane == 0) pend = atomicAdd(work + cls, chunk_of(chunk, cls));
        tried = 0;
        return true;
      }
      if (++tried >= 8) return false;
      cls = (cls + 1) & 7;
      if (lane == 0) pend = atomicAdd(work + cls, chunk_of(chunk, cls));
    }
  }
};

// Shift-mask region id of in-window position p for a window of wrap class `cls`
// (swin_v2_module.py:247-258: along a wrapped axis the last window straddles regions 1 | 2 at
// win - shift; every other window lies in region 0).
__device__ __forceinline__ int class_region_id(const WinShape& S, int cls, int p) {
  const int a2 = p % S.win[2]; const int t = p / S.win[2];
  const int a1 = t % S.win[1]; const int a0 = t / S.win[1];
  const int a[3] = {a0, a1, a2};
  int rid = 0;
#pragma unroll
  for (int x = 0; x < 3; ++x) rid = rid * 3 + ((cls >> x) & 1 ? (a[x] < S.win[x] - S.shift[x] ? 1 : 2) : 0);
  return rid;
}

// The per-CTA class LUTs, filled by threads t, t + nthreads, ...: pos[8][64] tile row -> window position and
// rid[8][64] window position -> shift-mask region id, per wrap class.
__device__ __forceinline__ void fill_class_luts(const WinShape& S, uint8_t* pos, uint8_t* rid, int t, int nthreads) {
  for (int i = t; i < 512; i += nthreads) {
    pos[i] = (uint8_t)piece_position(S, i >> 6, i & 63);
    rid[i] = (uint8_t)class_region_id(S, i >> 6, i & 63);
  }
}

// Per-class additive table in the item's tile order, in the log2 domain:
//   tbl[i][j] = log2(e) * (bias[pos(i)][pos(j)] + (region(pos i) != region(pos j) ? -100 : 0)).
// `bias` is this head's (64,64) fp32 table or null; `pos` the class's 64-entry tile-row -> window-position LUT;
// `rid` the class's window-position -> region-id LUT (class_region_id, tabulated once per CTA).  swz != 0: row i's float4
// j4 is stored at j4 ^ (i & swz) (an unpadded ld = 64 table that rows of a warp still read without bank conflicts).
__device__ __forceinline__ void build_class_table(float* tbl, int ld, const float* bias, const uint8_t* pos, const uint8_t* rid,
                                                  bool shift_mask, int t, int nthreads, int swz = 0) {
  // eight entries per round so that eight L2 loads are in flight per thread (one at a time, a rebuild took ~10 us)
  for (int e0 = t; e0 < kN * kN; e0 += 8 * nthreads) {
    float v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int e = e0 + u * nthreads;
      v[u] = (bias && e < kN * kN) ? __ldg(bias + (int)pos[e >> 6] * kN + pos[e & 63]) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int e = e0 + u * nthreads;
      if (e < kN * kN) {
        const int i = e >> 6, j = e & 63;
        if (shift_mask && rid[pos[i]] != rid[pos[j]]) v[u] -= 100.f;
        tbl[i * ld + ((((j >> 2) ^ (i & swz)) << 2) | (j & 3))] = v[u] * 1.4426950408889634f;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// TMA issue: per-lane box plans.
// An item of wrap class c is 2 windows x T tensors x 2^popc(c) pieces = up to 64 boxes; lane l owns boxes l and l + 32
// (box x = (slot, tensor, piece), piece fastest).  Which tensor map, which piece offset and which shared-memory offset a
// lane's boxes have depends only on the class, so they are tabulated once per class change (BoxPlan::build); per item a
// lane adds its piece offset to its window's start coordinates and issues.  The single-warp integer arithmetic per item
// was what bounded the producer (~1000 cycles per item before, box issue itself ~65 cycles per box).
// ------------------------------------------------------------------------------------------
struct WinStart {              // one window's first token (shifted frame, before the wrap) and sample
  int b, s0, s1, s2;
};

// Start coordinates and linear window index of the cursor's window (slot 0) -- or of the next one (slot 1).
__device__ __forceinline__ WinStart cursor_start(const WinShape& S, const ItemCursor& c, int slot, int& w) {
  ItemCursor t = c;
  if (slot) t.step_window();
  const int i0 = (t.cls & 1) ? S.nwin[0] - 1 : t.j0, i1 = (t.cls & 2) ? S.nwin[1] - 1 : t.j1, i2 = (t.cls & 4) ? S.nwin[2] - 1 : t.j2;
  w = t.b * S.nW + (i0 * S.nwin[1] + i1) * S.nwin[2] + i2;
  WinStart r;
  r.b = t.b;
  r.s0 = i0 * S.win[0] + S.shift[0]; r.s1 = i1 * S.win[1] + S.shift[1]; r.s2 = i2 * S.win[2] + S.shift[2];
  return r;
}
// Where a warp's T tensors go: map[t] = tensor t's eight per-class maps; dst_base[t] / slot_stride[t] = byte offset of its
// tile of slot 0 inside a stage, and the stride to slot 1.
template <int T>
struct BoxLayout {
  const CUtensorMap* map[T];
  int dst_base[T], slot_stride[T];
};

template <int T>
struct BoxPlan {
  int cls = -1, nbox = 0;
  int slot[2], o0[2], o1[2], o2[2], dst[2];
  const CUtensorMap* map[2];

  __device__ __forceinline__ void build(const WinShape& S, int c, int lane, const BoxLayout<T>& L) {
    cls = c;
    const int lp = __popc(c);
    nbox = (2 * T) << lp;
    const int psize_bytes = (kN >> lp) * 64;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int x = lane + 32 * r;
      const int piece = x & ((1 << lp) - 1);
      const int rest = x >> lp;
      const int sl = rest / T, t = rest - sl * T;
      int qq = piece, off[3];
#pragma unroll
      for (int a = 2; a >= 0; --a) {
        const int bit = (c >> a) & 1;
        off[a] = bit ? (qq & 1) * (S.win[a] >> 1) : 0;
        if (bit) qq >>= 1;
      }
      slot[r] = sl; o0[r] = off[0]; o1[r] = off[1]; o2[r] = off[2];
      const CUtensorMap* m = L.map[0];
      int d = L.dst_base[0], ss = L.slot_stride[0];
#pragma unroll
      for (int u = 1; u < T; ++u)
        if (t == u) { m = L.map[u]; d = L.dst_base[u]; ss = L.slot_stride[u]; }
      map[r] = m + c;
      dst[r] = d + sl * ss + piece * psize_bytes;
    }
  }

  template <bool LOAD>
  // map_ofs: tensor maps further on in the same array (dq[8] | dk[8] | dv[8]: the backward's store warp)
  __device__ __forceinline__ void issue(const WinShape& S, const WinStart& w0, const WinStart& w1, int nvalid, int chan, uint8_t* stage,
                                        uint64_t* bar, int lane, int map_ofs = 0) const {
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      if (lane + 32 * r < nbox && slot[r] < nvalid) {
        const WinStart& w = slot[r] ? w1 : w0;
        int c0 = w.s0 + o0[r], c1 = w.s1 + o1[r], c2 = w.s2 + o2[r];
        if (c0 >= S.grid[0]) c0 -= S.grid[0];
        if (c1 >= S.grid[1]) c1 -= S.grid[1];
        if (c2 >= S.grid[2]) c2 -= S.grid[2];
        if (LOAD) tma_load_5d(map[r] + map_ofs, bar, stage + dst[r], chan, c2, c1, c0, w.b);
        else tma_store_5d(map[r] + map_ofs, stage + dst[r], chan, c2, c1, c0, w.b);
      }
    }
  }
};

// ------------------------------------------------------------------------------------------
// Item descriptor ring.  Only the TMA producer knows the schedule: it publishes item n in entry n % DEPTH of a ring in
// shared memory before the barrier arrival that hands over item n's stage, and every other warp reads its items from
// there and stops at the end marker.  The producer may write entry n + DEPTH only once every reader of entry n is past
// it; each kernel's pipeline depth guarantees that (see its producer).
// Layout (kBytes): DEPTH int4 {wrap class, window of slot 0, of slot 1, valid slots}, then DEPTH x 2 int4 {sample, start
// coordinates} of the item's two windows.
// ------------------------------------------------------------------------------------------
struct RingItem {
  int cls;           // wrap class; -1 = end marker
  int win[2];        // linear window index of slot 0, slot 1
  int nvalid;        // valid slots: 1 for the last item of an odd class, else 2
  WinStart ws[2];
  __device__ __forceinline__ bool end() const { return cls < 0; }
};

template <int DEPTH>
struct ItemRing {
  static_assert((DEPTH & (DEPTH - 1)) == 0, "ring depth must be a power of two");
  static constexpr int kBytes = DEPTH * 3 * 16;
  int4* e;

  __device__ __forceinline__ void publish(int n, const RingItem& it) const {
    const int k = n & (DEPTH - 1);
    e[k] = make_int4(it.cls, it.win[0], it.win[1], it.nvalid);
    e[DEPTH + 2 * k] = make_int4(it.ws[0].b, it.ws[0].s0, it.ws[0].s1, it.ws[0].s2);
    e[DEPTH + 2 * k + 1] = make_int4(it.ws[1].b, it.ws[1].s0, it.ws[1].s1, it.ws[1].s2);
  }
  __device__ __forceinline__ void publish_end(int n) const { e[n & (DEPTH - 1)] = make_int4(-1, 0, 0, 0); }
  __device__ __forceinline__ RingItem read(int n) const {
    const int k = n & (DEPTH - 1);
    const int4 d = e[k], a0 = e[DEPTH + 2 * k], a1 = e[DEPTH + 2 * k + 1];
    return {d.x, {d.y, d.z}, d.w, {{a0.x, a0.y, a0.z, a0.w}, {a1.x, a1.y, a1.z, a1.w}}};
  }
};

// ------------------------------------------------------------------------------------------
// The producer's schedule walk: body(n, item) for this CTA's items in order, numbered n = n0, n0 + 1, ...  walk_range takes
// m items of the class-sorted list from item c0 (the deterministic backward's static range); walk_queue takes what the
// ClassQueue hands out.  Both return the number after the last item.  The bodies (the kernels' producers) compute their
// stage, rebuild their BoxPlan on a class change and publish the item.  They capture the parameter block, the shape and
// the plan by reference and everything else, the box layout included, by value: with other capture lists ptxas spilled
// more in the backward kernel, whose warps run at 56 to 104 registers.
// ------------------------------------------------------------------------------------------
template <class Body>
__device__ __forceinline__ int walk_range(const WinShape& S, const Sched& sc, int c0, int m, int n0, Body&& body) {
  ItemCursor cur;
  cur.seek(sc, c0);
  int n = n0;
  for (int t = 0; t < m; ++t, ++n, cur.next_item(sc)) {
    RingItem it;
    it.cls = cur.cls;
    it.nvalid = cur.slot_valid(1) ? 2 : 1;
    it.ws[0] = cursor_start(S, cur, 0, it.win[0]);
    it.ws[1] = cursor_start(S, cur, 1, it.win[1]);
    body(n, it);
  }
  return n;
}

template <class Body>
__device__ __forceinline__ int walk_queue(const WinShape& S, const Sched& sc, int home_item, int* work, int chunk, int lane, Body&& body) {
  ClassQueue wq;
  wq.init(sc, home_item, work, chunk, lane);
  int n = 0;
  for (int c0, m; wq.next(sc, work, chunk, lane, c0, m);) n = walk_range(S, sc, c0, m, n, body);
  return n;
}

}}  // namespace mmn::tc
