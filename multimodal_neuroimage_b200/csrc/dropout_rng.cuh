// dropout_rng.cuh -- the attention-dropout mask (multihead_attention.py:123, F.dropout on the probabilities) as a pure
// function of (seed, offset, item, query i, key j), shared by the generic kernels and the tensor-core MHA kernels so that
// every kernel of a forward / backward pair -- whatever path it runs on -- regenerates the SAME mask without storing it.
// One Philox4x32-10 call covers the 2 x 2 block (i >> 1, j >> 1): word (i & 1) * 2 + (j & 1) decides element (i, j).
// A thread that walks along a row (forward, dQ) and one that walks along a column (dK / dV: lane = key, columns = queries)
// both get two elements per call.  Element kept iff the word's top 24 bits >= ceil(p * 2^24).
// oracle/philox.py is the host-side transcription the tests compare the kernels' masks with.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace mmn {

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x, hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u; k.y += 0xBB67AE85u;
  }
  return c;
}

struct DropoutCfg {
  uint32_t thr;        // ceil(p * 2^24); 0 = no dropout
  uint32_t off_lo;
  uint2 key;
  float inv_keep;      // 1 / (1 - p)
};

// the stream-dependent half of the constants: counter word 3 and the key
__host__ __device__ __forceinline__ void dropout_set_stream(DropoutCfg& c, unsigned long long seed, unsigned long long offset) {
  c.off_lo = (uint32_t)offset;
  c.key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32) ^ (uint32_t)(offset >> 32));
}

inline DropoutCfg make_dropout(float p, unsigned long long seed, unsigned long long offset) {
  DropoutCfg c;
  const float scaled = p * 16777216.0f;                    // exact: a power-of-two multiple
  uint32_t t = (uint32_t)scaled;
  if ((float)t < scaled) ++t;
  c.thr = p > 0.f ? t : 0u;
  dropout_set_stream(c, seed, offset);
  c.inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  return c;
}

// The constants a kernel uses: `c` as make_dropout built them on the host, or -- with dropout on and `rng` given -- with the
// stream read from rng[0] = seed, rng[1] = offset in device memory at kernel entry.  A CUDA graph replays kernel parameters
// unchanged, so this is how a replay gets a fresh mask (the caller rewrites rng before each replay).  thr and inv_keep
// depend on p only and stay host-side.
__device__ __forceinline__ DropoutCfg dropout_at_entry(const DropoutCfg& c, const unsigned long long* rng) {
  DropoutCfg r = c;
  if (c.thr != 0u && rng != nullptr) dropout_set_stream(r, rng[0], rng[1]);
  return r;
}

// the four words of block (i2, j2) = (i >> 1, j >> 1) of attention item `item` (= batch * heads + head)
__device__ __forceinline__ uint4 dropout_block(const DropoutCfg& c, int item, int i2, int j2) {
  return philox4x32_10(make_uint4((uint32_t)j2, (uint32_t)i2, (uint32_t)item, c.off_lo), c.key);
}
__device__ __forceinline__ bool dropout_keep_word(uint32_t w, uint32_t thr) { return (w >> 8) >= thr; }
__device__ __forceinline__ bool dropout_keep(const DropoutCfg& c, int item, int i, int j) {
  const uint4 r = dropout_block(c, item, i >> 1, j >> 1);
  const int w = (i & 1) * 2 + (j & 1);
  return dropout_keep_word(w == 0 ? r.x : w == 1 ? r.y : w == 2 ? r.z : r.w, c.thr);
}

}  // namespace mmn
