// Counter-based dropout masks of the training step (internnav_b200/dropout.py holds the site table and the RNG state).
//
// The mask contract, shared by every kernel that applies dropout and restated independently in oracle/philox.py:
//   generator  Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC 2011)
//   key        (seed_lo, seed_hi)
//   counter    (g_lo, g_hi, site | rank << 16, step),  g = e >> 2,  e = the element's row-major linear index in the
//              site's tensor (attention probabilities [B, H, Sq, Sk]: e = ((b H + h) Sq + i) Sk + j)
//   word       output word e & 3 of that Philox block
//   keep rule  dropped iff word < thr, thr = floor(p 2^32) (host, double precision); kept values * scale = float(1/(1-p))
// The RNG state {seed_lo, seed_hi, step, rank} is read through a device pointer at run time, so a captured CUDA graph draws
// the masks of whatever step the buffer holds when it is replayed.  The backward recomputes the forward's mask.
#pragma once
#include <stdint.h>

#include "n1_ops.h"

namespace n1 {

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) k.x += 0x9E3779B9u, k.y += 0xBB67AE85u;
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
  }
  return c;
}

// Per-launch view of one site: the key and the two fixed counter words, loaded once from the device RNG state.
struct DropKey {
  uint2 key;
  uint32_t c2, c3, thr;
  float scale;
};

__device__ __forceinline__ DropKey drop_key(const DropoutDesc& d) {
  const uint4 s = *reinterpret_cast<const uint4*>(d.rng);   // {seed_lo, seed_hi, step, rank}
  DropKey k;
  k.key = make_uint2(s.x, s.y);
  k.c2 = (uint32_t)d.site | (s.w << 16);
  k.c3 = s.z;
  k.thr = d.thr;
  k.scale = d.scale;
  return k;
}

// the four words deciding elements 4g .. 4g + 3
__device__ __forceinline__ uint4 drop_words(const DropKey& k, unsigned long long g) {
  return philox4x32_10(make_uint4((uint32_t)g, (uint32_t)(g >> 32), k.c2, k.c3), k.key);
}

__device__ __forceinline__ uint32_t word_of(const uint4& w, int i) {
  return i == 0 ? w.x : i == 1 ? w.y : i == 2 ? w.z : w.w;
}

// multiplier of element e: 0 (dropped) or scale (kept)
__device__ __forceinline__ float drop_mul(const DropKey& k, unsigned long long e) {
  return word_of(drop_words(k, e >> 2), (int)(e & 3)) < k.thr ? 0.f : k.scale;
}

// multipliers of elements e and e + 1 (one Philox block unless e is the last word of its group)
__device__ __forceinline__ float2 drop_mul2(const DropKey& k, unsigned long long e) {
  const uint4 w = drop_words(k, e >> 2);
  const int i = (int)(e & 3);
  const uint32_t a = word_of(w, i);
  const uint32_t b = i < 3 ? word_of(w, i + 1) : drop_words(k, (e >> 2) + 1).x;
  return make_float2(a < k.thr ? 0.f : k.scale, b < k.thr ? 0.f : k.scale);
}

}  // namespace n1
