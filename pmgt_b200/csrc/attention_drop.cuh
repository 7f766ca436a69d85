// Dropout stream of the attn_reg attention family (attention_reg.cu), shared with the attention-map kernel
// (attention_maps.cu), which has to reproduce the mask attn_reg applied, element for element.
#pragma once
#include "common.cuh"

namespace pmgt {

// Dropout of the two probability matrices.  These kernels are bound by instruction issue, and a per-element copy of
// the common.cuh stream (one 32-bit mix per element and site, 64-bit index arithmetic) was 38 % of the forward
// kernel's instructions.  Here ONE word serves element (i, j) of both matrices of an item:
//     w = dmix32((i L + j) ^ k_item) ^ k2,   k_item = fmix32(item * 0x9E3779B9 ^ k1) ^ (item >> 32)
// (k1, k2: the per-(seed, site) keys of common.cuh); P1 keeps the element when the low 16 bits are >= round(p 65536),
// P2 when the high 16 bits are.  Forward and backward (both orientations) evaluate the same function of (item, i, j).
struct DropKey { uint32_t key, k2, thr; float scale; bool on; };
__device__ __forceinline__ DropKey drop_key(uint64_t seed, uint32_t site, float p, long long item) {
  DropKey k;
  const uint32_t k1 = fmix32((uint32_t)seed ^ (site * 0x9E3779B9u) ^ 0x5eedu);
  k.key = fmix32(((uint32_t)item * 0x9E3779B9u) ^ k1) ^ (uint32_t)((unsigned long long)item >> 32);
  k.k2 = fmix32((uint32_t)(seed >> 32) + site);
  k.thr = dropout_threshold(p);
  k.on = p > 0.f;
  k.scale = k.on ? 1.f / (1.f - p) : 1.f;
  return k;
}
// multipliers of element `local` = i L + j for P1 (f1) and P2 (f2)
__device__ __forceinline__ void drop_factors(const DropKey& k, uint32_t local, float& f1, float& f2) {
  if (!k.on) { f1 = 1.f; f2 = 1.f; return; }
  const uint32_t w = dmix32(local ^ k.key) ^ k.k2;
  f1 = (w & 0xffffu) >= k.thr ? k.scale : 0.f;
  f2 = (w >> 16) >= k.thr ? k.scale : 0.f;
}

}  // namespace pmgt
