// K3 attention core for long neighbour contexts (64 < L <= 128, head size 32 / 64 / 128).  Same algebra as
// attention.cu (dual-softmax "diversity promoting" attention of pmgt/pmgt/modeling_pmgt.py:435-526), laid out like
// attention_reg.cu: one CTA per (sequence, head), one warp per block of 16 query rows, Q / K / V / C (+ dO in the
// backward pass) staged once per CTA with cp.async into padded row tiles, every product an mma.sync m16n8k16 fed by
// ldmatrix.  attn_reg keeps whole 16 x L score rows in accumulator fragments; at L = 128 that is 64 fp32 registers per
// matrix per thread, and its backward pass holds five such matrices.  Here the keys are swept in column chunks, so the
// registers an L x L quantity takes are bounded by the chunk, not by L:
//   * forward, two sweeps per warp: (1) S1 = C C^T and S2 = Q K^T chunk by chunk, with the running row maximum and sum
//     of both softmaxes; (2) the chunk again, A = beta drop(P1) + (1 - beta) drop(P2) from the final statistics,
//     repacked as bf16 A operands of ctx += A V;
//   * backward, three sweeps per warp:
//       statistics      query rows: S1, S2, dA = dO V^T -> softmax maxima and sums, and the row dots
//                       D_i = sum_j g_ij P_ij of the softmax backward (online, rescaled with the maximum); published
//                       in shared memory (6 floats per row)
//       key rows        the transposed blocks K Q^T, C C^T, V dO^T with the query side's statistics -> dV, dK
//       query rows      S1, S2, dA and V dO^T once more -> dQ and the whole of dC: the row half dS1_rj and the column
//                       half dS1_jr of the cosine gradient land in one accumulator
//     Every dqkvc element is written exactly once, without atomics.
// Dropout draws the common.cuh element stream of the generic kernel, element for element: entry (i, j) of P1 of item
// `row * heads + head` is kept iff dropout_keep(seed, site, item L L + i L + j, p), P2 uses site + 1.  A shape that
// moved here from the generic kernel therefore keeps its exact mask.
#include "common.cuh"

namespace pmgt {

namespace {

__device__ __forceinline__ uint32_t lsaddr(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void lldsm4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void lldsm4t(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void lmma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void lcp16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ float lquad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  return v;
}
__device__ __forceinline__ float lquad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
  return v;
}

// The generic kernel's dropout stream (dropout_keep of common.cuh) for one element, evaluating only the one 32-bit
// word of the 8-element block that holds the element's 16-bit field.  `base` = item L L.
struct LongDrop { uint32_t k1a, k2a, k1b, k2b, thr; float scale; bool on; uint64_t base; };
__device__ __forceinline__ LongDrop long_drop(uint64_t seed, uint32_t site, float p, long long item, int L) {
  LongDrop d;
  d.k1a = fmix32((uint32_t)seed ^ (site * 0x9E3779B9u) ^ 0x5eedu);
  d.k2a = fmix32((uint32_t)(seed >> 32) + site);
  d.k1b = fmix32((uint32_t)seed ^ ((site + 1u) * 0x9E3779B9u) ^ 0x5eedu);
  d.k2b = fmix32((uint32_t)(seed >> 32) + site + 1u);
  d.thr = dropout_threshold(p);
  d.on = p > 0.f;
  d.scale = d.on ? 1.f / (1.f - p) : 1.f;
  d.base = (uint64_t)item * (uint64_t)L * (uint64_t)L;
  return d;
}
__device__ __forceinline__ bool long_keep(uint32_t k1, uint32_t k2, uint32_t thr, uint64_t idx) {
  const uint64_t blk = idx >> 3;
  const uint32_t w = dmix32((((uint32_t)blk << 2) + (((uint32_t)idx & 7u) >> 1)) ^ k1) ^ k2 ^ ((uint32_t)(blk >> 30) * 0x9E3779B9u);
  return ((idx & 1) ? (w >> 16) : (w & 0xffffu)) >= thr;
}
// multipliers of element local = i L + j for P1 (f1) and P2 (f2)
__device__ __forceinline__ void long_factors(const LongDrop& d, uint32_t local, float& f1, float& f2) {
  if (!d.on) { f1 = 1.f; f2 = 1.f; return; }
  const uint64_t idx = d.base + local;
  f1 = long_keep(d.k1a, d.k2a, d.thr, idx) ? d.scale : 0.f;
  f2 = long_keep(d.k1b, d.k2b, d.thr, idx) ? d.scale : 0.f;
}
__device__ __forceinline__ float long_factor1(const LongDrop& d, uint32_t local) {
  if (!d.on) return 1.f;
  return long_keep(d.k1a, d.k2a, d.thr, d.base + local) ? d.scale : 0.f;
}

template <int DH, int MT>
struct LongCfg {
  static constexpr int LP = 16 * MT;   // padded sequence length
  static constexpr int KS = DH / 16;   // k-steps over the head dimension
  static constexpr int ON = DH / 8;    // 8-wide column tiles of an output row block
  static constexpr int RS = DH + 8;    // row pitch of a staged tile (bf16 elements): 16-byte aligned, ldmatrix conflict-free
  static constexpr int THREADS = 32 * MT;
  static constexpr int TILE = LP * RS;  // elements
  // column chunks, in 16-column pairs: the forward sweeps hold two chunk matrices, the backward sweeps three or four
  // next to two DH-wide accumulators
  static constexpr int FWD_CP = 4;
  static constexpr int BWD_CP = DH == 128 ? 1 : 2;
  // CTAs per SM the launch bounds ask for: two where the registers that leaves (204 a thread at MT <= 6) hold the kernel
  // without spilling (dh = 128 fills the shared memory with one CTA anyway), one elsewhere
  static constexpr int MINB_FWD = DH < 128 && MT <= 6 ? 2 : 1;
  static constexpr int MINB_BWD = DH == 32 && MT <= 6 ? 2 : 1;
  static constexpr size_t kFwdSmem = 4 * (size_t)TILE * 2 + 2 * LP * 4;
  static constexpr size_t kBwdSmem = 5 * (size_t)TILE * 2 + 8 * LP * 4;
};

// rows [0, L) of one head of a [T][ld] bf16 matrix -> tile[LP][RS]; rows [L, LP) are zero
template <int DH, int MT>
__device__ __forceinline__ void stage_long(uint16_t* tile, const uint16_t* __restrict__ src, long long ld, int L, int tid) {
  using Cf = LongCfg<DH, MT>;
  constexpr int CPR = DH / 8;
  for (int e = tid; e < Cf::LP * CPR; e += Cf::THREADS) {
    const int i = e / CPR, c = e - i * CPR;
    uint16_t* dst = tile + i * Cf::RS + c * 8;
    if (i < L) lcp16(lsaddr(dst), src + (long long)i * ld + c * 8);
    else *reinterpret_cast<uint4*>(dst) = make_uint4(0u, 0u, 0u, 0u);
  }
}

// D[n][*] = A_rows(16 x DH, tile rows a_row0..) . B(tile rows col0 .. col0 + 16 CP)^T; pairs p >= npl (beyond the
// padded length) are left zero
template <int DH, int CP>
__device__ __forceinline__ void chunk_nt(float (&d)[2 * CP][4], const uint16_t* A, int a_row0, const uint16_t* B, int col0,
                                         int npl, int lane) {
  constexpr int RS = DH + 8;
#pragma unroll
  for (int n = 0; n < 2 * CP; ++n) { d[n][0] = 0.f; d[n][1] = 0.f; d[n][2] = 0.f; d[n][3] = 0.f; }
#pragma unroll
  for (int ks = 0; ks < DH / 16; ++ks) {
    uint32_t af[4];
    lldsm4(lsaddr(A + (a_row0 + (lane & 15)) * RS + ks * 16 + (lane >> 4) * 8), af);
#pragma unroll
    for (int np = 0; np < CP; ++np) if (np < npl) {
      uint32_t bf[4];
      lldsm4(lsaddr(B + (col0 + np * 16 + (lane & 7) + ((lane >> 4) << 3)) * RS + ks * 16 + ((lane >> 3) & 1) * 8), bf);
      lmma(d[2 * np], af, bf[0], bf[1]);
      lmma(d[2 * np + 1], af, bf[2], bf[3]);
    }
  }
}

// O[on][*] += P(16 x 16 CP chunk, accumulator fragments, bf16-rounded) . X(tile rows col0 .., DH)
template <int DH, int CP>
__device__ __forceinline__ void chunk_pv(float (&o)[DH / 8][4], const float (&pm)[2 * CP][4], const uint16_t* X, int col0,
                                         int npl, int lane) {
  constexpr int RS = DH + 8;
#pragma unroll
  for (int kk = 0; kk < CP; ++kk) if (kk < npl) {
    uint32_t af[4];
    af[0] = pack_bf16x2(pm[2 * kk][0], pm[2 * kk][1]);
    af[1] = pack_bf16x2(pm[2 * kk][2], pm[2 * kk][3]);
    af[2] = pack_bf16x2(pm[2 * kk + 1][0], pm[2 * kk + 1][1]);
    af[3] = pack_bf16x2(pm[2 * kk + 1][2], pm[2 * kk + 1][3]);
#pragma unroll
    for (int op = 0; op < DH / 16; ++op) {
      uint32_t bf[4];
      lldsm4t(lsaddr(X + (col0 + kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * RS + op * 16 + (lane >> 4) * 8), bf);
      lmma(o[2 * op], af, bf[0], bf[1]);
      lmma(o[2 * op + 1], af, bf[2], bf[3]);
    }
  }
}

template <int ON>
__device__ __forceinline__ void zero_long(float (&o)[ON][4]) {
#pragma unroll
  for (int n = 0; n < ON; ++n) { o[n][0] = 0.f; o[n][1] = 0.f; o[n][2] = 0.f; o[n][3] = 0.f; }
}

// rows r0 / r1 of an output block, scaled, as bf16 pairs
template <int ON>
__device__ __forceinline__ void store_long(uint16_t* dst0, uint16_t* dst1, bool ok0, bool ok1, const float (&o)[ON][4], float scale, int t) {
#pragma unroll
  for (int n = 0; n < ON; ++n) {
    const int col = n * 8 + 2 * t;
    if (ok0) *reinterpret_cast<uint32_t*>(dst0 + col) = pack_bf16x2(o[n][0] * scale, o[n][1] * scale);
    if (ok1) *reinterpret_cast<uint32_t*>(dst1 + col) = pack_bf16x2(o[n][2] * scale, o[n][3] * scale);
  }
}

// 1 / |c_i| and the additive key mask of every row; padded rows: norm 1, mask -inf (their keys drop out of every softmax)
template <int DH, int MT>
__device__ __forceinline__ void long_norms(const uint16_t* sC, const float* __restrict__ mask_row, int L, int tid, float* nrm, float* madd) {
  using Cf = LongCfg<DH, MT>;
  for (int i = tid; i < Cf::LP; i += Cf::THREADS) {
    float s = 0.f;
    if (i < L) {
#pragma unroll
      for (int c = 0; c < DH; c += 2) {
        float x, y;
        unpack_bf16x2(*reinterpret_cast<const uint32_t*>(sC + i * Cf::RS + c), x, y);
        s = fmaf(x, x, s);
        s = fmaf(y, y, s);
      }
    }
    nrm[i] = i < L ? 1.f / sqrtf(s) : 1.f;   // RECIPROCAL norm
    madd[i] = i < L ? (1.f - mask_row[i]) * -10000.f : -INFINITY;
  }
}

// the two raw scores of element (i, j) of a query-row block: s1 <- 1 - cos + [i == j] + madd_j, s2 <- s2 / sqrt(dh) + madd_j;
// column tiles beyond the padded length (nt >= 2 npl, in the last chunk) get -inf and drop out of the softmaxes
template <int CP>
__device__ __forceinline__ void long_scores(float (&s1)[2 * CP][4], float (&s2)[2 * CP][4], int col0, int npl, int i0, int i1,
                                            int t, float rn0, float rn1, const float* nrm, const float* madd, float inv_sqrt_dh) {
#pragma unroll
  for (int nt = 0; nt < 2 * CP; ++nt) {
    if (nt >= 2 * npl) {
#pragma unroll
      for (int e = 0; e < 4; ++e) { s1[nt][e] = -INFINITY; s2[nt][e] = -INFINITY; }
      continue;
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int j = col0 + nt * 8 + 2 * t + (e & 1);
      const int i = e < 2 ? i0 : i1;
      const float cs = s1[nt][e] * (e < 2 ? rn0 : rn1) * nrm[j];
      s1[nt][e] = 1.f - cs + (i == j ? 1.f : 0.f) + madd[j];
      s2[nt][e] = s2[nt][e] * inv_sqrt_dh + madd[j];
    }
  }
}

// maximum of rows a (e < 2) and b (e >= 2) of a chunk, over the quad
template <int CP>
__device__ __forceinline__ void chunk_max(const float (&s)[2 * CP][4], float& ma, float& mb) {
  ma = -INFINITY; mb = -INFINITY;
#pragma unroll
  for (int nt = 0; nt < 2 * CP; ++nt) {
    ma = fmaxf(ma, fmaxf(s[nt][0], s[nt][1]));
    mb = fmaxf(mb, fmaxf(s[nt][2], s[nt][3]));
  }
  ma = lquad_max(ma); mb = lquad_max(mb);
}

// ---------------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------------
template <int DH, int MT>
__global__ void __launch_bounds__(32 * MT, LongCfg<DH, MT>::MINB_FWD) attn_long_fwd_kernel(const pmgt_attn_args a) {
  using Cf = LongCfg<DH, MT>;
  constexpr int CP = Cf::FWD_CP;
  extern __shared__ __align__(16) unsigned char smem[];
  uint16_t* sQ = reinterpret_cast<uint16_t*>(smem);
  uint16_t* sK = sQ + Cf::TILE;
  uint16_t* sV = sK + Cf::TILE;
  uint16_t* sC = sV + Cf::TILE;
  float* nrm = reinterpret_cast<float*>(sC + Cf::TILE);
  float* madd = nrm + Cf::LP;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  const int L = a.L, H = a.H, heads = a.heads;
  const long long item = blockIdx.x;
  const long long row = item / heads;
  const int head = (int)(item - row * heads);
  const long long ld = 4ll * H;
  const uint16_t* src = a.qkvc + row * L * ld + head * DH;

  stage_long<DH, MT>(sQ, src, ld, L, tid);
  stage_long<DH, MT>(sK, src + H, ld, L, tid);
  stage_long<DH, MT>(sV, src + 2 * H, ld, L, tid);
  stage_long<DH, MT>(sC, src + 3 * H, ld, L, tid);
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  long_norms<DH, MT>(sC, a.mask + row * L, L, tid, nrm, madd);
  __syncthreads();

  const int i0 = warp * 16 + g, i1 = i0 + 8;
  const float inv_sqrt_dh = rsqrtf((float)DH);
  const float rn0 = nrm[i0], rn1 = nrm[i1];
  // sweep 1: running maxima and (per-thread partial) sums of both softmaxes
  float m1a = -INFINITY, m1b = -INFINITY, m2a = -INFINITY, m2b = -INFINITY;
  float z1a = 0.f, z1b = 0.f, z2a = 0.f, z2b = 0.f;
#pragma unroll 1
  for (int col0 = 0; col0 < Cf::LP; col0 += 16 * CP) {
    const int npl = (Cf::LP - col0) >> 4;
    float s1[2 * CP][4], s2[2 * CP][4];
    chunk_nt<DH, CP>(s1, sC, warp * 16, sC, col0, npl, lane);
    chunk_nt<DH, CP>(s2, sQ, warp * 16, sK, col0, npl, lane);
    long_scores<CP>(s1, s2, col0, npl, i0, i1, t, rn0, rn1, nrm, madd, inv_sqrt_dh);
    float c1a, c1b, c2a, c2b;
    chunk_max<CP>(s1, c1a, c1b);
    chunk_max<CP>(s2, c2a, c2b);
    // every chunk holds a real key (col0 < L), so the new maxima are finite
    c1a = fmaxf(c1a, m1a); c1b = fmaxf(c1b, m1b); c2a = fmaxf(c2a, m2a); c2b = fmaxf(c2b, m2b);
    z1a *= __expf(m1a - c1a); z1b *= __expf(m1b - c1b); z2a *= __expf(m2a - c2a); z2b *= __expf(m2b - c2b);
    m1a = c1a; m1b = c1b; m2a = c2a; m2b = c2b;
#pragma unroll
    for (int nt = 0; nt < 2 * CP; ++nt) {
      z1a += __expf(s1[nt][0] - m1a) + __expf(s1[nt][1] - m1a);
      z1b += __expf(s1[nt][2] - m1b) + __expf(s1[nt][3] - m1b);
      z2a += __expf(s2[nt][0] - m2a) + __expf(s2[nt][1] - m2a);
      z2b += __expf(s2[nt][2] - m2b) + __expf(s2[nt][3] - m2b);
    }
  }
  z1a = 1.f / lquad_sum(z1a); z1b = 1.f / lquad_sum(z1b); z2a = 1.f / lquad_sum(z2a); z2b = 1.f / lquad_sum(z2b);
  // sweep 2: A = beta drop(P1) + (1 - beta) drop(P2), ctx += A V
  const LongDrop dk = long_drop(a.dropout_seed, a.dropout_site, a.dropout_p, item, L);
  const float beta = a.beta;
  const uint32_t dbase0 = (uint32_t)(i0 * L), dbase1 = (uint32_t)(i1 * L);
  float o[Cf::ON][4];
  zero_long<Cf::ON>(o);
#pragma unroll 1
  for (int col0 = 0; col0 < Cf::LP; col0 += 16 * CP) {
    const int npl = (Cf::LP - col0) >> 4;
    float s1[2 * CP][4], s2[2 * CP][4];
    chunk_nt<DH, CP>(s1, sC, warp * 16, sC, col0, npl, lane);
    chunk_nt<DH, CP>(s2, sQ, warp * 16, sK, col0, npl, lane);
    long_scores<CP>(s1, s2, col0, npl, i0, i1, t, rn0, rn1, nrm, madd, inv_sqrt_dh);
#pragma unroll
    for (int nt = 0; nt < 2 * CP; ++nt) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int j = col0 + nt * 8 + 2 * t + (e & 1);
        float f1, f2;
        long_factors(dk, (e < 2 ? dbase0 : dbase1) + (uint32_t)j, f1, f2);
        const float p1 = __expf(s1[nt][e] - (e < 2 ? m1a : m1b)) * (e < 2 ? z1a : z1b) * f1;
        const float p2 = __expf(s2[nt][e] - (e < 2 ? m2a : m2b)) * (e < 2 ? z2a : z2b) * f2;
        s1[nt][e] = beta * p1 + (1.f - beta) * p2;
      }
    }
    chunk_pv<DH, CP>(o, s1, sV, col0, npl, lane);
  }
  uint16_t* dst = a.ctx + row * L * (long long)H + head * DH;
  store_long<Cf::ON>(dst + (long long)i0 * H, dst + (long long)i1 * H, i0 < L, i1 < L, o, 1.f, t);
}

// ---------------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------------
template <int DH, int MT>
__global__ void __launch_bounds__(32 * MT, LongCfg<DH, MT>::MINB_BWD) attn_long_bwd_kernel(const pmgt_attn_args a) {
  using Cf = LongCfg<DH, MT>;
  constexpr int CP = Cf::BWD_CP;
  extern __shared__ __align__(16) unsigned char smem[];
  uint16_t* sQ = reinterpret_cast<uint16_t*>(smem);
  uint16_t* sK = sQ + Cf::TILE;
  uint16_t* sV = sK + Cf::TILE;
  uint16_t* sC = sV + Cf::TILE;
  uint16_t* sO = sC + Cf::TILE;  // dctx
  float* nrm = reinterpret_cast<float*>(sO + Cf::TILE);
  float* madd = nrm + Cf::LP;
  float* st_m1 = madd + Cf::LP;   // per query row: softmax maxima, 1 / sums, row dots of the softmax backward
  float* st_z1 = st_m1 + Cf::LP;
  float* st_m2 = st_z1 + Cf::LP;
  float* st_z2 = st_m2 + Cf::LP;
  float* st_r1 = st_z2 + Cf::LP;
  float* st_r2 = st_r1 + Cf::LP;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  const int L = a.L, H = a.H, heads = a.heads;
  const long long item = blockIdx.x;
  const long long row = item / heads;
  const int head = (int)(item - row * heads);
  const long long ld = 4ll * H;
  const uint16_t* src = a.qkvc + row * L * ld + head * DH;

  stage_long<DH, MT>(sQ, src, ld, L, tid);
  stage_long<DH, MT>(sK, src + H, ld, L, tid);
  stage_long<DH, MT>(sV, src + 2 * H, ld, L, tid);
  stage_long<DH, MT>(sC, src + 3 * H, ld, L, tid);
  stage_long<DH, MT>(sO, a.dctx + row * L * (long long)H + head * DH, (long long)H, L, tid);
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  long_norms<DH, MT>(sC, a.mask + row * L, L, tid, nrm, madd);
  __syncthreads();

  const int r0 = warp * 16 + g, r1 = r0 + 8;  // this thread's two rows: queries, then keys, then queries again
  const float inv_sqrt_dh = rsqrtf((float)DH);
  const float rn0 = nrm[r0], rn1 = nrm[r1];
  const LongDrop dk = long_drop(a.dropout_seed, a.dropout_site, a.dropout_p, item, L);
  const float beta = a.beta;
  uint16_t* dst = a.dqkvc + row * L * ld + head * DH;
  uint16_t* d0 = dst + (long long)r0 * ld;
  uint16_t* d1 = dst + (long long)r1 * ld;
  const bool ok0 = r0 < L, ok1 = r1 < L;
  const uint32_t dbase0 = (uint32_t)(r0 * L), dbase1 = (uint32_t)(r1 * L);

  // ===================== sweep 1: statistics of the query rows =====================
  float m1a = -INFINITY, m1b = -INFINITY, m2a = -INFINITY, m2b = -INFINITY;
  float z1a = 0.f, z1b = 0.f, z2a = 0.f, z2b = 0.f;
  float u1a = 0.f, u1b = 0.f, u2a = 0.f, u2b = 0.f;   // sum_j g_ij e^{S_ij - m_i}
#pragma unroll 1
  for (int col0 = 0; col0 < Cf::LP; col0 += 16 * CP) {
    const int npl = (Cf::LP - col0) >> 4;
    float s1[2 * CP][4], s2[2 * CP][4], dA[2 * CP][4];
    chunk_nt<DH, CP>(s1, sC, warp * 16, sC, col0, npl, lane);
    chunk_nt<DH, CP>(s2, sQ, warp * 16, sK, col0, npl, lane);
    chunk_nt<DH, CP>(dA, sO, warp * 16, sV, col0, npl, lane);
    long_scores<CP>(s1, s2, col0, npl, r0, r1, t, rn0, rn1, nrm, madd, inv_sqrt_dh);
    float c1a, c1b, c2a, c2b;
    chunk_max<CP>(s1, c1a, c1b);
    chunk_max<CP>(s2, c2a, c2b);
    c1a = fmaxf(c1a, m1a); c1b = fmaxf(c1b, m1b); c2a = fmaxf(c2a, m2a); c2b = fmaxf(c2b, m2b);
    {
      const float x1a = __expf(m1a - c1a), x1b = __expf(m1b - c1b), x2a = __expf(m2a - c2a), x2b = __expf(m2b - c2b);
      z1a *= x1a; u1a *= x1a; z1b *= x1b; u1b *= x1b; z2a *= x2a; u2a *= x2a; z2b *= x2b; u2b *= x2b;
    }
    m1a = c1a; m1b = c1b; m2a = c2a; m2b = c2b;
#pragma unroll
    for (int nt = 0; nt < 2 * CP; ++nt) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int j = col0 + nt * 8 + 2 * t + (e & 1);
        float f1, f2;
        long_factors(dk, (e < 2 ? dbase0 : dbase1) + (uint32_t)j, f1, f2);
        const float e1 = __expf(s1[nt][e] - (e < 2 ? m1a : m1b));
        const float e2 = __expf(s2[nt][e] - (e < 2 ? m2a : m2b));
        const float ga = beta * dA[nt][e] * f1, gb = (1.f - beta) * dA[nt][e] * f2;
        if (e < 2) { z1a += e1; z2a += e2; u1a = fmaf(ga, e1, u1a); u2a = fmaf(gb, e2, u2a); }
        else { z1b += e1; z2b += e2; u1b = fmaf(ga, e1, u1b); u2b = fmaf(gb, e2, u2b); }
      }
    }
  }
  z1a = 1.f / lquad_sum(z1a); z1b = 1.f / lquad_sum(z1b); z2a = 1.f / lquad_sum(z2a); z2b = 1.f / lquad_sum(z2b);
  const float q1a = lquad_sum(u1a) * z1a, q1b = lquad_sum(u1b) * z1b;   // D1 / D2 of rows r0 / r1
  const float q2a = lquad_sum(u2a) * z2a, q2b = lquad_sum(u2b) * z2b;
  if (t == 0) {
    st_m1[r0] = m1a; st_z1[r0] = z1a; st_m2[r0] = m2a; st_z2[r0] = z2a; st_r1[r0] = q1a; st_r2[r0] = q2a;
    st_m1[r1] = m1b; st_z1[r1] = z1b; st_m2[r1] = m2b; st_z2[r1] = z2b; st_r1[r1] = q1b; st_r2[r1] = q2b;
  }
  __syncthreads();  // every query row's statistics are in shared memory

  // ===================== sweep 2: rows = keys, columns = queries -> dV, dK =====================
  {
    const float ma0 = madd[r0], ma1 = madd[r1];
    float dv[Cf::ON][4], dkk[Cf::ON][4];
    zero_long<Cf::ON>(dv);
    zero_long<Cf::ON>(dkk);
#pragma unroll 1
  for (int col0 = 0; col0 < Cf::LP; col0 += 16 * CP) {
      const int npl = (Cf::LP - col0) >> 4;
      float gr[2 * CP][4], s2[2 * CP][4], dA[2 * CP][4];
      chunk_nt<DH, CP>(gr, sC, warp * 16, sC, col0, npl, lane);   // C_j . C_i
      chunk_nt<DH, CP>(s2, sK, warp * 16, sQ, col0, npl, lane);   // K_j . Q_i
      chunk_nt<DH, CP>(dA, sV, warp * 16, sO, col0, npl, lane);   // V_j . dO_i
#pragma unroll
      for (int nt = 0; nt < 2 * CP; ++nt) if (nt < 2 * npl) {   // tiles past LP: chunk_pv skips them
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int i = col0 + nt * 8 + 2 * t + (e & 1);   // query (column)
          const int j = e < 2 ? r0 : r1;                   // key (row)
          const float rnj = e < 2 ? rn0 : rn1;
          const float mj = e < 2 ? ma0 : ma1;
          const bool live = i < L;                         // padded queries contribute nothing
          const float cs = gr[nt][e] * rnj * nrm[i];
          const float p1 = live ? __expf(1.f - cs + (i == j ? 1.f : 0.f) + mj - st_m1[i]) * st_z1[i] : 0.f;
          const float p2 = live ? __expf(s2[nt][e] * inv_sqrt_dh + mj - st_m2[i]) * st_z2[i] : 0.f;
          float f1, f2;
          long_factors(dk, (uint32_t)(i * L + j), f1, f2);
          gr[nt][e] = beta * p1 * f1 + (1.f - beta) * p2 * f2;             // A_ij
          s2[nt][e] = live ? p2 * ((1.f - beta) * dA[nt][e] * f2 - st_r2[i]) : 0.f;   // dS2_ij
        }
      }
      chunk_pv<DH, CP>(dv, gr, sO, col0, npl, lane);    // dV_j = sum_i A_ij dO_i
      chunk_pv<DH, CP>(dkk, s2, sQ, col0, npl, lane);   // dK_j = sum_i dS2_ij Q_i / sqrt(dh)
    }
    store_long<Cf::ON>(d0 + 2 * H, d1 + 2 * H, ok0, ok1, dv, 1.f, t);
    store_long<Cf::ON>(d0 + H, d1 + H, ok0, ok1, dkk, inv_sqrt_dh, t);
  }

  // ===================== sweep 3: rows = queries -> dQ and dC =====================
  {
    float dq[Cf::ON][4], accC[Cf::ON][4];   // accC_r = sum_j (dS1_rj + dS1_jr) / (n_r n_j) C_j
    zero_long<Cf::ON>(dq);
    zero_long<Cf::ON>(accC);
    float rc0 = 0.f, rc1 = 0.f;              // sum_j (dS1_rj + dS1_jr) cos_rj
    const float ma0 = madd[r0], ma1 = madd[r1];
#pragma unroll 1
  for (int col0 = 0; col0 < Cf::LP; col0 += 16 * CP) {
      const int npl = (Cf::LP - col0) >> 4;
      float gr[2 * CP][4], s2[2 * CP][4], dA[2 * CP][4], dAt[2 * CP][4];
      chunk_nt<DH, CP>(gr, sC, warp * 16, sC, col0, npl, lane);    // C_r . C_j
      chunk_nt<DH, CP>(s2, sQ, warp * 16, sK, col0, npl, lane);    // Q_r . K_j
      chunk_nt<DH, CP>(dA, sO, warp * 16, sV, col0, npl, lane);    // dO_r . V_j
      chunk_nt<DH, CP>(dAt, sV, warp * 16, sO, col0, npl, lane);   // V_r . dO_j
#pragma unroll
      for (int nt = 0; nt < 2 * CP; ++nt) if (nt < 2 * npl) {   // tiles past LP: chunk_pv skips them
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int j = col0 + nt * 8 + 2 * t + (e & 1);
          const bool lo = e < 2;
          const int r = lo ? r0 : r1;
          const float rnr = lo ? rn0 : rn1, rnj = nrm[j];
          const float cs = gr[nt][e] * rnr * rnj;
          // (r, j): r the query
          const float p1 = __expf(1.f - cs + (r == j ? 1.f : 0.f) + madd[j] - (lo ? m1a : m1b)) * (lo ? z1a : z1b);
          const float p2 = __expf(s2[nt][e] * inv_sqrt_dh + madd[j] - (lo ? m2a : m2b)) * (lo ? z2a : z2b);
          float f1, f2;
          long_factors(dk, (lo ? dbase0 : dbase1) + (uint32_t)j, f1, f2);
          const float ds1 = p1 * (beta * dA[nt][e] * f1 - (lo ? q1a : q1b));
          s2[nt][e] = p2 * ((1.f - beta) * dA[nt][e] * f2 - (lo ? q2a : q2b));   // dS2_rj
          // (j, r): j the query, r the key
          float ds1t = 0.f;
          if (j < L) {
            const float pt = __expf(1.f - cs + (r == j ? 1.f : 0.f) + (lo ? ma0 : ma1) - st_m1[j]) * st_z1[j];
            const float ft = long_factor1(dk, (uint32_t)(j * L + r));
            ds1t = pt * (beta * dAt[nt][e] * ft - st_r1[j]);
          }
          const float dsum = ds1 + ds1t;
          if (lo) rc0 = fmaf(dsum, cs, rc0); else rc1 = fmaf(dsum, cs, rc1);
          gr[nt][e] = dsum * rnr * rnj;
        }
      }
      chunk_pv<DH, CP>(dq, s2, sK, col0, npl, lane);     // dQ_r = sum_j dS2_rj K_j / sqrt(dh)
      chunk_pv<DH, CP>(accC, gr, sC, col0, npl, lane);
    }
    store_long<Cf::ON>(d0, d1, ok0, ok1, dq, inv_sqrt_dh, t);
    // dC_r = -accC_r + (rc_r / n_r^2) C_r
    rc0 = lquad_sum(rc0) * rn0 * rn0;
    rc1 = lquad_sum(rc1) * rn1 * rn1;
#pragma unroll
    for (int n = 0; n < Cf::ON; ++n) {
      const int col = n * 8 + 2 * t;
      float c00, c01, c10, c11;
      unpack_bf16x2(*reinterpret_cast<const uint32_t*>(sC + r0 * Cf::RS + col), c00, c01);
      unpack_bf16x2(*reinterpret_cast<const uint32_t*>(sC + r1 * Cf::RS + col), c10, c11);
      if (ok0) *reinterpret_cast<uint32_t*>(d0 + 3 * H + col) = pack_bf16x2(fmaf(rc0, c00, -accC[n][0]), fmaf(rc0, c01, -accC[n][1]));
      if (ok1) *reinterpret_cast<uint32_t*>(d1 + 3 * H + col) = pack_bf16x2(fmaf(rc1, c10, -accC[n][2]), fmaf(rc1, c11, -accC[n][3]));
    }
  }
}

template <int DH, int MT, bool BWD>
int launch_long(const pmgt_attn_args* a, cudaStream_t st) {
  using Cf = LongCfg<DH, MT>;
  const size_t smem = BWD ? Cf::kBwdSmem : Cf::kFwdSmem;
  static unsigned long long configured = 0;
  if (first_use_on_device(configured)) {
    if (BWD) PMGT_CHECK_CUDA(cudaFuncSetAttribute(attn_long_bwd_kernel<DH, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    else PMGT_CHECK_CUDA(cudaFuncSetAttribute(attn_long_fwd_kernel<DH, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  const long long items = a->rows * a->heads;  // <= 2^31 - 1 (attn_family in attention.cu)
  if (BWD) attn_long_bwd_kernel<DH, MT><<<(unsigned)items, 32 * MT, smem, st>>>(*a);
  else attn_long_fwd_kernel<DH, MT><<<(unsigned)items, 32 * MT, smem, st>>>(*a);
  PMGT_LAUNCH_CHECK();
  return PMGT_OK;
}

// 64 < L <= 128, head size 32 / 64 / 128
template <bool BWD>
int dispatch_long(const pmgt_attn_args* a, cudaStream_t st) {
  const int dh = a->H / a->heads;
  const int mt = a->L > 64 && a->L <= 128 ? (a->L + 15) / 16 : 0;
#define PMGT_LONG_CASE(D, M) if (dh == D && mt == M) return launch_long<D, M, BWD>(a, st)
  PMGT_LONG_CASE(32, 5); PMGT_LONG_CASE(32, 6); PMGT_LONG_CASE(32, 7); PMGT_LONG_CASE(32, 8);
  PMGT_LONG_CASE(64, 5); PMGT_LONG_CASE(64, 6); PMGT_LONG_CASE(64, 7); PMGT_LONG_CASE(64, 8);
  PMGT_LONG_CASE(128, 5); PMGT_LONG_CASE(128, 6); PMGT_LONG_CASE(128, 7); PMGT_LONG_CASE(128, 8);
#undef PMGT_LONG_CASE
  set_error("attn_long: no kernel for L=%d, head size %d", a->L, dh);
  return PMGT_ERR_INVALID;
}

}  // namespace

int attn_long_fwd(const pmgt_attn_args* a, cudaStream_t st) { return dispatch_long<false>(a, st); }
int attn_long_bwd(const pmgt_attn_args* a, cudaStream_t st) { return dispatch_long<true>(a, st); }

}  // namespace pmgt
