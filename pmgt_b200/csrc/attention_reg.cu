// K3 attention core for medium sequence lengths (8 < L <= 64), register-resident: BASELINE config 5 (32 sampled
// neighbours, L = 33, 12 heads of 64).  Same algebra as attention.cu (dual-softmax "diversity promoting" attention of
// pmgt/pmgt/modeling_pmgt.py:435-526).  attention_mid.cu kept the L x L score matrices as fp32 in shared memory and
// ran softmax, dropout and the softmax / cosine backward as scalar passes between block barriers (0.08 of the HBM
// roofline); here every L x L quantity lives in mma.sync accumulator fragments from the product that creates it to the
// product that consumes it:
//   * one CTA per (sequence, head), one WARP per block of 16 rows (L = 33 -> 3 warps); K, V, C (+ Q, dO in the
//     backward pass) are staged once with cp.async into padded row tiles shared by the warps;
//   * forward: S1 = C C^T and S2 = Q K^T row blocks (m16n8k16, ldmatrix operands), cosine / mask / softmax / dropout
//     on the accumulator registers (row reductions = two quad shuffles), the accumulators repacked as the A operand
//     of A V;
//   * backward in two orientations per warp, so that no L x L matrix is ever transposed or exchanged:
//       query-row orientation  P1, P2, dA = dO V^T -> softmax statistics + row dots (to shared memory, 6 floats per
//                              row), dS1, dS2 -> dQ and the row half of dC;
//       key-row orientation    the same blocks transposed (K Q^T, V dO^T, C C^T) with the other side's statistics
//                              -> dV, dK and the column half of dC, which lands in the same accumulators.
#include "attention_drop.cuh"

#ifndef PMGT_REG_BWD_REGS
#define PMGT_REG_BWD_REGS 216   // register budget per thread the backward kernel's launch bounds aim at
#endif

namespace pmgt {

namespace {

__device__ __forceinline__ uint32_t rsaddr(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void rldsm4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void rldsm4t(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void rmma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void rcp16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  return v;
}
__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
  return v;
}

// Dropout: DropKey / drop_key / drop_factors (attention_drop.cuh), one word per element (i, j) for both matrices.

template <int DH, int MT>
struct RegCfg {
  static constexpr int LP = 16 * MT;   // padded sequence length
  static constexpr int NT = 2 * MT;    // 8-wide column tiles of an L x L block row
  static constexpr int KS = DH / 16;   // k-steps over the head dimension
  static constexpr int ON = DH / 8;    // 8-wide column tiles of an output row block
  static constexpr int RS = DH + 8;    // row pitch of a staged tile (bf16 elements): 16-byte aligned, ldmatrix conflict-free
  static constexpr int THREADS = 32 * MT;
  static constexpr int TILE = LP * RS;  // elements
  static constexpr size_t kFwdSmem = 3 * (size_t)TILE * 2 + 2 * LP * 4;
  static constexpr size_t kBwdSmem = 5 * (size_t)TILE * 2 + 8 * LP * 4;
};

// rows [0, L) of one head of a [T][ld] bf16 matrix -> tile[LP][RS]; rows [L, LP) are zero
template <int DH, int MT>
__device__ __forceinline__ void stage_tile_async(uint16_t* tile, const uint16_t* __restrict__ src, long long ld, int L, int tid) {
  using Cf = RegCfg<DH, MT>;
  constexpr int CPR = DH / 8;
  for (int e = tid; e < Cf::LP * CPR; e += Cf::THREADS) {
    const int i = e / CPR, c = e - i * CPR;
    uint16_t* dst = tile + i * Cf::RS + c * 8;
    if (i < L) rcp16(rsaddr(dst), src + (long long)i * ld + c * 8);
    else *reinterpret_cast<uint4*>(dst) = make_uint4(0u, 0u, 0u, 0u);
  }
}

// D[nt][*] += A_rows(16 x DH, tile rows a_row0..) . B(all LP rows)^T : the "row block x all rows" L x L product
template <int DH, int MT>
__device__ __forceinline__ void block_nt(float (&d)[2 * MT][4], const uint16_t* A, int a_row0, const uint16_t* B, int lane, int L) {
  using Cf = RegCfg<DH, MT>;
#pragma unroll
  for (int ks = 0; ks < Cf::KS; ++ks) {
    uint32_t af[4];
    rldsm4(rsaddr(A + (a_row0 + (lane & 15)) * Cf::RS + ks * 16 + (lane >> 4) * 8), af);
#pragma unroll
    for (int np = 0; np < MT; ++np) {
      uint32_t bf[4];
      rldsm4(rsaddr(B + (np * 16 + (lane & 7) + ((lane >> 4) << 3)) * Cf::RS + ks * 16 + ((lane >> 3) & 1) * 8), bf);
      rmma(d[2 * np], af, bf[0], bf[1]);
      if ((2 * np + 1) * 8 < L) rmma(d[2 * np + 1], af, bf[2], bf[3]);   // a column tile beyond L stays zero
    }
  }
}

// O[on][*] += P(16 x LP, accumulator fragments, bf16-rounded) . X(LP x DH, staged tile)
template <int DH, int MT>
__device__ __forceinline__ void block_pv(float (&o)[DH / 8][4], const float (&pm)[2 * MT][4], const uint16_t* X, int lane) {
  using Cf = RegCfg<DH, MT>;
#pragma unroll
  for (int kk = 0; kk < MT; ++kk) {
    uint32_t af[4];
    af[0] = pack_bf16x2(pm[2 * kk][0], pm[2 * kk][1]);
    af[1] = pack_bf16x2(pm[2 * kk][2], pm[2 * kk][3]);
    af[2] = pack_bf16x2(pm[2 * kk + 1][0], pm[2 * kk + 1][1]);
    af[3] = pack_bf16x2(pm[2 * kk + 1][2], pm[2 * kk + 1][3]);
#pragma unroll
    for (int op = 0; op < Cf::ON / 2; ++op) {
      uint32_t bf[4];
      rldsm4t(rsaddr(X + (kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * Cf::RS + op * 16 + (lane >> 4) * 8), bf);
      rmma(o[2 * op], af, bf[0], bf[1]);
      rmma(o[2 * op + 1], af, bf[2], bf[3]);
    }
  }
}

template <int ON>
__device__ __forceinline__ void zero_acc(float (&o)[ON][4]) {
#pragma unroll
  for (int n = 0; n < ON; ++n) { o[n][0] = 0.f; o[n][1] = 0.f; o[n][2] = 0.f; o[n][3] = 0.f; }
}

// rows r0 / r1 of an output block, scaled, as bf16 pairs
template <int ON>
__device__ __forceinline__ void store_rows(uint16_t* dst0, uint16_t* dst1, bool ok0, bool ok1, const float (&o)[ON][4], float scale, int t) {
#pragma unroll
  for (int n = 0; n < ON; ++n) {
    const int col = n * 8 + 2 * t;
    if (ok0) *reinterpret_cast<uint32_t*>(dst0 + col) = pack_bf16x2(o[n][0] * scale, o[n][1] * scale);
    if (ok1) *reinterpret_cast<uint32_t*>(dst1 + col) = pack_bf16x2(o[n][2] * scale, o[n][3] * scale);
  }
}

// 1 / |c_i| and the additive key mask of every row; padded rows: norm 1, mask -inf (their keys drop out of every softmax)
template <int DH, int MT>
__device__ __forceinline__ void norms_and_mask(const uint16_t* sC, const float* __restrict__ mask_row, int L, int tid, float* nrm, float* madd) {
  using Cf = RegCfg<DH, MT>;
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

// ---------------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------------
template <int DH, int MT>
__global__ void __launch_bounds__(32 * MT) attn_reg_fwd_kernel(const pmgt_attn_args a) {
  using Cf = RegCfg<DH, MT>;
  extern __shared__ __align__(16) unsigned char smem[];
  uint16_t* sK = reinterpret_cast<uint16_t*>(smem);
  uint16_t* sV = sK + Cf::TILE;
  uint16_t* sC = sV + Cf::TILE;
  float* nrm = reinterpret_cast<float*>(sC + Cf::TILE);
  float* madd = nrm + Cf::LP;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  const int L = a.L, H = a.H, heads = a.heads;
  const int nt_live = (L + 7) >> 3;   // 8-wide column tiles that hold at least one real position (L = 33: 5 of 6)
  const long long item = blockIdx.x;
  const long long row = item / heads;
  const int head = (int)(item - row * heads);
  const long long ld = 4ll * H;
  const uint16_t* src = a.qkvc + row * L * ld + head * DH;

  stage_tile_async<DH, MT>(sK, src + H, ld, L, tid);
  stage_tile_async<DH, MT>(sV, src + 2 * H, ld, L, tid);
  stage_tile_async<DH, MT>(sC, src + 3 * H, ld, L, tid);
  asm volatile("cp.async.commit_group;" ::: "memory");
  // Q fragments of this warp's 16 rows straight from global memory (each element is used by this warp only)
  const int i0 = warp * 16 + g, i1 = i0 + 8;
  uint32_t qf[Cf::KS][4];
#pragma unroll
  for (int ks = 0; ks < Cf::KS; ++ks) {
    const int col = ks * 16 + 2 * t;
    qf[ks][0] = i0 < L ? __ldg(reinterpret_cast<const uint32_t*>(src + (long long)i0 * ld + col)) : 0u;
    qf[ks][1] = i1 < L ? __ldg(reinterpret_cast<const uint32_t*>(src + (long long)i1 * ld + col)) : 0u;
    qf[ks][2] = i0 < L ? __ldg(reinterpret_cast<const uint32_t*>(src + (long long)i0 * ld + col + 8)) : 0u;
    qf[ks][3] = i1 < L ? __ldg(reinterpret_cast<const uint32_t*>(src + (long long)i1 * ld + col + 8)) : 0u;
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  norms_and_mask<DH, MT>(sC, a.mask + row * L, L, tid, nrm, madd);
  __syncthreads();

  float s1[Cf::NT][4], s2[Cf::NT][4];
  zero_acc<Cf::NT>(s1);
  zero_acc<Cf::NT>(s2);
  block_nt<DH, MT>(s1, sC, warp * 16, sC, lane, L);
#pragma unroll
  for (int ks = 0; ks < Cf::KS; ++ks) {
#pragma unroll
    for (int np = 0; np < MT; ++np) {
      uint32_t bf[4];
      rldsm4(rsaddr(sK + (np * 16 + (lane & 7) + ((lane >> 4) << 3)) * Cf::RS + ks * 16 + ((lane >> 3) & 1) * 8), bf);
      rmma(s2[2 * np], qf[ks], bf[0], bf[1]);
      if ((2 * np + 1) * 8 < L) rmma(s2[2 * np + 1], qf[ks], bf[2], bf[3]);
    }
  }
  // scores -> probabilities, in place
  const float inv_sqrt_dh = rsqrtf((float)DH);
  const float rn0 = nrm[i0], rn1 = nrm[i1];
  float m1a = -INFINITY, m1b = -INFINITY, m2a = -INFINITY, m2b = -INFINITY;
#pragma unroll
  for (int nt = 0; nt < Cf::NT; ++nt) if (nt < nt_live) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int j = nt * 8 + 2 * t + (e & 1);
      const int i = e < 2 ? i0 : i1;
      const float cs = s1[nt][e] * (e < 2 ? rn0 : rn1) * nrm[j];
      s1[nt][e] = 1.f - cs + (i == j ? 1.f : 0.f) + madd[j];
      s2[nt][e] = s2[nt][e] * inv_sqrt_dh + madd[j];
    }
    m1a = fmaxf(m1a, fmaxf(s1[nt][0], s1[nt][1]));
    m1b = fmaxf(m1b, fmaxf(s1[nt][2], s1[nt][3]));
    m2a = fmaxf(m2a, fmaxf(s2[nt][0], s2[nt][1]));
    m2b = fmaxf(m2b, fmaxf(s2[nt][2], s2[nt][3]));
  }
  m1a = quad_max(m1a); m1b = quad_max(m1b); m2a = quad_max(m2a); m2b = quad_max(m2b);
  float z1a = 0.f, z1b = 0.f, z2a = 0.f, z2b = 0.f;
#pragma unroll
  for (int nt = 0; nt < Cf::NT; ++nt) if (nt < nt_live) {
    s1[nt][0] = __expf(s1[nt][0] - m1a); s1[nt][1] = __expf(s1[nt][1] - m1a);
    s1[nt][2] = __expf(s1[nt][2] - m1b); s1[nt][3] = __expf(s1[nt][3] - m1b);
    s2[nt][0] = __expf(s2[nt][0] - m2a); s2[nt][1] = __expf(s2[nt][1] - m2a);
    s2[nt][2] = __expf(s2[nt][2] - m2b); s2[nt][3] = __expf(s2[nt][3] - m2b);
    z1a += s1[nt][0] + s1[nt][1]; z1b += s1[nt][2] + s1[nt][3];
    z2a += s2[nt][0] + s2[nt][1]; z2b += s2[nt][2] + s2[nt][3];
  }
  z1a = 1.f / quad_sum(z1a); z1b = 1.f / quad_sum(z1b); z2a = 1.f / quad_sum(z2a); z2b = 1.f / quad_sum(z2b);
  // A = beta drop(P1) + (1 - beta) drop(P2), kept in s1
  const DropKey dk = drop_key(a.dropout_seed, a.dropout_site, a.dropout_p, item);
  const float beta = a.beta;
  const uint32_t dbase0 = (uint32_t)(i0 * L), dbase1 = (uint32_t)(i1 * L);
#pragma unroll
  for (int nt = 0; nt < Cf::NT; ++nt) if (nt < nt_live) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int j = nt * 8 + 2 * t + (e & 1);
      float f1, f2;
      drop_factors(dk, (e < 2 ? dbase0 : dbase1) + (uint32_t)j, f1, f2);
      const float p1 = s1[nt][e] * (e < 2 ? z1a : z1b) * f1;
      const float p2 = s2[nt][e] * (e < 2 ? z2a : z2b) * f2;
      s1[nt][e] = beta * p1 + (1.f - beta) * p2;
    }
  }
  float o[Cf::ON][4];
  zero_acc<Cf::ON>(o);
  block_pv<DH, MT>(o, s1, sV, lane);
  uint16_t* dst = a.ctx + row * L * (long long)H + head * DH;
  store_rows<Cf::ON>(dst + (long long)i0 * H, dst + (long long)i1 * H, i0 < L, i1 < L, o, 1.f, t);
}

// ---------------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------------
template <int DH, int MT>
__global__ void __launch_bounds__(32 * MT, 65536 / (32 * MT * PMGT_REG_BWD_REGS)) attn_reg_bwd_kernel(const pmgt_attn_args a) {
  using Cf = RegCfg<DH, MT>;
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
  const int nt_live = (L + 7) >> 3;   // 8-wide column tiles that hold at least one real position (L = 33: 5 of 6)
  const long long item = blockIdx.x;
  const long long row = item / heads;
  const int head = (int)(item - row * heads);
  const long long ld = 4ll * H;
  const uint16_t* src = a.qkvc + row * L * ld + head * DH;

  stage_tile_async<DH, MT>(sQ, src, ld, L, tid);
  stage_tile_async<DH, MT>(sK, src + H, ld, L, tid);
  stage_tile_async<DH, MT>(sV, src + 2 * H, ld, L, tid);
  stage_tile_async<DH, MT>(sC, src + 3 * H, ld, L, tid);
  stage_tile_async<DH, MT>(sO, a.dctx + row * L * (long long)H + head * DH, (long long)H, L, tid);
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  norms_and_mask<DH, MT>(sC, a.mask + row * L, L, tid, nrm, madd);
  __syncthreads();

  const int r0 = warp * 16 + g, r1 = r0 + 8;  // this thread's two rows: queries in phase A, keys in phase B
  const float inv_sqrt_dh = rsqrtf((float)DH);
  const float rn0 = nrm[r0], rn1 = nrm[r1];
  const DropKey dk = drop_key(a.dropout_seed, a.dropout_site, a.dropout_p, item);
  const float beta = a.beta;
  uint16_t* dst = a.dqkvc + row * L * ld + head * DH;
  uint16_t* d0 = dst + (long long)r0 * ld;
  uint16_t* d1 = dst + (long long)r1 * ld;
  const bool ok0 = r0 < L, ok1 = r1 < L;
  const uint32_t dbase0 = (uint32_t)(r0 * L), dbase1 = (uint32_t)(r1 * L);  // phase A: + j; phase B: i L + r

  float gram[Cf::NT][4];  // raw C C^T block of these rows: symmetric, so it serves both orientations
  zero_acc<Cf::NT>(gram);
  block_nt<DH, MT>(gram, sC, warp * 16, sC, lane, L);
  float accC[Cf::ON][4];  // sum_j [dS1_ij + dS1_ji] / (n_i n_j) C_j for rows r0 / r1
  zero_acc<Cf::ON>(accC);
  float rc0 = 0.f, rc1 = 0.f;  // sum_j (dS1_ij + dS1_ji) cos_ij

  // ===================== phase A: rows = queries =====================
  {
    float p1[Cf::NT][4], p2[Cf::NT][4], dA[Cf::NT][4];
    zero_acc<Cf::NT>(p1);
    zero_acc<Cf::NT>(p2);
    zero_acc<Cf::NT>(dA);
    block_nt<DH, MT>(p2, sQ, warp * 16, sK, lane, L);
    block_nt<DH, MT>(dA, sO, warp * 16, sV, lane, L);
    float m1a = -INFINITY, m1b = -INFINITY, m2a = -INFINITY, m2b = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < Cf::NT; ++nt) if (nt < nt_live) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int j = nt * 8 + 2 * t + (e & 1);
        const int i = e < 2 ? r0 : r1;
        const float cs = gram[nt][e] * (e < 2 ? rn0 : rn1) * nrm[j];
        p1[nt][e] = 1.f - cs + (i == j ? 1.f : 0.f) + madd[j];
        p2[nt][e] = p2[nt][e] * inv_sqrt_dh + madd[j];
      }
      m1a = fmaxf(m1a, fmaxf(p1[nt][0], p1[nt][1]));
      m1b = fmaxf(m1b, fmaxf(p1[nt][2], p1[nt][3]));
      m2a = fmaxf(m2a, fmaxf(p2[nt][0], p2[nt][1]));
      m2b = fmaxf(m2b, fmaxf(p2[nt][2], p2[nt][3]));
    }
    m1a = quad_max(m1a); m1b = quad_max(m1b); m2a = quad_max(m2a); m2b = quad_max(m2b);
    float z1a = 0.f, z1b = 0.f, z2a = 0.f, z2b = 0.f;
#pragma unroll
    for (int nt = 0; nt < Cf::NT; ++nt) if (nt < nt_live) {
      p1[nt][0] = __expf(p1[nt][0] - m1a); p1[nt][1] = __expf(p1[nt][1] - m1a);
      p1[nt][2] = __expf(p1[nt][2] - m1b); p1[nt][3] = __expf(p1[nt][3] - m1b);
      p2[nt][0] = __expf(p2[nt][0] - m2a); p2[nt][1] = __expf(p2[nt][1] - m2a);
      p2[nt][2] = __expf(p2[nt][2] - m2b); p2[nt][3] = __expf(p2[nt][3] - m2b);
      z1a += p1[nt][0] + p1[nt][1]; z1b += p1[nt][2] + p1[nt][3];
      z2a += p2[nt][0] + p2[nt][1]; z2b += p2[nt][2] + p2[nt][3];
    }
    z1a = 1.f / quad_sum(z1a); z1b = 1.f / quad_sum(z1b); z2a = 1.f / quad_sum(z2a); z2b = 1.f / quad_sum(z2b);
    // g1 = beta dA drop1, g2 = (1 - beta) dA drop2 (into dA / p-independent temporaries), row dots r = sum_j g P
    float r1a = 0.f, r1b = 0.f, r2a = 0.f, r2b = 0.f;
    float g2[Cf::NT][4];
    zero_acc<Cf::NT>(g2);
#pragma unroll
    for (int nt = 0; nt < Cf::NT; ++nt) if (nt < nt_live) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int j = nt * 8 + 2 * t + (e & 1);
        float f1, f2;
        drop_factors(dk, (e < 2 ? dbase0 : dbase1) + (uint32_t)j, f1, f2);
        p1[nt][e] *= (e < 2 ? z1a : z1b);
        p2[nt][e] *= (e < 2 ? z2a : z2b);
        const float ga = beta * dA[nt][e] * f1;
        const float gb = (1.f - beta) * dA[nt][e] * f2;
        dA[nt][e] = ga;
        g2[nt][e] = gb;
        if (e < 2) { r1a = fmaf(ga, p1[nt][e], r1a); r2a = fmaf(gb, p2[nt][e], r2a); }
        else { r1b = fmaf(ga, p1[nt][e], r1b); r2b = fmaf(gb, p2[nt][e], r2b); }
      }
    }
    r1a = quad_sum(r1a); r1b = quad_sum(r1b); r2a = quad_sum(r2a); r2b = quad_sum(r2b);
    if (t == 0) {
      st_m1[r0] = m1a; st_z1[r0] = z1a; st_m2[r0] = m2a; st_z2[r0] = z2a; st_r1[r0] = r1a; st_r2[r0] = r2a;
      st_m1[r1] = m1b; st_z1[r1] = z1b; st_m2[r1] = m2b; st_z2[r1] = z2b; st_r1[r1] = r1b; st_r2[r1] = r2b;
    }
    // dS2 -> g2 (in place), dS1 / (n_i n_j) -> dA (in place); cosine row dot
#pragma unroll
    for (int nt = 0; nt < Cf::NT; ++nt) if (nt < nt_live) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int j = nt * 8 + 2 * t + (e & 1);
        const float rn = e < 2 ? rn0 : rn1;
        const float ds1 = p1[nt][e] * (dA[nt][e] - (e < 2 ? r1a : r1b));
        g2[nt][e] = p2[nt][e] * (g2[nt][e] - (e < 2 ? r2a : r2b));
        const float rnj = nrm[j];
        const float cs = gram[nt][e] * rn * rnj;
        if (e < 2) rc0 = fmaf(ds1, cs, rc0); else rc1 = fmaf(ds1, cs, rc1);
        dA[nt][e] = ds1 * rn * rnj;
      }
    }
    float o[Cf::ON][4];
    zero_acc<Cf::ON>(o);
    block_pv<DH, MT>(o, g2, sK, lane);                       // dQ_i = sum_j dS2_ij K_j / sqrt(dh)
    store_rows<Cf::ON>(d0, d1, ok0, ok1, o, inv_sqrt_dh, t);
    block_pv<DH, MT>(accC, dA, sC, lane);                    // row half of dC
  }
  __syncthreads();  // every query row's statistics are in shared memory

  // ===================== phase B: rows = keys, columns = queries =====================
  {
    float p2[Cf::NT][4], dA[Cf::NT][4];
    zero_acc<Cf::NT>(p2);
    zero_acc<Cf::NT>(dA);
    block_nt<DH, MT>(p2, sK, warp * 16, sQ, lane, L);   // K_j . Q_i
    block_nt<DH, MT>(dA, sV, warp * 16, sO, lane, L);   // V_j . dO_i
    const float ma0 = madd[r0], ma1 = madd[r1];
    float am[Cf::NT][4];  // A_ij (with dropout) for dV
    zero_acc<Cf::NT>(am);
#pragma unroll
    for (int nt = 0; nt < Cf::NT; ++nt) if (nt < nt_live) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int i = nt * 8 + 2 * t + (e & 1);   // query (column)
        const int j = e < 2 ? r0 : r1;            // key (row)
        const float rnj = e < 2 ? rn0 : rn1;
        const float mj = e < 2 ? ma0 : ma1;
        const bool live = i < L;                  // padded queries contribute nothing
        const float rni = nrm[i];
        const float cs = gram[nt][e] * rnj * rni;
        const float q1 = live ? __expf(1.f - cs + (i == j ? 1.f : 0.f) + mj - st_m1[i]) * st_z1[i] : 0.f;
        const float q2 = live ? __expf(p2[nt][e] * inv_sqrt_dh + mj - st_m2[i]) * st_z2[i] : 0.f;
        float f1, f2;
        drop_factors(dk, (uint32_t)(i * L + j), f1, f2);
        am[nt][e] = beta * q1 * f1 + (1.f - beta) * q2 * f2;
        const float ga = beta * dA[nt][e] * f1;
        const float gb = (1.f - beta) * dA[nt][e] * f2;
        const float ds1 = live ? q1 * (ga - st_r1[i]) : 0.f;
        p2[nt][e] = live ? q2 * (gb - st_r2[i]) : 0.f;   // dS2_ij
        if (e < 2) rc0 = fmaf(ds1, cs, rc0); else rc1 = fmaf(ds1, cs, rc1);
        dA[nt][e] = ds1 * rnj * rni;
      }
    }
    float o[Cf::ON][4];
    zero_acc<Cf::ON>(o);
    block_pv<DH, MT>(o, am, sO, lane);                        // dV_j = sum_i A_ij dO_i
    store_rows<Cf::ON>(d0 + 2 * H, d1 + 2 * H, ok0, ok1, o, 1.f, t);
    zero_acc<Cf::ON>(o);
    block_pv<DH, MT>(o, p2, sQ, lane);                        // dK_j = sum_i dS2_ij Q_i / sqrt(dh)
    store_rows<Cf::ON>(d0 + H, d1 + H, ok0, ok1, o, inv_sqrt_dh, t);
    block_pv<DH, MT>(accC, dA, sC, lane);                     // column half of dC
  }
  // dC_r = -accC_r + (rc_r / n_r^2) C_r
  rc0 = quad_sum(rc0) * rn0 * rn0;
  rc1 = quad_sum(rc1) * rn1 * rn1;
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

template <int DH, int MT, bool BWD>
int launch_reg(const pmgt_attn_args* a, cudaStream_t st) {
  using Cf = RegCfg<DH, MT>;
  const size_t smem = BWD ? Cf::kBwdSmem : Cf::kFwdSmem;
  static unsigned long long configured = 0;
  if (first_use_on_device(configured)) {
    if (BWD) PMGT_CHECK_CUDA(cudaFuncSetAttribute(attn_reg_bwd_kernel<DH, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    else PMGT_CHECK_CUDA(cudaFuncSetAttribute(attn_reg_fwd_kernel<DH, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  const long long items = a->rows * a->heads;  // <= 2^31 - 1 (attn_family in attention.cu)
  if (BWD) attn_reg_bwd_kernel<DH, MT><<<(unsigned)items, 32 * MT, smem, st>>>(*a);
  else attn_reg_fwd_kernel<DH, MT><<<(unsigned)items, 32 * MT, smem, st>>>(*a);
  PMGT_LAUNCH_CHECK();
  return PMGT_OK;
}

// 8 < L <= 64, head size 32 / 64 / 128
template <bool BWD>
int dispatch_reg(const pmgt_attn_args* a, cudaStream_t st) {
  const int dh = a->H / a->heads;
  const int mt = a->L > 8 && a->L <= 64 ? (a->L + 15) / 16 : 0;
#define PMGT_REG_CASE(D, M) if (dh == D && mt == M) return launch_reg<D, M, BWD>(a, st)
  PMGT_REG_CASE(32, 1); PMGT_REG_CASE(32, 2); PMGT_REG_CASE(32, 3); PMGT_REG_CASE(32, 4);
  PMGT_REG_CASE(64, 1); PMGT_REG_CASE(64, 2); PMGT_REG_CASE(64, 3); PMGT_REG_CASE(64, 4);
  PMGT_REG_CASE(128, 1); PMGT_REG_CASE(128, 2); PMGT_REG_CASE(128, 3); PMGT_REG_CASE(128, 4);
#undef PMGT_REG_CASE
  set_error("attn_reg: no kernel for L=%d, head size %d", a->L, dh);
  return PMGT_ERR_INVALID;
}

}  // namespace

int attn_reg_fwd(const pmgt_attn_args* a, cudaStream_t st) { return dispatch_reg<false>(a, st); }
int attn_reg_bwd(const pmgt_attn_args* a, cudaStream_t st) { return dispatch_reg<true>(a, st); }

}  // namespace pmgt
