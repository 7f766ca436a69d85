// K3 attention core for short sequences (L <= 8), warp-level tensor-core tiles.
//
// The dual-softmax attention of PMGTSelfAttention (pmgt/pmgt/modeling_pmgt.py:435-526; formulas in
// attention.cu) on a 6-token sequence is a handful of [6 x dh] x [dh x 6] and [6 x 6] x [6 x dh] products per
// (sequence, head): far below the 64/128-row tiles of tcgen05, and as scalar FMAs they were instruction-bound
// (the scalar kernel this one replaced reached 27 % of the HBM roofline in backward).  Here one warp owns one
// (sequence, head):
//   * the Q/K/V/C (and dctx) rows are staged with 16-byte cp.async into a padded shared-memory tile,
//     double-buffered so the next item streams in while the current one is computed;
//   * every product runs as m16n8k16 bf16 MMAs with fp32 accumulation (ldmatrix / ldmatrix.trans operand
//     fragments straight from the staged rows; rows 6..7 of each tile are zero padding);
//   * the L x L score algebra (dual softmax, dropout, softmax / cosine backward) lives in the accumulator
//     fragment layout: lane (g, t) holds row g, columns 2t and 2t+1, so row reductions are two quad shuffles
//     and an accumulator fragment IS the A operand of the next product (movmatrix for the transposed ones).
// The kernel is then bound by HBM: forward 10*H, backward 18*H bytes per token.
#include "common.cuh"

namespace pmgt {

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit_group() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ uint32_t movmatrix_trans(uint32_t a) {
  uint32_t d;
  asm volatile("movmatrix.sync.aligned.m8n8.trans.b16 %0, %1;" : "=r"(d) : "r"(a));
  return d;
}
// D(16x8, fp32) += A(16x16, bf16, row) * B(16x8, bf16, col); rows 8..15 of A are zero (a1 = a3 = 0)
__device__ __forceinline__ void mma16816(float (&d)[4], uint32_t a0, uint32_t a2, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a0), "r"(0u), "r"(a2), "r"(0u), "r"(b0), "r"(b1));
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

// keep bits of elements base_idx .. base_idx + LL - 1 (LL <= 64) for dropout sites `site` (k1) and `site + 1`
// (k2): lanes 0..NB-1 run the Philox blocks (8 elements each) of the first site, lanes 16..16+NB-1 those of the
// second, then an OR reduction within each half-warp (stream of common.cuh).
template <int LL>
__device__ __forceinline__ void warp_dropout_bits2(uint64_t seed, uint32_t site, uint64_t base_idx, float p, int lane,
                                                   uint64_t& k1, uint64_t& k2) {
  constexpr int NB = (LL + 7) / 8 + 1;
  static_assert(NB <= 16, "one Philox block per lane of a half-warp");
  const uint64_t b0 = base_idx & ~(uint64_t)7;
  const int hl = lane & 15;
  uint64_t bits = 0;
  const uint64_t i8 = b0 + 8ull * hl;
  if (hl < NB && i8 < base_idx + LL) {
    const uint64_t m = dropout_keep8(seed, site + (uint32_t)(lane >> 4), i8, p);
    const long long sh = (long long)i8 - (long long)base_idx;
    bits = sh >= 0 ? (m << sh) : (m >> (-sh));
  }
  uint32_t lo = (uint32_t)bits, hi = (uint32_t)(bits >> 32);
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) {
    lo |= __shfl_xor_sync(0xffffffffu, lo, o);
    hi |= __shfl_xor_sync(0xffffffffu, hi, o);
  }
  const uint32_t lo2 = __shfl_xor_sync(0xffffffffu, lo, 16), hi2 = __shfl_xor_sync(0xffffffffu, hi, 16);
  uint64_t mine = ((uint64_t)hi << 32) | lo, other = ((uint64_t)hi2 << 32) | lo2;
  if (LL < 64) {
    mine &= (1ull << (LL & 63)) - 1ull;
    other &= (1ull << (LL & 63)) - 1ull;
  }
  k1 = (lane < 16) ? mine : other;
  k2 = (lane < 16) ? other : mine;
}

template <int L, int DH>
struct AttnTile {
  static constexpr int kStride = DH * 2 + 16;       // bytes per staged row (padding keeps ldmatrix conflict-free)
  static constexpr int kTensor = L * kStride;       // L data rows; fragment rows L..7 read the warp's zero row
};

// shared-memory address of fragment row r (< 8) of a staged tensor: rows >= L alias the zero row
template <int L, int DH>
__device__ __forceinline__ uint32_t frag_row(const unsigned char* t, const unsigned char* zero, int r) {
  return smem_addr(r < L ? t + r * AttnTile<L, DH>::kStride : zero);
}

// stage rows [0, L) of NT tensors of one item: tensor t < 4 comes from qkvc (+ t*H), tensor 4 from dctx
template <int L, int DH, int NT>
__device__ __forceinline__ void stage_item(unsigned char* buf, const uint16_t* __restrict__ qkvc_item, long long ld,
                                           int H, const uint16_t* __restrict__ dctx_item, int lane) {
  constexpr int CPR = DH / 8;  // 16-byte chunks per row
  constexpr int TOTAL = NT * L * CPR;
  using Tile = AttnTile<L, DH>;
  if constexpr (CPR == 16 && L % 2 == 0) {
    // one warp iteration = two consecutive rows of one tensor: (tensor, row pair) are compile-time constants
    const int sub = lane >> 4, ch = lane & 15;
    const uint16_t* s_q = qkvc_item + (long long)sub * ld + ch * 8;
    const uint16_t* s_d = (NT > 4) ? dctx_item + (long long)sub * H + ch * 8 : nullptr;
    const uint32_t d0 = smem_addr(buf) + sub * Tile::kStride + ch * 16;
#pragma unroll
    for (int k = 0; k < NT * L / 2; ++k) {
      const int t = (2 * k) / L, row = (2 * k) % L;
      const uint16_t* src = (t < 4) ? s_q + (long long)row * ld + t * H : s_d + (long long)row * H;
      cp_async16(d0 + t * Tile::kTensor + row * Tile::kStride, src);
    }
  } else {
#pragma unroll
    for (int c = lane; c < TOTAL; c += 32) {
      const int t = c / (L * CPR), rem = c - t * (L * CPR);
      const int row = rem / CPR, ch = rem - row * CPR;
      const uint16_t* src = (t < 4) ? qkvc_item + (long long)row * ld + t * H + ch * 8
                                    : dctx_item + (long long)row * H + ch * 8;
      cp_async16(smem_addr(buf + t * Tile::kTensor + row * Tile::kStride + ch * 16), src);
    }
  }
}

// NP independent products acc[p] (16x8) = X_p rows (as A, K = DH) * Y_p rows (as B: n = row of Y), all staged
// K-major.  Each product is split over even / odd k-steps, so 2 * NP accumulator chains are in flight.
template <int L, int DH, int NP>
__device__ __forceinline__ void mma_rows_rows(float (&acc)[NP][4], const unsigned char* const (&x)[NP],
                                              const unsigned char* const (&y)[NP], const unsigned char* zero, int lane) {
  // ldmatrix.x4: matrix m = lane / 8 -> (k-step = m >> 1, k-half = m & 1), row = lane % 8
  const int m = lane >> 3, r = lane & 7;
  const uint32_t koff = (uint32_t)(((m >> 1) * 16 + (m & 1) * 8) * 2);
  uint32_t xo[NP], yo[NP];
  float odd[NP][4];
#pragma unroll
  for (int p = 0; p < NP; ++p) {
    xo[p] = frag_row<L, DH>(x[p], zero, r) + koff;
    yo[p] = frag_row<L, DH>(y[p], zero, r) + koff;
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[p][i] = odd[p][i] = 0.f;
  }
#pragma unroll
  for (int ks = 0; ks < DH / 16; ks += 2) {
    uint32_t a[NP][4], b[NP][4];
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      ldsm_x4(xo[p] + ks * 32, a[p]);
      ldsm_x4(yo[p] + ks * 32, b[p]);
    }
#pragma unroll
    for (int p = 0; p < NP; ++p) mma16816(acc[p], a[p][0], a[p][1], b[p][0], b[p][1]);
#pragma unroll
    for (int p = 0; p < NP; ++p) mma16816(odd[p], a[p][2], a[p][3], b[p][2], b[p][3]);
  }
#pragma unroll
  for (int p = 0; p < NP; ++p)
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[p][i] += odd[p][i];
}

// out[i][dim] = sum_j M[i][j] * Y[j][dim]: afrag = bf16x2 fragment of M (rows i, k = j), Y staged rows j.
// The bf16 result rows i < L are collected in the shared-memory tile `stg` (a staged tensor that is no longer
// needed) and leave as full 16-byte chunks: 4-byte fragment stores would half-fill every 32-byte sector.
template <int L, int DH>
__device__ __forceinline__ void mma_small_rows_store(uint32_t afrag, const unsigned char* y, unsigned char* stg,
                                                     uint16_t* __restrict__ dst, long long ldo, const unsigned char* zero,
                                                     int lane) {
  using Tile = AttnTile<L, DH>;
  const int g = lane >> 2, tg = lane & 3;
  // ldmatrix.x4.trans: matrix m = lane / 8 -> n-tile (8 dims), row = lane % 8 = j
  const bool data_row = (lane & 7) < L;
  const uint32_t yo = frag_row<L, DH>(y, zero, lane & 7) + (data_row ? (lane >> 3) * 16 : 0);
  unsigned char* srow = stg + (g < L ? g : 0) * Tile::kStride + tg * 4;
#pragma unroll
  for (int nt = 0; nt < DH / 8; nt += 4) {
    uint32_t b[4];
    ldsm_x4_trans(yo + (data_row ? nt * 16 : 0), b);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      mma16816(acc, afrag, 0u, b[q], 0u);
      if (g < L) *reinterpret_cast<uint32_t*>(srow + (nt + q) * 16) = pack_bf16x2(acc[0], acc[1]);
    }
  }
  __syncwarp();
  constexpr int CPR = DH / 8;
#pragma unroll
  for (int c = lane; c < L * CPR; c += 32) {
    const int row = c / CPR, ch = c - row * CPR;
    *reinterpret_cast<uint4*>(dst + (long long)row * ldo + ch * 8) =
        *reinterpret_cast<const uint4*>(stg + row * Tile::kStride + ch * 16);
  }
  __syncwarp();
}

// Dual softmax in fragment layout.  In: s2 = raw Q K^T, gm = C C^T (this lane: row g, columns 2t, 2t+1).
// mask_lane: lane j < L holds the 0/1 attention mask of key j.  Out: p1, p2 probabilities, cs = cosine entries, nr / nc0 / nc1 = norms of row g and of the two columns.
template <int L, int DH>
__device__ __forceinline__ void frag_dual_softmax(const float (&s2)[4], const float (&gm)[4], float mask_lane,
                                                  int lane, float (&p1)[2], float (&p2)[2], float (&cs)[2], float& nr,
                                                  float (&nc)[2]) {
  const int g = lane >> 2, tg = lane & 3;
  const int j0 = 2 * tg, j1 = 2 * tg + 1;
  const bool vi = g < L, v0 = j0 < L, v1 = j1 < L;
  // diagonal of the Gram matrix: G[i][i] sits in lane 4i + i/2, slot i & 1
  const float mine = (g & 1) ? gm[1] : gm[0];
  const float dr = __shfl_sync(0xffffffffu, mine, 4 * g + (g >> 1));
  const float d0 = __shfl_sync(0xffffffffu, mine, 9 * tg);      // 4*(2t) + t
  const float d1 = __shfl_sync(0xffffffffu, mine, 9 * tg + 4);  // 4*(2t+1) + t
  nr = vi ? sqrtf(dr) : 1.f;
  nc[0] = v0 ? sqrtf(d0) : 1.f;
  nc[1] = v1 ? sqrtf(d1) : 1.f;
  const float mk0 = __shfl_sync(0xffffffffu, mask_lane, j0), mk1 = __shfl_sync(0xffffffffu, mask_lane, j1);
  const float m0 = v0 ? (1.f - mk0) * -10000.f : 0.f;
  const float m1 = v1 ? (1.f - mk1) * -10000.f : 0.f;
  const float inv_sqrt_dh = rsqrtf((float)DH);
  cs[0] = (vi && v0) ? gm[0] / (nr * nc[0]) : 0.f;
  cs[1] = (vi && v1) ? gm[1] / (nr * nc[1]) : 0.f;
  float a0 = v0 ? 1.f - cs[0] + (g == j0 ? 1.f : 0.f) + m0 : -INFINITY;
  float a1 = v1 ? 1.f - cs[1] + (g == j1 ? 1.f : 0.f) + m1 : -INFINITY;
  float b0 = v0 ? s2[0] * inv_sqrt_dh + m0 : -INFINITY;
  float b1 = v1 ? s2[1] * inv_sqrt_dh + m1 : -INFINITY;
  if (!vi) { a0 = a1 = b0 = b1 = v0 ? 0.f : -INFINITY; }
  const float ma = quad_max(fmaxf(a0, a1)), mb = quad_max(fmaxf(b0, b1));
  a0 = __expf(a0 - ma); a1 = __expf(a1 - ma);
  b0 = __expf(b0 - mb); b1 = __expf(b1 - mb);
  const float ra = 1.f / quad_sum(a0 + a1), rb = 1.f / quad_sum(b0 + b1);
  p1[0] = vi ? a0 * ra : 0.f; p1[1] = vi ? a1 * ra : 0.f;
  p2[0] = vi ? b0 * rb : 0.f; p2[1] = vi ? b1 * rb : 0.f;
}

template <int L, int DH, int NT>
struct AttnRing {
  static constexpr int kItem = NT * AttnTile<L, DH>::kTensor;
  static constexpr int kZero = AttnTile<L, DH>::kStride;
  // the kernel is issue-latency-bound per warp (ncu: stall_wait / short_scoreboard), so shared memory buys
  // WARPS first: double buffering only, and as many warps as fit (<= 16, a multiple of 4)
  static constexpr int kStages = 2;
  static constexpr int kPerWarp = kStages * kItem + kZero;
  static constexpr int kFit = (227 * 1024) / kPerWarp;
  static constexpr int kWarps = kFit >= 16 ? 16 : (kFit >= 12 ? 12 : (kFit >= 8 ? 8 : 4));
};

template <int L, int DH>
__global__ void __launch_bounds__(AttnRing<L, DH, 4>::kWarps * 32, 1) attn_mma_fwd_kernel(const pmgt_attn_args a, const int reverse) {
  using Tile = AttnTile<L, DH>;
  using Ring = AttnRing<L, DH, 4>;
  constexpr int S = Ring::kStages;
  extern __shared__ __align__(128) unsigned char smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  unsigned char* wbuf = smem + (size_t)wib * Ring::kPerWarp;
  unsigned char* zero = wbuf + S * Ring::kItem;
  pdl_launch_dependents();
  for (int i = lane * 16; i < Ring::kZero; i += 32 * 16) *reinterpret_cast<uint4*>(zero + i) = make_uint4(0, 0, 0, 0);
  __syncwarp();
  pdl_wait();
  const int H = a.H, heads = a.heads;
  const long long ld = 4ll * H;
  const long long n_items = a.rows * heads;
  const long long w0 = (long long)blockIdx.x * (blockDim.x >> 5) + wib;
  const long long nw = (long long)gridDim.x * (blockDim.x >> 5);
  const int g = lane >> 2, tg = lane & 3;
  const float ks = a.dropout_p > 0.f ? 1.f / (1.f - a.dropout_p) : 1.f;

  static_assert(S == 2, "the mask prefetch below runs exactly one item ahead");
  float mask_next = 1.f;
  auto stage = [&](long long litem, int slot) {
    if (litem < n_items) {
      const long long item = reverse ? n_items - 1 - litem : litem;  // alternating traversal order (next_tile_order)
      const long long row = heads == 1 ? item : item / heads;
      const int head = (int)(item - row * heads);
      stage_item<L, DH, 4>(wbuf + slot * Ring::kItem, a.qkvc + row * L * ld + head * DH, ld, H, nullptr, lane);
      mask_next = lane < L ? a.mask[row * L + lane] : 1.f;
    }
    cp_async_commit_group();
  };
#pragma unroll
  for (int s = 0; s < S - 1; ++s) stage(w0 + (long long)s * nw, s);
  int cur = 0;
  for (long long litem = w0; litem < n_items; litem += nw) {
    const long long item = reverse ? n_items - 1 - litem : litem;
    const float mask_cur = mask_next;
    // slot (cur + S - 1) % S was consumed in the previous iteration (a __syncwarp separates it from this refill)
    stage(litem + (long long)(S - 1) * nw, (cur + S - 1) % S);
    cp_async_wait_group<S - 1>();
    __syncwarp();
    unsigned char* buf = wbuf + cur * Ring::kItem;
    unsigned char* q = buf;
    const unsigned char *k = buf + Tile::kTensor, *v = buf + 2 * Tile::kTensor, *c = buf + 3 * Tile::kTensor;
    float acc[2][4];
    {
      const unsigned char* const xs[2] = {q, c};
      const unsigned char* const ys[2] = {k, c};
      mma_rows_rows<L, DH, 2>(acc, xs, ys, zero, lane);
    }
    const long long row = heads == 1 ? item : item / heads;
    const int head = (int)(item - row * heads);
    float p1[2], p2[2], cs[2], nr, nc[2];
    frag_dual_softmax<L, DH>(acc[0], acc[1], mask_cur, lane, p1, p2, cs, nr, nc);
    if (a.dropout_p > 0.f) {
      const uint64_t base = (uint64_t)item * (L * L);
      uint64_t k1, k2;
      warp_dropout_bits2<L * L>(a.dropout_seed, a.dropout_site, base, a.dropout_p, lane, k1, k2);
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const int e = (g * L + 2 * tg + s) & 63;
        p1[s] = (k1 >> e) & 1ull ? p1[s] * ks : 0.f;
        p2[s] = (k2 >> e) & 1ull ? p2[s] * ks : 0.f;
      }
    }
    const bool in = g < L;
    const float w0v = (in && 2 * tg < L) ? a.beta * p1[0] + (1.f - a.beta) * p2[0] : 0.f;
    const float w1v = (in && 2 * tg + 1 < L) ? a.beta * p1[1] + (1.f - a.beta) * p2[1] : 0.f;
    // the Q tile is dead after the score products: it collects the context rows
    mma_small_rows_store<L, DH>(pack_bf16x2(w0v, w1v), v, q, a.ctx + row * L * (long long)H + head * DH, H, zero, lane);
    cur = (cur + 1) % S;
  }
  cp_async_wait_group<0>();
}

template <int L, int DH>
__global__ void __launch_bounds__(AttnRing<L, DH, 5>::kWarps * 32, 1) attn_mma_bwd_kernel(const pmgt_attn_args a, const int reverse) {
  using Tile = AttnTile<L, DH>;
  using Ring = AttnRing<L, DH, 5>;
  constexpr int S = Ring::kStages;
  extern __shared__ __align__(128) unsigned char smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  unsigned char* wbuf = smem + (size_t)wib * Ring::kPerWarp;
  unsigned char* zero = wbuf + S * Ring::kItem;
  pdl_launch_dependents();
  for (int i = lane * 16; i < Ring::kZero; i += 32 * 16) *reinterpret_cast<uint4*>(zero + i) = make_uint4(0, 0, 0, 0);
  __syncwarp();
  pdl_wait();
  const int H = a.H, heads = a.heads;
  const long long ld = 4ll * H;
  const long long n_items = a.rows * heads;
  const long long w0 = (long long)blockIdx.x * (blockDim.x >> 5) + wib;
  const long long nw = (long long)gridDim.x * (blockDim.x >> 5);
  const int g = lane >> 2, tg = lane & 3;
  const int j0 = 2 * tg, j1 = 2 * tg + 1;
  const float ks = a.dropout_p > 0.f ? 1.f / (1.f - a.dropout_p) : 1.f;
  const float inv_sqrt_dh = rsqrtf((float)DH);

  static_assert(S == 2, "the mask prefetch below runs exactly one item ahead");
  float mask_next = 1.f;
  auto stage = [&](long long litem, int slot) {
    if (litem < n_items) {
      const long long item = reverse ? n_items - 1 - litem : litem;  // alternating traversal order (next_tile_order)
      const long long row = heads == 1 ? item : item / heads;
      const int head = (int)(item - row * heads);
      stage_item<L, DH, 5>(wbuf + slot * Ring::kItem, a.qkvc + row * L * ld + head * DH, ld, H,
                           a.dctx + row * L * (long long)H + head * DH, lane);
      mask_next = lane < L ? a.mask[row * L + lane] : 1.f;
    }
    cp_async_commit_group();
  };
#pragma unroll
  for (int s = 0; s < S - 1; ++s) stage(w0 + (long long)s * nw, s);
  int cur = 0;
  for (long long litem = w0; litem < n_items; litem += nw) {
    const long long item = reverse ? n_items - 1 - litem : litem;
    const float mask_cur = mask_next;
    stage(litem + (long long)(S - 1) * nw, (cur + S - 1) % S);
    cp_async_wait_group<S - 1>();
    __syncwarp();
    unsigned char* buf = wbuf + cur * Ring::kItem;
    unsigned char* v = buf + 2 * Tile::kTensor;  // dead after the dA product: collects the output rows
    const unsigned char *q = buf, *k = buf + Tile::kTensor, *c = buf + 3 * Tile::kTensor, *dO = buf + 4 * Tile::kTensor;
    float acc[3][4];  // s2 = Q K^T, gm = C C^T, dA_ij = dctx_i . v_j
    {
      const unsigned char* const xs[3] = {q, c, dO};
      const unsigned char* const ys[3] = {k, c, v};
      mma_rows_rows<L, DH, 3>(acc, xs, ys, zero, lane);
    }
    const float(&dA)[4] = acc[2];
    const long long row = heads == 1 ? item : item / heads;
    const int head = (int)(item - row * heads);
    float p1[2], p2[2], cs[2], nr, nc[2];
    frag_dual_softmax<L, DH>(acc[0], acc[1], mask_cur, lane, p1, p2, cs, nr, nc);
    uint64_t k1 = ~0ull, k2 = ~0ull;
    if (a.dropout_p > 0.f) {
      const uint64_t base = (uint64_t)item * (L * L);
      warp_dropout_bits2<L * L>(a.dropout_seed, a.dropout_site, base, a.dropout_p, lane, k1, k2);
    }
    const bool vi = g < L;
    const bool vj[2] = {j0 < L, j1 < L};
    float A[2], g1[2], g2[2];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      const int e = (g * L + 2 * tg + s) & 63;
      const bool ok = vi && vj[s];
      const float f1 = ((k1 >> e) & 1ull) ? ks : 0.f, f2 = ((k2 >> e) & 1ull) ? ks : 0.f;
      A[s] = ok ? a.beta * p1[s] * f1 + (1.f - a.beta) * p2[s] * f2 : 0.f;
      g1[s] = ok ? a.beta * dA[s] * f1 : 0.f;
      g2[s] = ok ? (1.f - a.beta) * dA[s] * f2 : 0.f;
    }
    uint16_t* dst = a.dqkvc + row * L * ld + head * DH;
    // dV = A^T dctx
    mma_small_rows_store<L, DH>(movmatrix_trans(pack_bf16x2(A[0], A[1])), dO, v, dst + 2 * H, ld, zero, lane);
    // softmax backward of both branches
    const float r1 = quad_sum(g1[0] * p1[0] + g1[1] * p1[1]);
    const float r2 = quad_sum(g2[0] * p2[0] + g2[1] * p2[1]);
    float dS1[2], dS2[2];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      dS1[s] = p1[s] * (g1[s] - r1);
      dS2[s] = p2[s] * (g2[s] - r2) * inv_sqrt_dh;
    }
    const uint32_t f_dS2 = pack_bf16x2(dS2[0], dS2[1]);
    mma_small_rows_store<L, DH>(f_dS2, k, v, dst, ld, zero, lane);                        // dQ = dS2 K
    mma_small_rows_store<L, DH>(movmatrix_trans(f_dS2), q, v, dst + H, ld, zero, lane);   // dK = dS2^T Q
    // cosine branch: D = -(dS1 + dS1^T); E_ij = D_ij / (n_i n_j) - [i == j] (sum_j' D_ij' cos_ij') / n_i^2
    float E[2];
    {
      // dS1^T: element (j, i) sits in lane 4j + i/2, slot i & 1
      const float t00 = __shfl_sync(0xffffffffu, dS1[0], (4 * j0 + (g >> 1)) & 31);
      const float t01 = __shfl_sync(0xffffffffu, dS1[1], (4 * j0 + (g >> 1)) & 31);
      const float t10 = __shfl_sync(0xffffffffu, dS1[0], (4 * j1 + (g >> 1)) & 31);
      const float t11 = __shfl_sync(0xffffffffu, dS1[1], (4 * j1 + (g >> 1)) & 31);
      const float tr0 = (g & 1) ? t01 : t00, tr1 = (g & 1) ? t11 : t10;
      const float D0 = (vi && vj[0]) ? -(dS1[0] + tr0) : 0.f;
      const float D1 = (vi && vj[1]) ? -(dS1[1] + tr1) : 0.f;
      const float sdc = quad_sum(D0 * cs[0] + D1 * cs[1]);
      E[0] = D0 / (nr * nc[0]) - (g == j0 ? sdc / (nr * nr) : 0.f);
      E[1] = D1 / (nr * nc[1]) - (g == j1 ? sdc / (nr * nr) : 0.f);
      if (!vi) E[0] = E[1] = 0.f;
      if (!vj[0]) E[0] = 0.f;
      if (!vj[1]) E[1] = 0.f;
    }
    mma_small_rows_store<L, DH>(pack_bf16x2(E[0], E[1]), c, v, dst + 3 * H, ld, zero, lane);  // dC = E C
    cur = (cur + 1) % S;
  }
  cp_async_wait_group<0>();
}

template <int L, int DH, bool BWD>
static int launch_mma(const pmgt_attn_args* a, cudaStream_t st) {
  constexpr int kWarps = AttnRing<L, DH, (BWD ? 5 : 4)>::kWarps;
  constexpr int smem = kWarps * AttnRing<L, DH, (BWD ? 5 : 4)>::kPerWarp;
  static_assert(smem <= 227 * 1024, "shared memory budget");
  static unsigned long long configured = 0;
  if (first_use_on_device(configured)) {
    if (BWD) PMGT_CHECK_CUDA(cudaFuncSetAttribute(attn_mma_bwd_kernel<L, DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    else PMGT_CHECK_CUDA(cudaFuncSetAttribute(attn_mma_fwd_kernel<L, DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  }
  const long long items = a->rows * a->heads;
  long long ctas = (items + kWarps - 1) / kWarps;
  const long long per_sm = (227 * 1024) / smem;
  const long long cap = (long long)num_sms() * (per_sm < 1 ? 1 : per_sm);
  if (ctas > cap) ctas = cap;
  if (BWD)
    PMGT_CHECK_CUDA(launch_kernel(true, attn_mma_bwd_kernel<L, DH>, dim3((unsigned)ctas), dim3(kWarps * 32), smem, st, *a, next_tile_order()));
  else
    PMGT_CHECK_CUDA(launch_kernel(true, attn_mma_fwd_kernel<L, DH>, dim3((unsigned)ctas), dim3(kWarps * 32), smem, st, *a, next_tile_order()));
  return PMGT_OK;
}

// L = 6, head size 32 / 64 / 128 (attn_family in attention.cu)
template <bool BWD>
static int dispatch_mma(const pmgt_attn_args* a, cudaStream_t st) {
  const int dh = a->H / a->heads;
  if (a->L == 6 && dh == 128) return launch_mma<6, 128, BWD>(a, st);
  if (a->L == 6 && dh == 64) return launch_mma<6, 64, BWD>(a, st);
  if (a->L == 6 && dh == 32) return launch_mma<6, 32, BWD>(a, st);
  set_error("attn_mma: no kernel for L=%d, head size %d", a->L, dh);
  return PMGT_ERR_INVALID;
}

int attn_mma_fwd(const pmgt_attn_args* a, cudaStream_t st) { return dispatch_mma<false>(a, st); }
int attn_mma_bwd(const pmgt_attn_args* a, cudaStream_t st) { return dispatch_mma<true>(a, st); }

}  // namespace pmgt
