// K3 attention core for medium sequence lengths (8 < L <= 64, head size a multiple of 16): BASELINE config 5
// (32 sampled neighbours, L = 33, 12 heads of 64).  Same algebra as attention.cu (dual-softmax "diversity promoting"
// attention of pmgt/pmgt/modeling_pmgt.py:435-526, formulas there); what changes is where the FLOPs run.  The generic
// kernel forms every L x L x dh product with scalar FMAs fed by two shared-memory loads each (~4 TFLOP/s, 58 % of a
// wide-encoder step); here a CTA of four warps owns one (sequence, head) at a time (six CTAs fit per SM), and
//   * Q K^T, C C^T and dO V^T are m16n8k16 bf16 MMAs whose operands come straight from the staged row tiles with
//     ldmatrix (rows padded to a multiple of 16 and kept zero, row pitch dh + 8 so that rows stay 16-byte aligned and
//     ldmatrix is bank-conflict free), results land in the fp32 L x L score matrices in shared memory;
//   * the products with an L x L left operand (A V, A^T dO, dS K, dS^T Q, D' C) build their A fragments from those
//     fp32 matrices on the fly -- transposed or rescaled as needed, zero beyond L -- and fetch the right operand with
//     ldmatrix.trans; accumulators go to global memory as bf16 pairs.
// Softmax, dropout and the softmax / cosine backward stay scalar per row: they are O(L^2) per item, not O(L^2 dh).
#include "common.cuh"

namespace pmgt {

namespace {

constexpr int kMidPad = 8;
constexpr int kMidThreads = 128;  // four warps share one (sequence, head): tile pairs / output blocks are dealt to the warps
constexpr int kMidWarps = kMidThreads / 32;

struct MidLayout {
  int rs, Lp;
  size_t tile_bytes, mat_bytes, vec_bytes, per_warp_fwd, per_warp_bwd;
};

MidLayout mid_layout(int L, int dh) {
  MidLayout s;
  s.rs = dh + kMidPad;
  s.Lp = (L + 15) & ~15;
  s.tile_bytes = (size_t)s.Lp * s.rs * 2;
  s.mat_bytes = ((size_t)L * L * 4 + 15) & ~(size_t)15;
  s.vec_bytes = ((size_t)L * 4 + 15) & ~(size_t)15;
  s.per_warp_fwd = 4 * s.tile_bytes + 2 * s.mat_bytes + 2 * s.vec_bytes;
  s.per_warp_bwd = 5 * s.tile_bytes + 5 * s.mat_bytes + 3 * s.vec_bytes;
  return s;
}

__device__ __forceinline__ uint32_t saddr(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void ldsm4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void ldsm4t(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
// D(16x8, fp32) += A(16x16, bf16, row-major fragment) * B(16x8, bf16, column fragment)
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// rows [0, L) of one head of a [T][ld] bf16 matrix -> tile[L][rs] (16-byte copies); pad rows are never written
__device__ __forceinline__ void stage_tile(uint16_t* tile, int rs, const uint16_t* __restrict__ src, long long ld, int L,
                                           int dh, int tid) {
  const int cpr = dh >> 3;
  for (int e = tid; e < L * cpr; e += kMidThreads) {
    const int i = e / cpr, c = e - i * cpr;
    *reinterpret_cast<uint4*>(tile + i * rs + c * 8) = __ldg(reinterpret_cast<const uint4*>(src + (long long)i * ld + c * 8));
  }
}

// out[i][j] = scale * sum_k A[i][k] B[j][k]   (i, j < L; k < dh), both operands staged row tiles
__device__ __forceinline__ void mma_nt(float* __restrict__ out, int L, int Lp, const uint16_t* A, const uint16_t* B, int rs,
                                       int dh, float scale, int lane, int warp) {
  const int g = lane >> 2, t = lane & 3;
  const int nt = Lp >> 4;
  for (int pr = warp; pr < nt * nt; pr += kMidWarps) {
    const int m0 = (pr / nt) * 16, n0 = (pr % nt) * 16;
    {
      float c0[4] = {0.f, 0.f, 0.f, 0.f}, c1[4] = {0.f, 0.f, 0.f, 0.f};
      for (int k0 = 0; k0 < dh; k0 += 16) {
        uint32_t a[4], b[4];
        ldsm4(saddr(A + (m0 + (lane & 15)) * rs + k0 + (lane >> 4) * 8), a);
        ldsm4(saddr(B + (n0 + (lane & 7) + ((lane >> 4) << 3)) * rs + k0 + ((lane >> 3) & 1) * 8), b);
        mma_bf16(c0, a, b[0], b[1]);
        mma_bf16(c1, a, b[2], b[3]);
      }
      const int r0 = m0 + g, r1 = r0 + 8, j0 = n0 + 2 * t, j1 = j0 + 8;
      if (r0 < L) {
        if (j0 < L) out[r0 * L + j0] = c0[0] * scale;
        if (j0 + 1 < L) out[r0 * L + j0 + 1] = c0[1] * scale;
        if (j1 < L) out[r0 * L + j1] = c1[0] * scale;
        if (j1 + 1 < L) out[r0 * L + j1 + 1] = c1[1] * scale;
      }
      if (r1 < L) {
        if (j0 < L) out[r1 * L + j0] = c0[2] * scale;
        if (j0 + 1 < L) out[r1 * L + j0 + 1] = c0[3] * scale;
        if (j1 < L) out[r1 * L + j1] = c1[2] * scale;
        if (j1 + 1 < L) out[r1 * L + j1 + 1] = c1[3] * scale;
      }
    }
  }
}

// dst[i][n] = scale * sum_k af(i, k) X[k][n] - rowsub(i) * S[i][n]   (i < L, k < L, n < dh)
// af: element of the L x L left operand (already zero-safe for i, k < L); X: staged tile whose pad rows are zero.
// The optional subtraction (S != nullptr) is the "- cos_ij c_i / n_i^2" term of the cosine backward.
template <class AF>
__device__ __forceinline__ void mma_sn(uint16_t* __restrict__ dst, long long ld_dst, int L, int Lp, int dh, const uint16_t* X,
                                       int rs, AF af, float scale, const uint16_t* S, const float* rowsub, int lane, int warp) {
  const int g = lane >> 2, t = lane & 3;
  const int nkt = Lp >> 4;  // <= 4
  const int nnb = dh >> 4;
  for (int u = warp; u < nkt * nnb; u += kMidWarps) {
    const int m0 = (u / nnb) * 16, n0 = (u % nnb) * 16;
    const int r0 = m0 + g, r1 = r0 + 8;
    uint32_t afr[4][4];
#pragma unroll
    for (int kt = 0; kt < 4; ++kt) {
      if (kt < nkt) {
        const int c = kt * 16 + 2 * t;
        auto el = [&](int i, int k) -> float { return (i < L && k < L) ? af(i, k) : 0.f; };
        afr[kt][0] = pack_bf16x2(el(r0, c), el(r0, c + 1));
        afr[kt][1] = pack_bf16x2(el(r1, c), el(r1, c + 1));
        afr[kt][2] = pack_bf16x2(el(r0, c + 8), el(r0, c + 9));
        afr[kt][3] = pack_bf16x2(el(r1, c + 8), el(r1, c + 9));
      }
    }
    const float s0 = (S && r0 < L) ? rowsub[r0] : 0.f, s1 = (S && r1 < L) ? rowsub[r1] : 0.f;
    {
      float c0[4] = {0.f, 0.f, 0.f, 0.f}, c1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int kt = 0; kt < 4; ++kt) {
        if (kt < nkt) {
          uint32_t b[4];
          ldsm4t(saddr(X + (kt * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * rs + n0 + (lane >> 4) * 8), b);
          mma_bf16(c0, afr[kt], b[0], b[1]);
          mma_bf16(c1, afr[kt], b[2], b[3]);
        }
      }
      const int na = n0 + 2 * t, nb = na + 8;
      if (r0 < L) {
        float x0 = c0[0] * scale, x1 = c0[1] * scale, y0 = c1[0] * scale, y1 = c1[1] * scale;
        if (S) {
          float p, q;
          unpack_bf16x2(*reinterpret_cast<const uint32_t*>(S + r0 * rs + na), p, q);
          x0 -= s0 * p; x1 -= s0 * q;
          unpack_bf16x2(*reinterpret_cast<const uint32_t*>(S + r0 * rs + nb), p, q);
          y0 -= s0 * p; y1 -= s0 * q;
        }
        *reinterpret_cast<uint32_t*>(dst + (long long)r0 * ld_dst + na) = pack_bf16x2(x0, x1);
        *reinterpret_cast<uint32_t*>(dst + (long long)r0 * ld_dst + nb) = pack_bf16x2(y0, y1);
      }
      if (r1 < L) {
        float x0 = c0[2] * scale, x1 = c0[3] * scale, y0 = c1[2] * scale, y1 = c1[3] * scale;
        if (S) {
          float p, q;
          unpack_bf16x2(*reinterpret_cast<const uint32_t*>(S + r1 * rs + na), p, q);
          x0 -= s1 * p; x1 -= s1 * q;
          unpack_bf16x2(*reinterpret_cast<const uint32_t*>(S + r1 * rs + nb), p, q);
          y0 -= s1 * p; y1 -= s1 * q;
        }
        *reinterpret_cast<uint32_t*>(dst + (long long)r1 * ld_dst + na) = pack_bf16x2(x0, x1);
        *reinterpret_cast<uint32_t*>(dst + (long long)r1 * ld_dst + nb) = pack_bf16x2(y0, y1);
      }
    }
  }
}

// raw scores + both softmaxes: P1 -> s1, P2 -> s2, |c_i| -> nrm, key mask add -> madd, cosine matrix -> cosm (if any)
__device__ __forceinline__ void scores_and_probs_mid(const uint16_t* q, const uint16_t* k, const uint16_t* c, int rs, int Lp,
                                                     const float* __restrict__ mask_row, int L, int dh, int tid, float* s1,
                                                     float* s2, float* nrm, float* madd, float* cosm) {
  const int lane = tid & 31, warp = tid >> 5;
  mma_nt(s1, L, Lp, c, c, rs, dh, 1.f, lane, warp);
  mma_nt(s2, L, Lp, q, k, rs, dh, rsqrtf((float)dh), lane, warp);
  __syncthreads();
  for (int i = tid; i < L; i += kMidThreads) {
    nrm[i] = sqrtf(s1[i * L + i]);
    madd[i] = (1.f - mask_row[i]) * -10000.f;
  }
  __syncthreads();
  for (int e = tid; e < L * L; e += kMidThreads) {
    const int i = e / L, j = e - i * L;
    const float cs = s1[e] / (nrm[i] * nrm[j]);
    if (cosm) cosm[e] = cs;
    s1[e] = 1.f - cs + (i == j ? 1.f : 0.f) + madd[j];
    s2[e] += madd[j];
  }
  __syncthreads();
  // the two softmaxes run side by side: threads [0, 64) take P1's rows, [64, 128) P2's
  if (tid < 64) {
    for (int i = tid; i < L; i += 64) {
      float* r = s1 + i * L;
      float mx = -INFINITY;
      for (int j = 0; j < L; ++j) mx = fmaxf(mx, r[j]);
      float sum = 0.f;
      for (int j = 0; j < L; ++j) { const float e = __expf(r[j] - mx); r[j] = e; sum += e; }
      const float inv = 1.f / sum;
      for (int j = 0; j < L; ++j) r[j] *= inv;
    }
  } else {
    for (int i = tid - 64; i < L; i += 64) {
      float* r = s2 + i * L;
      float mx = -INFINITY;
      for (int j = 0; j < L; ++j) mx = fmaxf(mx, r[j]);
      float sum = 0.f;
      for (int j = 0; j < L; ++j) { const float e = __expf(r[j] - mx); r[j] = e; sum += e; }
      const float inv = 1.f / sum;
      for (int j = 0; j < L; ++j) r[j] *= inv;
    }
  }
  __syncthreads();
}

__device__ __forceinline__ void zero_pad_rows(uint16_t* tile, int rs, int L, int Lp, int tid) {
  for (int e = tid; e < (Lp - L) * rs; e += kMidThreads) tile[L * rs + e] = 0;
}

__global__ void __launch_bounds__(kMidThreads) attn_mid_fwd_kernel(const pmgt_attn_args a, MidLayout lay) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int L = a.L, H = a.H, heads = a.heads, dh = H / heads, rs = lay.rs, Lp = lay.Lp;
  unsigned char* base = smem;
  uint16_t* q = reinterpret_cast<uint16_t*>(base);
  uint16_t* k = reinterpret_cast<uint16_t*>(base + lay.tile_bytes);
  uint16_t* v = reinterpret_cast<uint16_t*>(base + 2 * lay.tile_bytes);
  uint16_t* c = reinterpret_cast<uint16_t*>(base + 3 * lay.tile_bytes);
  float* s1 = reinterpret_cast<float*>(base + 4 * lay.tile_bytes);
  float* s2 = reinterpret_cast<float*>(base + 4 * lay.tile_bytes + lay.mat_bytes);
  float* nrm = reinterpret_cast<float*>(base + 4 * lay.tile_bytes + 2 * lay.mat_bytes);
  float* madd = reinterpret_cast<float*>(base + 4 * lay.tile_bytes + 2 * lay.mat_bytes + lay.vec_bytes);
  zero_pad_rows(q, rs, L, Lp, tid);
  zero_pad_rows(k, rs, L, Lp, tid);
  zero_pad_rows(v, rs, L, Lp, tid);
  zero_pad_rows(c, rs, L, Lp, tid);
  const long long n_items = a.rows * heads;
  const long long ld = 4ll * H;
  const float keep_scale = a.dropout_p > 0.f ? 1.f / (1.f - a.dropout_p) : 1.f;
  for (long long item = blockIdx.x; item < n_items; item += gridDim.x) {
    const long long row = item / heads;
    const int head = (int)(item - row * heads);
    const uint16_t* src = a.qkvc + row * L * ld + head * dh;
    __syncthreads();  // the previous item's last readers are done with the tiles
    stage_tile(q, rs, src, ld, L, dh, tid);
    stage_tile(k, rs, src + H, ld, L, dh, tid);
    stage_tile(v, rs, src + 2 * H, ld, L, dh, tid);
    stage_tile(c, rs, src + 3 * H, ld, L, dh, tid);
    __syncthreads();
    scores_and_probs_mid(q, k, c, rs, Lp, a.mask + row * L, L, dh, tid, s1, s2, nrm, madd, nullptr);
    // A = beta * drop(P1) + (1 - beta) * drop(P2), stored in s1
    for (int e = tid; e < L * L; e += kMidThreads) {
      float p1 = s1[e], p2 = s2[e];
      if (a.dropout_p > 0.f) {
        const uint64_t idx = (uint64_t)item * L * L + e;
        p1 = dropout_keep(a.dropout_seed, a.dropout_site, idx, a.dropout_p) ? p1 * keep_scale : 0.f;
        p2 = dropout_keep(a.dropout_seed, a.dropout_site + 1, idx, a.dropout_p) ? p2 * keep_scale : 0.f;
      }
      s1[e] = a.beta * p1 + (1.f - a.beta) * p2;
    }
    __syncthreads();
    uint16_t* dst = a.ctx + row * L * (long long)H + head * dh;
    mma_sn(dst, (long long)H, L, Lp, dh, v, rs, [&](int i, int j) { return s1[i * L + j]; }, 1.f, nullptr, nullptr, lane, warp);
  }
}

__global__ void __launch_bounds__(kMidThreads) attn_mid_bwd_kernel(const pmgt_attn_args a, MidLayout lay) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int L = a.L, H = a.H, heads = a.heads, dh = H / heads, rs = lay.rs, Lp = lay.Lp;
  unsigned char* base = smem;
  uint16_t* q = reinterpret_cast<uint16_t*>(base);
  uint16_t* k = reinterpret_cast<uint16_t*>(base + lay.tile_bytes);
  uint16_t* v = reinterpret_cast<uint16_t*>(base + 2 * lay.tile_bytes);
  uint16_t* c = reinterpret_cast<uint16_t*>(base + 3 * lay.tile_bytes);
  uint16_t* dc = reinterpret_cast<uint16_t*>(base + 4 * lay.tile_bytes);  // staged dctx
  unsigned char* mats = base + 5 * lay.tile_bytes;
  float* p1 = reinterpret_cast<float*>(mats);
  float* p2 = reinterpret_cast<float*>(mats + lay.mat_bytes);
  float* cosm = reinterpret_cast<float*>(mats + 2 * lay.mat_bytes);
  float* dA = reinterpret_cast<float*>(mats + 3 * lay.mat_bytes);   // dA, then dS2
  float* dS1 = reinterpret_cast<float*>(mats + 4 * lay.mat_bytes);  // A, then dS1
  float* nrm = reinterpret_cast<float*>(mats + 5 * lay.mat_bytes);
  float* madd = reinterpret_cast<float*>(mats + 5 * lay.mat_bytes + lay.vec_bytes);
  float* rsub = reinterpret_cast<float*>(mats + 5 * lay.mat_bytes + 2 * lay.vec_bytes);
  zero_pad_rows(q, rs, L, Lp, tid);
  zero_pad_rows(k, rs, L, Lp, tid);
  zero_pad_rows(v, rs, L, Lp, tid);
  zero_pad_rows(c, rs, L, Lp, tid);
  zero_pad_rows(dc, rs, L, Lp, tid);
  const long long n_items = a.rows * heads;
  const long long ld = 4ll * H;
  const float keep_scale = a.dropout_p > 0.f ? 1.f / (1.f - a.dropout_p) : 1.f;
  const float inv_sqrt_dh = rsqrtf((float)dh);
  for (long long item = blockIdx.x; item < n_items; item += gridDim.x) {
    const long long row = item / heads;
    const int head = (int)(item - row * heads);
    const uint16_t* src = a.qkvc + row * L * ld + head * dh;
    __syncthreads();  // the previous item's last readers are done with the tiles and matrices
    stage_tile(q, rs, src, ld, L, dh, tid);
    stage_tile(k, rs, src + H, ld, L, dh, tid);
    stage_tile(v, rs, src + 2 * H, ld, L, dh, tid);
    stage_tile(c, rs, src + 3 * H, ld, L, dh, tid);
    stage_tile(dc, rs, a.dctx + row * L * (long long)H + head * dh, H, L, dh, tid);
    __syncthreads();
    scores_and_probs_mid(q, k, c, rs, Lp, a.mask + row * L, L, dh, tid, p1, p2, nrm, madd, cosm);
    // dA_ij = dctx_i . v_j ;  A_ij (with dropout) kept in dS1 for the dV product
    mma_nt(dA, L, Lp, dc, v, rs, dh, 1.f, lane, warp);
    for (int e = tid; e < L * L; e += kMidThreads) {
      float d1 = p1[e], d2 = p2[e];
      if (a.dropout_p > 0.f) {
        const uint64_t idx = (uint64_t)item * L * L + e;
        d1 = dropout_keep(a.dropout_seed, a.dropout_site, idx, a.dropout_p) ? d1 * keep_scale : 0.f;
        d2 = dropout_keep(a.dropout_seed, a.dropout_site + 1, idx, a.dropout_p) ? d2 * keep_scale : 0.f;
      }
      dS1[e] = a.beta * d1 + (1.f - a.beta) * d2;
    }
    __syncthreads();
    uint16_t* dst = a.dqkvc + row * L * ld + head * dh;
    // dV_j = sum_i A_ij dctx_i
    mma_sn(dst + 2 * H, ld, L, Lp, dh, dc, rs, [&](int j, int i) { return dS1[i * L + j]; }, 1.f, nullptr, nullptr, lane, warp);
    __syncthreads();
    // softmax backward, one thread per row: dS = P * (dP - sum_j dP P)
    for (int i = tid; i < L; i += kMidThreads) {
      float r1 = 0.f, r2 = 0.f;
      for (int j = 0; j < L; ++j) {
        const int e = i * L + j;
        float g1 = a.beta * dA[e], g2 = (1.f - a.beta) * dA[e];
        if (a.dropout_p > 0.f) {
          const uint64_t idx = (uint64_t)item * L * L + e;
          g1 = dropout_keep(a.dropout_seed, a.dropout_site, idx, a.dropout_p) ? g1 * keep_scale : 0.f;
          g2 = dropout_keep(a.dropout_seed, a.dropout_site + 1, idx, a.dropout_p) ? g2 * keep_scale : 0.f;
        }
        r1 += g1 * p1[e];
        r2 += g2 * p2[e];
        dS1[e] = g1;
        dA[e] = g2;
      }
      for (int j = 0; j < L; ++j) {
        const int e = i * L + j;
        dS1[e] = p1[e] * (dS1[e] - r1);
        dA[e] = p2[e] * (dA[e] - r2);  // = dS2
      }
    }
    __syncthreads();
    // D = dcos + dcos^T with dcos = -dS1 -> p1 ; then pre-divided by n_i n_j, rsub_i = sum_j D_ij cos_ij / n_i^2
    for (int e = tid; e < L * L; e += kMidThreads) {
      const int i = e / L, j = e - i * L;
      p1[e] = -(dS1[e] + dS1[j * L + i]);
    }
    __syncthreads();
    for (int i = tid; i < L; i += kMidThreads) {
      float sacc = 0.f;
      const float ni = nrm[i];
      for (int j = 0; j < L; ++j) {
        const int e = i * L + j;
        sacc = fmaf(p1[e], cosm[e], sacc);
        p1[e] = p1[e] / (ni * nrm[j]);
      }
      rsub[i] = sacc / (ni * ni);
    }
    __syncthreads();
    mma_sn(dst, ld, L, Lp, dh, k, rs, [&](int i, int j) { return dA[i * L + j]; }, inv_sqrt_dh, nullptr, nullptr, lane, warp);      // dQ
    mma_sn(dst + H, ld, L, Lp, dh, q, rs, [&](int j, int i) { return dA[i * L + j]; }, inv_sqrt_dh, nullptr, nullptr, lane, warp);  // dK
    mma_sn(dst + 3 * H, ld, L, Lp, dh, c, rs, [&](int i, int j) { return p1[i * L + j]; }, 1.f, c, rsub, lane, warp);               // dC
  }
}

constexpr size_t kMidSmemMax = 220 * 1024;  // shared memory of one CTA (= one item in flight)

template <bool BWD>
int launch_mid(const pmgt_attn_args* a, cudaStream_t st) {
  const MidLayout lay = mid_layout(a->L, a->H / a->heads);
  const size_t smem = BWD ? lay.per_warp_bwd : lay.per_warp_fwd;
  static unsigned long long configured = 0;
  if (first_use_on_device(configured)) {
    if (BWD) PMGT_CHECK_CUDA(cudaFuncSetAttribute(attn_mid_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMidSmemMax));
    else PMGT_CHECK_CUDA(cudaFuncSetAttribute(attn_mid_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMidSmemMax));
  }
  int per_sm = (int)((224 * 1024) / (smem + 1024));  // CTAs that fit per SM
  if (per_sm > 16) per_sm = 16;
  if (per_sm < 1) per_sm = 1;
  const long long items = a->rows * a->heads;
  long long ctas = (long long)num_sms() * per_sm;
  if (ctas > items) ctas = items;
  if (BWD) attn_mid_bwd_kernel<<<(unsigned)ctas, kMidThreads, smem, st>>>(*a, lay);
  else attn_mid_fwd_kernel<<<(unsigned)ctas, kMidThreads, smem, st>>>(*a, lay);
  PMGT_LAUNCH_CHECK();
  return PMGT_OK;
}

}  // namespace

// Whether the mid kernels take (L, dh): the backward layout, the larger one, decides for both directions.
bool attn_mid_fits(int L, int dh) { return mid_layout(L, dh).per_warp_bwd <= kMidSmemMax; }

int attn_mid_fwd(const pmgt_attn_args* a, cudaStream_t st) { return launch_mid<false>(a, st); }
int attn_mid_bwd(const pmgt_attn_args* a, cudaStream_t st) { return launch_mid<true>(a, st); }

}  // namespace pmgt
