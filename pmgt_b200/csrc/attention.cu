// K3 attention core: the dual-softmax "diversity promoting" self-attention of
// PMGTSelfAttention.forward (pmgt/pmgt/modeling_pmgt.py:435-526), forward and
// backward, over sequences of L = max_ctx_neigh + 1 tokens (6 by default).
//
// pmgt_attn_core_fwd / _bwd validate the arguments and pick one kernel family
// from the shape alone (attn_family):
//   attn_mma  (attention_mma.cu)  L = 6,           head size 32 / 64 / 128
//   attn_reg  (attention_reg.cu)  8 < L <= 64,     head size 32 / 64 / 128
//   attn_mid  (attention_mid.cu)  8 < L <= 64,     other head sizes that are a multiple of 16, if its
//                                                  backward shared-memory layout fits
//   generic   (this file)         everything else, L <= 128, even head size
//
// The generic kernel: one warp owns one (sequence, head).  Q/K/V/C rows of that
// head are staged in a per-warp shared-memory tile (bf16, row stride dh+2 to stay
// bank-conflict free), the L x L score matrices live in shared memory as fp32,
// and the (i, j) pairs / the dh columns are spread over the 32 lanes.
//
//   G   = C C^T,  n_i = sqrt(G_ii)
//   S1  = 1 - G / (n n^T) + I + maskadd     P1 = dropout(softmax(S1))
//   S2  = Q K^T / sqrt(dh) + maskadd        P2 = dropout(softmax(S2))
//   ctx = (beta P1 + (1 - beta) P2) V
// maskadd_j = (1 - mask_j) * -10000  (transformers 4.11.2
// get_extended_attention_mask, key side only).  Like the reference there is no
// epsilon in G / (n n^T).
#include "common.cuh"

namespace pmgt {

constexpr int kAttnPad = 2;

struct AttnSmemLayout {
  int row_stride;      // bf16 elements per staged row
  size_t tile_bytes;   // one [L][row_stride] bf16 tile
  size_t mat_bytes;    // one L x L fp32 matrix
  size_t per_warp_fwd, per_warp_bwd;
};

static AttnSmemLayout attn_layout(int L, int dh) {
  AttnSmemLayout s;
  s.row_stride = dh + kAttnPad;
  s.tile_bytes = ((size_t)L * s.row_stride * 2 + 15) & ~(size_t)15;
  s.mat_bytes = ((size_t)L * L * 4 + 15) & ~(size_t)15;
  const size_t vec = ((size_t)L * 4 + 15) & ~(size_t)15;
  s.per_warp_fwd = 4 * s.tile_bytes + 2 * s.mat_bytes + 2 * vec;
  s.per_warp_bwd = 5 * s.tile_bytes + 5 * s.mat_bytes + 2 * vec;
  return s;
}

__device__ __forceinline__ void stage_rows(uint16_t* tile, int row_stride, const uint16_t* __restrict__ src,
                                           long long ld, int L, int dh, int lane) {
  const int words = dh >> 1;
  for (int e = lane; e < L * words; e += 32) {
    const int i = e / words, w = e - i * words;
    const uint32_t v = *reinterpret_cast<const uint32_t*>(src + (long long)i * ld + 2 * w);
    *reinterpret_cast<uint32_t*>(tile + i * row_stride + 2 * w) = v;
  }
}

__device__ __forceinline__ float dot_rows(const uint16_t* a, const uint16_t* b, int dh) {
  float s = 0.f;
  for (int w = 0; w < dh; w += 2) {
    float a0, a1, b0, b1;
    unpack_bf16x2(*reinterpret_cast<const uint32_t*>(a + w), a0, a1);
    unpack_bf16x2(*reinterpret_cast<const uint32_t*>(b + w), b0, b1);
    s = fmaf(a0, b0, s);
    s = fmaf(a1, b1, s);
  }
  return s;
}

// softmax of each row of S (in place); one lane per row
__device__ __forceinline__ void softmax_rows(float* S, int L, int lane) {
  for (int i = lane; i < L; i += 32) {
    float* r = S + i * L;
    float mx = -INFINITY;
    for (int j = 0; j < L; ++j) mx = fmaxf(mx, r[j]);
    float sum = 0.f;
    for (int j = 0; j < L; ++j) { const float e = __expf(r[j] - mx); r[j] = e; sum += e; }
    const float inv = 1.f / sum;
    for (int j = 0; j < L; ++j) r[j] *= inv;
  }
}

// raw scores + softmaxes; leaves P1 in s1, P2 in s2, norms in nrm, mask add in madd.
// If cosm != nullptr the cosine matrix G/(n n^T) is kept there (backward).
__device__ __forceinline__ void scores_and_probs(const uint16_t* q, const uint16_t* k, const uint16_t* c, int rs,
                                                 const float* __restrict__ mask_row, int L, int dh, int lane,
                                                 float* s1, float* s2, float* nrm, float* madd, float* cosm) {
  const float inv_sqrt_dh = rsqrtf((float)dh);
  for (int e = lane; e < L * L; e += 32) {
    const int i = e / L, j = e - i * L;
    s1[e] = dot_rows(c + i * rs, c + j * rs, dh);
    s2[e] = dot_rows(q + i * rs, k + j * rs, dh) * inv_sqrt_dh;
  }
  __syncwarp();
  for (int i = lane; i < L; i += 32) {
    nrm[i] = sqrtf(s1[i * L + i]);
    madd[i] = (1.f - mask_row[i]) * -10000.f;
  }
  __syncwarp();
  for (int e = lane; e < L * L; e += 32) {
    const int i = e / L, j = e - i * L;
    const float cs = s1[e] / (nrm[i] * nrm[j]);
    if (cosm) cosm[e] = cs;
    s1[e] = 1.f - cs + (i == j ? 1.f : 0.f) + madd[j];
    s2[e] += madd[j];
  }
  __syncwarp();
  softmax_rows(s1, L, lane);
  softmax_rows(s2, L, lane);
  __syncwarp();
}

__global__ void __launch_bounds__(128) attn_core_fwd_kernel(const pmgt_attn_args a, int warps_per_cta,
                                                            AttnSmemLayout lay) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  if (wib >= warps_per_cta) return;
  const int L = a.L, H = a.H, heads = a.heads, dh = H / heads, rs = lay.row_stride;
  unsigned char* base = smem + (size_t)wib * lay.per_warp_fwd;
  uint16_t* q = reinterpret_cast<uint16_t*>(base);
  uint16_t* k = reinterpret_cast<uint16_t*>(base + lay.tile_bytes);
  uint16_t* v = reinterpret_cast<uint16_t*>(base + 2 * lay.tile_bytes);
  uint16_t* c = reinterpret_cast<uint16_t*>(base + 3 * lay.tile_bytes);
  float* s1 = reinterpret_cast<float*>(base + 4 * lay.tile_bytes);
  float* s2 = reinterpret_cast<float*>(base + 4 * lay.tile_bytes + lay.mat_bytes);
  float* nrm = reinterpret_cast<float*>(base + 4 * lay.tile_bytes + 2 * lay.mat_bytes);
  float* madd = nrm + ((L + 3) & ~3);
  const long long n_items = a.rows * heads;
  const long long w0 = (long long)blockIdx.x * warps_per_cta + wib;
  const long long nw = (long long)gridDim.x * warps_per_cta;
  const long long ld = 4ll * H;
  const float keep_scale = a.dropout_p > 0.f ? 1.f / (1.f - a.dropout_p) : 1.f;
  for (long long item = w0; item < n_items; item += nw) {
    const long long row = item / heads;
    const int head = (int)(item - row * heads);
    const uint16_t* src = a.qkvc + row * L * ld + head * dh;
    stage_rows(q, rs, src, ld, L, dh, lane);
    stage_rows(k, rs, src + H, ld, L, dh, lane);
    stage_rows(v, rs, src + 2 * H, ld, L, dh, lane);
    stage_rows(c, rs, src + 3 * H, ld, L, dh, lane);
    __syncwarp();
    scores_and_probs(q, k, c, rs, a.mask + row * L, L, dh, lane, s1, s2, nrm, madd, nullptr);
    // A = beta * drop(P1) + (1 - beta) * drop(P2), stored in s1
    for (int e = lane; e < L * L; e += 32) {
      float p1 = s1[e], p2 = s2[e];
      if (a.dropout_p > 0.f) {
        const uint64_t idx = (uint64_t)item * L * L + e;
        p1 = dropout_keep(a.dropout_seed, a.dropout_site, idx, a.dropout_p) ? p1 * keep_scale : 0.f;
        p2 = dropout_keep(a.dropout_seed, a.dropout_site + 1, idx, a.dropout_p) ? p2 * keep_scale : 0.f;
      }
      s1[e] = a.beta * p1 + (1.f - a.beta) * p2;
    }
    __syncwarp();
    uint16_t* dst = a.ctx + row * L * (long long)H + head * dh;
    for (int w = 2 * lane; w < dh; w += 64) {
      for (int i = 0; i < L; ++i) {
        float acc0 = 0.f, acc1 = 0.f;
        for (int j = 0; j < L; ++j) {
          float v0, v1;
          unpack_bf16x2(*reinterpret_cast<const uint32_t*>(v + j * rs + w), v0, v1);
          const float pj = s1[i * L + j];
          acc0 = fmaf(pj, v0, acc0);
          acc1 = fmaf(pj, v1, acc1);
        }
        *reinterpret_cast<uint32_t*>(dst + (long long)i * H + w) = pack_bf16x2(acc0, acc1);
      }
    }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(128) attn_core_bwd_kernel(const pmgt_attn_args a, int warps_per_cta,
                                                            AttnSmemLayout lay) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  if (wib >= warps_per_cta) return;
  const int L = a.L, H = a.H, heads = a.heads, dh = H / heads, rs = lay.row_stride;
  unsigned char* base = smem + (size_t)wib * lay.per_warp_bwd;
  uint16_t* q = reinterpret_cast<uint16_t*>(base);
  uint16_t* k = reinterpret_cast<uint16_t*>(base + lay.tile_bytes);
  uint16_t* v = reinterpret_cast<uint16_t*>(base + 2 * lay.tile_bytes);
  uint16_t* c = reinterpret_cast<uint16_t*>(base + 3 * lay.tile_bytes);
  uint16_t* dc = reinterpret_cast<uint16_t*>(base + 4 * lay.tile_bytes);  // staged dctx
  float* p1 = reinterpret_cast<float*>(base + 5 * lay.tile_bytes);
  float* p2 = reinterpret_cast<float*>(base + 5 * lay.tile_bytes + lay.mat_bytes);
  float* cosm = reinterpret_cast<float*>(base + 5 * lay.tile_bytes + 2 * lay.mat_bytes);
  float* dA = reinterpret_cast<float*>(base + 5 * lay.tile_bytes + 3 * lay.mat_bytes);   // dA, then dS2
  float* dS1 = reinterpret_cast<float*>(base + 5 * lay.tile_bytes + 4 * lay.mat_bytes);  // A, then dS1
  float* nrm = reinterpret_cast<float*>(base + 5 * lay.tile_bytes + 5 * lay.mat_bytes);
  float* madd = nrm + ((L + 3) & ~3);
  const long long n_items = a.rows * heads;
  const long long w0 = (long long)blockIdx.x * warps_per_cta + wib;
  const long long nw = (long long)gridDim.x * warps_per_cta;
  const long long ld = 4ll * H;
  const float keep_scale = a.dropout_p > 0.f ? 1.f / (1.f - a.dropout_p) : 1.f;
  const float inv_sqrt_dh = rsqrtf((float)dh);
  for (long long item = w0; item < n_items; item += nw) {
    const long long row = item / heads;
    const int head = (int)(item - row * heads);
    const uint16_t* src = a.qkvc + row * L * ld + head * dh;
    stage_rows(q, rs, src, ld, L, dh, lane);
    stage_rows(k, rs, src + H, ld, L, dh, lane);
    stage_rows(v, rs, src + 2 * H, ld, L, dh, lane);
    stage_rows(c, rs, src + 3 * H, ld, L, dh, lane);
    stage_rows(dc, rs, a.dctx + row * L * (long long)H + head * dh, H, L, dh, lane);
    __syncwarp();
    scores_and_probs(q, k, c, rs, a.mask + row * L, L, dh, lane, p1, p2, nrm, madd, cosm);
    // dA_ij = dctx_i . v_j ;  A_ij (with dropout) kept in dS1 for the dV product
    for (int e = lane; e < L * L; e += 32) {
      const int i = e / L, j = e - i * L;
      dA[e] = dot_rows(dc + i * rs, v + j * rs, dh);
      float d1 = p1[e], d2 = p2[e];
      if (a.dropout_p > 0.f) {
        const uint64_t idx = (uint64_t)item * L * L + e;
        d1 = dropout_keep(a.dropout_seed, a.dropout_site, idx, a.dropout_p) ? d1 * keep_scale : 0.f;
        d2 = dropout_keep(a.dropout_seed, a.dropout_site + 1, idx, a.dropout_p) ? d2 * keep_scale : 0.f;
      }
      dS1[e] = a.beta * d1 + (1.f - a.beta) * d2;
    }
    __syncwarp();
    uint16_t* dst = a.dqkvc + row * L * ld + head * dh;
    // dV_j = sum_i A_ij dctx_i
    for (int w = 2 * lane; w < dh; w += 64) {
      for (int j = 0; j < L; ++j) {
        float acc0 = 0.f, acc1 = 0.f;
        for (int i = 0; i < L; ++i) {
          float g0, g1;
          unpack_bf16x2(*reinterpret_cast<const uint32_t*>(dc + i * rs + w), g0, g1);
          const float aij = dS1[i * L + j];
          acc0 = fmaf(aij, g0, acc0);
          acc1 = fmaf(aij, g1, acc1);
        }
        *reinterpret_cast<uint32_t*>(dst + 2 * H + (long long)j * ld + w) = pack_bf16x2(acc0, acc1);
      }
    }
    __syncwarp();
    // softmax backward, one lane per row: dS = P * (dP - sum_j dP P)
    for (int i = lane; i < L; i += 32) {
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
    __syncwarp();
    // D = dcos + dcos^T with dcos = -dS1 ; store D in p1 (P1 no longer needed)
    for (int e = lane; e < L * L; e += 32) {
      const int i = e / L, j = e - i * L;
      p1[e] = -(dS1[e] + dS1[j * L + i]);
    }
    __syncwarp();
    for (int w = 2 * lane; w < dh; w += 64) {
      for (int i = 0; i < L; ++i) {
        float dq0 = 0.f, dq1 = 0.f, dk0 = 0.f, dk1 = 0.f, dc0 = 0.f, dc1 = 0.f;
        float ci0, ci1;
        unpack_bf16x2(*reinterpret_cast<const uint32_t*>(c + i * rs + w), ci0, ci1);
        const float ni = nrm[i];
        for (int j = 0; j < L; ++j) {
          float k0, k1, q0, q1, cj0, cj1;
          unpack_bf16x2(*reinterpret_cast<const uint32_t*>(k + j * rs + w), k0, k1);
          unpack_bf16x2(*reinterpret_cast<const uint32_t*>(q + j * rs + w), q0, q1);
          unpack_bf16x2(*reinterpret_cast<const uint32_t*>(c + j * rs + w), cj0, cj1);
          const float ds_ij = dA[i * L + j], ds_ji = dA[j * L + i];
          dq0 = fmaf(ds_ij, k0, dq0); dq1 = fmaf(ds_ij, k1, dq1);
          dk0 = fmaf(ds_ji, q0, dk0); dk1 = fmaf(ds_ji, q1, dk1);
          const float Dij = p1[i * L + j];
          const float inv = 1.f / (ni * nrm[j]);
          const float cs = cosm[i * L + j] / (ni * ni);
          dc0 += Dij * (cj0 * inv - cs * ci0);
          dc1 += Dij * (cj1 * inv - cs * ci1);
        }
        *reinterpret_cast<uint32_t*>(dst + (long long)i * ld + w) = pack_bf16x2(dq0 * inv_sqrt_dh, dq1 * inv_sqrt_dh);
        *reinterpret_cast<uint32_t*>(dst + H + (long long)i * ld + w) = pack_bf16x2(dk0 * inv_sqrt_dh, dk1 * inv_sqrt_dh);
        *reinterpret_cast<uint32_t*>(dst + 3 * H + (long long)i * ld + w) = pack_bf16x2(dc0, dc1);
      }
    }
    __syncwarp();
  }
}

static int attn_generic(const pmgt_attn_args* a, bool bwd, cudaStream_t st) {
  const int dh = a->H / a->heads;
  const AttnSmemLayout lay = attn_layout(a->L, dh);
  const size_t per = bwd ? lay.per_warp_bwd : lay.per_warp_fwd;
  const size_t budget = 200 * 1024;
  PMGT_REQUIRE(per <= budget, "attention: L=%d, head size %d needs %zu bytes of shared memory per warp (> %zu)", a->L, dh,
               per, budget);
  int warps = (int)(budget / per);
  if (warps > 4) warps = 4;
  const size_t smem = per * warps;
  if (smem > 48 * 1024) {
    if (bwd) PMGT_CHECK_CUDA(cudaFuncSetAttribute(attn_core_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    else PMGT_CHECK_CUDA(cudaFuncSetAttribute(attn_core_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  const long long items = a->rows * a->heads;
  long long ctas = (items + warps - 1) / warps;
  const long long cap = (long long)num_sms() * 8;
  if (ctas > cap) ctas = cap;
  if (bwd) attn_core_bwd_kernel<<<(unsigned)ctas, 128, smem, st>>>(*a, warps, lay);
  else attn_core_fwd_kernel<<<(unsigned)ctas, 128, smem, st>>>(*a, warps, lay);
  PMGT_LAUNCH_CHECK();
  return PMGT_OK;
}

// Launchers of the other kernel families; each assumes attn_family() chose it.
int attn_mma_fwd(const pmgt_attn_args* a, cudaStream_t st);  // attention_mma.cu
int attn_mma_bwd(const pmgt_attn_args* a, cudaStream_t st);
int attn_reg_fwd(const pmgt_attn_args* a, cudaStream_t st);  // attention_reg.cu
int attn_reg_bwd(const pmgt_attn_args* a, cudaStream_t st);
int attn_mid_fwd(const pmgt_attn_args* a, cudaStream_t st);  // attention_mid.cu
int attn_mid_bwd(const pmgt_attn_args* a, cudaStream_t st);
bool attn_mid_fits(int L, int dh);

enum class AttnFamily { Mma, Reg, Mid, Generic };

// The table at the top of this file.  Only the shape decides, not pointers and not the direction, so the backward pass
// runs the family of its forward pass and regenerates the dropout mask that one drew (attn_reg has a stream of its
// own).  The head sizes below are multiples of 16, so H is a multiple of 8 and, with the base pointers 16-byte aligned
// (attn_check), so is every row the tensor-core families stage.
static AttnFamily attn_family(const pmgt_attn_args* a) {
  const int L = a->L, dh = a->H / a->heads;
  const bool reg_dh = dh == 32 || dh == 64 || dh == 128;
  if (L == 6 && reg_dh) return AttnFamily::Mma;
  if (L > 8 && L <= 64) {
    if (reg_dh && a->rows * a->heads <= 0x7fffffffll) return AttnFamily::Reg;  // one CTA per (sequence, head)
    if (dh % 16 == 0 && attn_mid_fits(L, dh)) return AttnFamily::Mid;
  }
  return AttnFamily::Generic;
}

static bool misaligned16(const void* p) { return ((uintptr_t)p & 15) != 0; }

// the argument checks of both entry points, made before any CUDA call
static int attn_check(const pmgt_attn_args* a, bool bwd) {
  const char* fn = bwd ? "pmgt_attn_core_bwd" : "pmgt_attn_core_fwd";
  PMGT_REQUIRE(a && a->qkvc && a->mask && (bwd ? a->dctx && a->dqkvc : a->ctx != nullptr), "%s: null argument", fn);
  PMGT_REQUIRE(!misaligned16(a->qkvc), "%s: qkvc must be 16-byte aligned", fn);
  if (bwd) {
    PMGT_REQUIRE(!misaligned16(a->dctx), "%s: dctx must be 16-byte aligned", fn);
    PMGT_REQUIRE(!misaligned16(a->dqkvc), "%s: dqkvc must be 16-byte aligned", fn);
  } else {
    PMGT_REQUIRE(!misaligned16(a->ctx), "%s: ctx must be 16-byte aligned", fn);
  }
  PMGT_REQUIRE(a->heads >= 1 && a->H % a->heads == 0, "attention: H must be divisible by heads");
  PMGT_REQUIRE((a->H / a->heads) % 2 == 0, "attention: head size must be even");
  PMGT_REQUIRE(a->L >= 1 && a->L <= 128, "attention: L must be in [1,128]");
  return PMGT_OK;
}

}  // namespace pmgt

using namespace pmgt;

extern "C" {

int pmgt_attn_core_fwd(const pmgt_attn_args* a, void* stream) {
  const int rc = attn_check(a, false);
  if (rc || a->rows == 0) return rc;
  const cudaStream_t st = (cudaStream_t)stream;
  switch (attn_family(a)) {
    case AttnFamily::Mma: return attn_mma_fwd(a, st);
    case AttnFamily::Reg: return attn_reg_fwd(a, st);
    case AttnFamily::Mid: return attn_mid_fwd(a, st);
    default: return attn_generic(a, false, st);
  }
}

int pmgt_attn_core_bwd(const pmgt_attn_args* a, void* stream) {
  int rc = attn_check(a, true);
  if (rc || a->rows == 0) return rc;
  const cudaStream_t st = (cudaStream_t)stream;
  switch (attn_family(a)) {
    case AttnFamily::Mma: rc = attn_mma_bwd(a, st); break;
    case AttnFamily::Reg: rc = attn_reg_bwd(a, st); break;
    case AttnFamily::Mid: rc = attn_mid_bwd(a, st); break;
    default: rc = attn_generic(a, true, st);
  }
  if (rc == PMGT_OK && a->d_bias_qkvc) rc = pmgt_colsum_bf16(a->dqkvc, a->rows * a->L, 4ll * a->H, 4ll * a->H, a->d_bias_qkvc, stream);
  return rc;
}

}  // extern "C"
