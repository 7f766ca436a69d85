// Attention maps of the K3 attention core: for every (sequence, head) the L x L matrix the core multiplies V with,
//   A = beta drop(P1) + (1 - beta) drop(P2),   P1 = softmax(1 - cos(C_i, C_j) + I + mask),  P2 = softmax(Q K^T / sqrt(dh) + mask)
// written as fp32 [rows][heads][L][L] (pmgt_attn_maps_fwd in attention.cu validates and dispatches).  This file holds
// the tensor-core path, for head sizes that are a multiple of 16; other even head sizes run a scalar kernel in
// attention.cu that shares the generic core's code.
//
// Layout: one CTA per (sequence, head), one warp per 16 query rows (MT = ceil(L / 16) warps, L <= 128), like attn_reg /
// attn_long.  Both products run as mma.sync m16n8k16 on ldmatrix operands, over the head dimension in 64-column
// chunks staged in shared memory, so shared memory does not grow with dh:
//   pass 1  S1 = C C^T (+ the squared norms of C), cosine, mask, softmax, dropout -> beta drop(P1) into a per-warp
//           fp32 row buffer;
//   pass 2  S2 = Q K^T, scale, mask, softmax, dropout -> (1 - beta) drop(P2) added to the buffer;
// then each warp writes its 16 rows, a contiguous range of the output, with coalesced stores.
// The arithmetic is that of the cores: fp32 scores, reciprocal norms, the additive -10000 key mask, padded key columns
// at -inf, max-subtracted exponentials.  The dropout mask is the one the core of the same shape applied: attn_reg's
// own stream (attention_drop.cuh) when attn_family() picks attn_reg, else the common.cuh element stream
// dropout_keep(seed, site, item L L + i L + j) with site + 1 for P2 (attn_mma, attn_mid, attn_long, generic).
#include "attention_drop.cuh"

namespace pmgt {

namespace {

constexpr int kMapKC = 64;            // head-dimension columns staged per chunk
constexpr int kMapRS = kMapKC + 8;    // row pitch of a staged chunk (bf16): 16-byte aligned, ldmatrix conflict-free

__device__ __forceinline__ uint32_t maddr(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mldsm4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void mmma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float mquad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  return v;
}
__device__ __forceinline__ float mquad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
  return v;
}

template <int MT>
struct MapCfg {
  static constexpr int LP = 16 * MT;       // padded sequence length
  static constexpr int NT = 2 * MT;        // 8-wide column tiles of a score row block
  static constexpr int THREADS = 32 * MT;
  static constexpr int BP = LP + 4;        // row pitch of the fp32 row buffer
  static constexpr size_t kSmem = 2 * (size_t)LP * kMapRS * 2 + 2 * (size_t)LP * 4 + (size_t)MT * 16 * BP * 4;
};

// columns [0, kw) of rows [0, L) of one head -> tile[LP][kMapRS]; rows [L, LP) are zero
template <int MT>
__device__ __forceinline__ void stage_chunk(uint16_t* tile, const uint16_t* __restrict__ src, long long ld, int L, int kw,
                                            int tid) {
  using Cf = MapCfg<MT>;
  const int cpr = kw >> 3;
  for (int e = tid; e < Cf::LP * cpr; e += Cf::THREADS) {
    const int i = e / cpr, c = e - i * cpr;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (i < L) v = __ldg(reinterpret_cast<const uint4*>(src + (long long)i * ld + c * 8));
    *reinterpret_cast<uint4*>(tile + i * kMapRS + c * 8) = v;
  }
}

// d[nt][*] += A(rows warp * 16 .. + 15, columns [0, kw)) . B(all LP rows, same columns)^T
template <int MT>
__device__ __forceinline__ void chunk_nt(float (&d)[2 * MT][4], const uint16_t* A, const uint16_t* B, int warp, int lane,
                                         int kw) {
  for (int ks = 0; ks < kw; ks += 16) {
    uint32_t af[4];
    mldsm4(maddr(A + (warp * 16 + (lane & 15)) * kMapRS + ks + (lane >> 4) * 8), af);
#pragma unroll
    for (int np = 0; np < MT; ++np) {
      uint32_t bf[4];
      mldsm4(maddr(B + (np * 16 + (lane & 7) + ((lane >> 4) << 3)) * kMapRS + ks + ((lane >> 3) & 1) * 8), bf);
      mmma(d[2 * np], af, bf[0], bf[1]);
      mmma(d[2 * np + 1], af, bf[2], bf[3]);
    }
  }
}

// dropout multipliers of element (i, j) of P1 (f1) and P2 (f2), from the stream of the core that owns this shape
struct MapDrop {
  DropKey dk;          // attn_reg stream
  uint64_t base;       // common.cuh stream: item L L
  bool reg, on;
  float scale;
};
__device__ __forceinline__ void map_drop(const MapDrop& d, const pmgt_attn_args& a, int i, int j, int L, float& f1,
                                         float& f2) {
  if (d.reg) {
    drop_factors(d.dk, (uint32_t)(i * L + j), f1, f2);
  } else if (d.on) {
    const uint64_t idx = d.base + (uint64_t)(i * L + j);
    f1 = dropout_keep(a.dropout_seed, a.dropout_site, idx, a.dropout_p) ? d.scale : 0.f;
    f2 = dropout_keep(a.dropout_seed, a.dropout_site + 1, idx, a.dropout_p) ? d.scale : 0.f;
  } else {
    f1 = 1.f;
    f2 = 1.f;
  }
}

// row softmax of a score block in accumulator layout (rows g / g + 8 of the warp's 16), in place
template <int NT>
__device__ __forceinline__ void frag_softmax(float (&s)[NT][4]) {
  float ma = -INFINITY, mb = -INFINITY;
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    ma = fmaxf(ma, fmaxf(s[nt][0], s[nt][1]));
    mb = fmaxf(mb, fmaxf(s[nt][2], s[nt][3]));
  }
  ma = mquad_max(ma);
  mb = mquad_max(mb);
  float za = 0.f, zb = 0.f;
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    s[nt][0] = __expf(s[nt][0] - ma); s[nt][1] = __expf(s[nt][1] - ma);
    s[nt][2] = __expf(s[nt][2] - mb); s[nt][3] = __expf(s[nt][3] - mb);
    za += s[nt][0] + s[nt][1];
    zb += s[nt][2] + s[nt][3];
  }
  za = 1.f / mquad_sum(za);
  zb = 1.f / mquad_sum(zb);
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    s[nt][0] *= za; s[nt][1] *= za;
    s[nt][2] *= zb; s[nt][3] *= zb;
  }
}

template <int MT>
__global__ void __launch_bounds__(32 * MT) attn_maps_mma_kernel(const pmgt_attn_args a, float* __restrict__ maps,
                                                                int reg_stream) {
  using Cf = MapCfg<MT>;
  extern __shared__ __align__(16) unsigned char smem[];
  uint16_t* tA = reinterpret_cast<uint16_t*>(smem);
  uint16_t* tB = tA + Cf::LP * kMapRS;
  float* rn = reinterpret_cast<float*>(tB + Cf::LP * kMapRS);   // squared norms of C, then their reciprocal roots
  float* madd = rn + Cf::LP;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  float* wbuf = madd + Cf::LP + warp * 16 * Cf::BP;
  const int L = a.L, H = a.H, heads = a.heads, dh = H / heads;
  const long long ld = 4ll * H;
  const long long n_items = a.rows * heads;
  const float inv_sqrt_dh = rsqrtf((float)dh);
  const float beta = a.beta;
  const int i0 = warp * 16 + g, i1 = i0 + 8;
  MapDrop md;
  md.reg = reg_stream != 0;
  md.on = a.dropout_p > 0.f;
  md.scale = md.on ? 1.f / (1.f - a.dropout_p) : 1.f;
  for (long long item = blockIdx.x; item < n_items; item += gridDim.x) {
    const long long row = item / heads;
    const int head = (int)(item - row * heads);
    const uint16_t* src = a.qkvc + row * L * ld + (long long)head * dh;
    md.base = (uint64_t)item * (uint64_t)L * (uint64_t)L;
    if (md.reg) md.dk = drop_key(a.dropout_seed, a.dropout_site, a.dropout_p, item);
    __syncthreads();  // the previous item's readers of rn / madd are done
    for (int i = tid; i < Cf::LP; i += Cf::THREADS) {
      rn[i] = 0.f;
      madd[i] = i < L ? (1.f - a.mask[row * L + i]) * -10000.f : -INFINITY;
    }
    float s[Cf::NT][4];
    // ---- pass 1: S1 = C C^T and the squared norms of C
#pragma unroll
    for (int nt = 0; nt < Cf::NT; ++nt) s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
    for (int kc = 0; kc < dh; kc += kMapKC) {
      const int kw = min(kMapKC, dh - kc);
      __syncthreads();  // the previous chunk's readers are done
      stage_chunk<MT>(tA, src + 3 * H + kc, ld, L, kw, tid);
      __syncthreads();
      for (int i = tid; i < L; i += Cf::THREADS) {  // the same thread owns row i in every chunk
        float q = rn[i];
        for (int c = 0; c < kw; c += 2) {
          float x, y;
          unpack_bf16x2(*reinterpret_cast<const uint32_t*>(tA + i * kMapRS + c), x, y);
          q = fmaf(x, x, q);
          q = fmaf(y, y, q);
        }
        rn[i] = q;
      }
      chunk_nt<MT>(s, tA, tA, warp, lane, kw);
    }
    __syncthreads();
    for (int i = tid; i < Cf::LP; i += Cf::THREADS) rn[i] = i < L ? 1.f / sqrtf(rn[i]) : 1.f;
    __syncthreads();
    {
      const float rn0 = rn[i0], rn1 = rn[i1];
#pragma unroll
      for (int nt = 0; nt < Cf::NT; ++nt) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int j = nt * 8 + 2 * t + (e & 1);
          const int i = e < 2 ? i0 : i1;
          const float cs = s[nt][e] * (e < 2 ? rn0 : rn1) * rn[j];
          s[nt][e] = 1.f - cs + (i == j ? 1.f : 0.f) + madd[j];
        }
      }
      frag_softmax<Cf::NT>(s);
#pragma unroll
      for (int nt = 0; nt < Cf::NT; ++nt) {
        const int j = nt * 8 + 2 * t;
        float f1a, f2a, f1b, f2b, f1c, f2c, f1d, f2d;
        map_drop(md, a, i0, j, L, f1a, f2a);
        map_drop(md, a, i0, j + 1, L, f1b, f2b);
        map_drop(md, a, i1, j, L, f1c, f2c);
        map_drop(md, a, i1, j + 1, L, f1d, f2d);
        *reinterpret_cast<float2*>(wbuf + g * Cf::BP + j) = make_float2(beta * (s[nt][0] * f1a), beta * (s[nt][1] * f1b));
        *reinterpret_cast<float2*>(wbuf + (g + 8) * Cf::BP + j) =
            make_float2(beta * (s[nt][2] * f1c), beta * (s[nt][3] * f1d));
      }
    }
    // ---- pass 2: S2 = Q K^T
#pragma unroll
    for (int nt = 0; nt < Cf::NT; ++nt) s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
    for (int kc = 0; kc < dh; kc += kMapKC) {
      const int kw = min(kMapKC, dh - kc);
      __syncthreads();
      stage_chunk<MT>(tA, src + kc, ld, L, kw, tid);
      stage_chunk<MT>(tB, src + H + kc, ld, L, kw, tid);
      __syncthreads();
      chunk_nt<MT>(s, tA, tB, warp, lane, kw);
    }
#pragma unroll
    for (int nt = 0; nt < Cf::NT; ++nt) {
#pragma unroll
      for (int e = 0; e < 4; ++e) s[nt][e] = s[nt][e] * inv_sqrt_dh + madd[nt * 8 + 2 * t + (e & 1)];
    }
    frag_softmax<Cf::NT>(s);
    const float omb = 1.f - beta;
#pragma unroll
    for (int nt = 0; nt < Cf::NT; ++nt) {
      const int j = nt * 8 + 2 * t;
      float f1a, f2a, f1b, f2b, f1c, f2c, f1d, f2d;
      map_drop(md, a, i0, j, L, f1a, f2a);
      map_drop(md, a, i0, j + 1, L, f1b, f2b);
      map_drop(md, a, i1, j, L, f1c, f2c);
      map_drop(md, a, i1, j + 1, L, f1d, f2d);
      float2* r0 = reinterpret_cast<float2*>(wbuf + g * Cf::BP + j);
      float2* r1 = reinterpret_cast<float2*>(wbuf + (g + 8) * Cf::BP + j);
      float2 v0 = *r0, v1 = *r1;
      v0.x += omb * (s[nt][0] * f2a); v0.y += omb * (s[nt][1] * f2b);
      v1.x += omb * (s[nt][2] * f2c); v1.y += omb * (s[nt][3] * f2d);
      *r0 = v0;
      *r1 = v1;
    }
    __syncwarp();
    // this warp's rows [warp * 16, min(L, warp * 16 + 16)) are one contiguous range of the output
    const int nr = min(16, L - warp * 16);
    float* out = maps + item * L * L + (long long)warp * 16 * L;
    for (int e = lane; e < nr * L; e += 32) {
      const int r = e / L, c = e - r * L;
      out[e] = wbuf[r * Cf::BP + c];
    }
    __syncwarp();
  }
}

template <int MT>
int launch_maps(const pmgt_attn_args* a, float* maps, bool reg_stream, cudaStream_t st) {
  using Cf = MapCfg<MT>;
  static unsigned long long configured = 0;
  if (first_use_on_device(configured))
    PMGT_CHECK_CUDA(cudaFuncSetAttribute(attn_maps_mma_kernel<MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cf::kSmem));
  const long long items = a->rows * a->heads;
  long long ctas = items;
  const long long cap = (long long)num_sms() * 32;  // items beyond the resident CTAs are taken in a grid-stride loop
  if (ctas > cap) ctas = cap;
  attn_maps_mma_kernel<MT><<<(unsigned)ctas, Cf::THREADS, Cf::kSmem, st>>>(*a, maps, reg_stream ? 1 : 0);
  PMGT_LAUNCH_CHECK();
  return PMGT_OK;
}

}  // namespace

// 1 <= L <= 128, head size a multiple of 16; reg_stream: attn_family() chose attn_reg for this shape
int attn_maps_mma(const pmgt_attn_args* a, float* maps, bool reg_stream, cudaStream_t st) {
  switch ((a->L + 15) / 16) {
    case 1: return launch_maps<1>(a, maps, reg_stream, st);
    case 2: return launch_maps<2>(a, maps, reg_stream, st);
    case 3: return launch_maps<3>(a, maps, reg_stream, st);
    case 4: return launch_maps<4>(a, maps, reg_stream, st);
    case 5: return launch_maps<5>(a, maps, reg_stream, st);
    case 6: return launch_maps<6>(a, maps, reg_stream, st);
    case 7: return launch_maps<7>(a, maps, reg_stream, st);
    case 8: return launch_maps<8>(a, maps, reg_stream, st);
    default: break;
  }
  set_error("attn_maps: no kernel for L=%d", a->L);
  return PMGT_ERR_INVALID;
}

}  // namespace pmgt
