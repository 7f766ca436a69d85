// PMGTEmbeddings fusion (modeling_pmgt.py:199-208) for M = 1, 3 or 4 feature modalities: tanh of the M projected
// rows, M logits s_k = w_att[k] . [tanh e_0; ..; tanh e_{M-1}] + b_att[k], an M-way softmax, the weighted sum plus
// position and role, LayerNorm and dropout -- and the backward pass.  M = 2 keeps its own kernels (embed128.cu,
// rowwise.cu); pmgt_embed_multi_fwd / _bwd forward that case to pmgt_embed_fuse_fwd / _bwd unchanged.
//
// Two variants, each templated on M:
//  * H = 128 (the default encoder): the layout of embed128.cu -- half a warp per token, eight columns per lane, the
//    next token's M rows prefetched into registers.  w_att (M^2 * 128 fp32, 8 KB at M = 4) lives in shared memory in a
//    lane-interleaved layout.  Backward keeps d LayerNorm, d position and the M projection-bias gradients in registers;
//    the d_w_att partial sums go to shared-memory rows private to each half-warp (no atomics, no shuffles), folded
//    once per CTA at the end with one global atomic per value.  Only the rows k < M - 1 are accumulated: the softmax
//    gradient sums to zero over k (sum_k a_k (da_k - sum_j a_j da_j) = 0), so row M - 1 is minus the sum of the others.
//  * generic H (a multiple of 8 up to 1024): a warp per token like rowwise.cu, per-CTA shared-memory accumulators
//    of (3 + M + M^2) * H floats.
//
// Dropout uses the stream of every other embedding kernel: element tok * H + h, the caller's seed and site, so the mask
// does not depend on M and forward and backward may mix variants.  At M = 1 the softmax weight is exactly 1 and the
// w_att / b_att gradients are exactly 0.
#include "common.cuh"

namespace pmgt {

namespace {

constexpr int kThreads = 256;

__device__ __forceinline__ float half_sum(float v) {  // reduction over the 16 lanes of a half-warp
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ void ld8(const float* __restrict__ p, float (&v)[8]) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p));
  const float4 b = __ldg(reinterpret_cast<const float4*>(p + 4));
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

__device__ __forceinline__ void unpack8(const uint4& u, float (&v)[8]) {
  unpack_bf16x2(u.x, v[0], v[1]); unpack_bf16x2(u.y, v[2], v[3]);
  unpack_bf16x2(u.z, v[4], v[5]); unpack_bf16x2(u.w, v[6], v[7]);
}

__device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
  uint4 u;
  u.x = pack_bf16x2(v[0], v[1]); u.y = pack_bf16x2(v[2], v[3]);
  u.z = pack_bf16x2(v[4], v[5]); u.w = pack_bf16x2(v[6], v[7]);
  return u;
}

__device__ __forceinline__ uint4 ldg16(const uint16_t* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }

__device__ __forceinline__ void red_v4(float* addr, float x, float y, float z, float w) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}

// ---------------------------------------------------------------------------------------------------------------------
// H = 128
// ---------------------------------------------------------------------------------------------------------------------
// Shared-memory layout of a [rows][128] fp32 matrix as read by the half-warp lanes: the eight columns 8 hl .. 8 hl + 7
// of row r are the float4s [(2 r + q) * 16 + hl], q = 0, 1.  Sixteen lanes read 256 consecutive bytes: no bank conflict.
__device__ __forceinline__ int il(int row, int q, int hl) { return (row * 2 + q) * 16 + hl; }

// a shared-memory load the compiler may not hoist out of the token loop: left to itself it keeps all 2 M^2 float4s of
// w_att in registers (128 at M = 4) and spills
__device__ __forceinline__ float4 lds4(const float4* p) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"((uint32_t)__cvta_generic_to_shared(p)));
  return v;
}

template <int M>
__device__ __forceinline__ void stage_w128(const float* __restrict__ w, float4* ws) {
  for (int i = threadIdx.x; i < M * M * 32; i += kThreads) {  // float4 i of w_att: row i / 32, columns 4 (i % 32) ..
    const int r = i & 31;
    ws[il(i >> 5, r & 1, r >> 1)] = __ldg(reinterpret_cast<const float4*>(w) + i);
  }
}

__device__ __forceinline__ float dot8(const float4& a, const float4& b, const float (&t)[8]) {
  return a.x * t[0] + a.y * t[1] + a.z * t[2] + a.w * t[3] + b.x * t[4] + b.y * t[5] + b.z * t[6] + b.w * t[7];
}

__device__ __forceinline__ void tanh8(const uint4& u, float (&t)[8]) {
  unpack8(u, t);
#pragma unroll
  for (int j = 0; j < 8; ++j) t[j] = tanhf(t[j]);
}

// Forward math of one token shared by both passes.  In: the M packed projected rows, staged w_att, b_att, position +
// role.  Out: softmax weights att, z (pre-LayerNorm), mean, rstd.
template <int M>
__device__ __forceinline__ void fuse128(const uint4 (&c)[M], const float4* __restrict__ ws, int hl, const float (&ba)[M],
                                        const float (&pr)[8], float eps, float (&att)[M], float (&z)[8], float& mean,
                                        float& rstd) {
  if constexpr (M == 1) {
    att[0] = 1.f;
  } else {
    float s[M];
#pragma unroll
    for (int k = 0; k < M; ++k) s[k] = 0.f;
#pragma unroll
    for (int m = 0; m < M; ++m) {
      float t[8];
      tanh8(c[m], t);
#pragma unroll
      for (int k = 0; k < M; ++k) s[k] += dot8(lds4(ws + il(k * M + m, 0, hl)), lds4(ws + il(k * M + m, 1, hl)), t);
    }
    float mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < M; ++k) {
      s[k] = half_sum(s[k]) + ba[k];
      mx = fmaxf(mx, s[k]);
    }
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < M; ++k) {
      s[k] = __expf(s[k] - mx);
      sum += s[k];
    }
    const float inv = 1.f / sum;
#pragma unroll
    for (int k = 0; k < M; ++k) att[k] = s[k] * inv;
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) z[j] = pr[j];
#pragma unroll
  for (int m = 0; m < M; ++m) {
    float e[8];
    unpack8(c[m], e);
#pragma unroll
    for (int j = 0; j < 8; ++j) z[j] = fmaf(att[m], e[j], z[j]);
  }
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) s += z[j];
  mean = half_sum(s) * (1.f / 128.f);
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) { const float d = z[j] - mean; q = fmaf(d, d, q); }
  rstd = rsqrtf(half_sum(q) * (1.f / 128.f) + eps);
}

template <int M>
__global__ void __launch_bounds__(kThreads, 2) embed_multi_fwd128_kernel(const pmgt_embed_multi_args a) {
  extern __shared__ float4 ws[];  // [M * M][128] w_att, layout il()
  stage_w128<M>(a.w_att, ws);
  __syncthreads();
  const int lane = threadIdx.x & 31, hl = lane & 15, sub = lane >> 4;
  const int h0 = hl * 8;
  float ba[M];
#pragma unroll
  for (int k = 0; k < M; ++k) ba[k] = __ldg(a.b_att + k);
  const float ks = a.dropout_p > 0.f ? 1.f / (1.f - a.dropout_p) : 1.f;
  const long long T = a.rows * a.L;
  const long long stride = (long long)gridDim.x * (kThreads / 32) * 2;
  long long base = ((long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5)) * 2;
  if (base >= T) return;
  uint4 nx[M];  // register double buffer: operands of the token after this one
  {
    const long long t0 = min(base + sub, T - 1);
    const long long er = a.row_idx ? __ldg(a.row_idx + t0) : t0;
#pragma unroll
    for (int m = 0; m < M; ++m) nx[m] = ldg16(a.e[m] + er * 128 + h0);
  }
  const int l_step = (int)(stride % a.L);
  int l = (int)((base + sub) % a.L);
  for (; base < T; base += stride) {
    const long long tok = base + sub;
    const bool valid = tok < T;
    uint4 cx[M];
#pragma unroll
    for (int m = 0; m < M; ++m) cx[m] = nx[m];
    if (base + stride < T) {
      const long long t1 = min(base + stride + sub, T - 1);
      const long long er = a.row_idx ? __ldg(a.row_idx + t1) : t1;
#pragma unroll
      for (int m = 0; m < M; ++m) nx[m] = ldg16(a.e[m] + er * 128 + h0);
    }
    const long long tc = valid ? tok : T - 1;
    float pr[8], rr[8];
    ld8(a.pos + (long long)l * 128 + h0, pr);
    ld8(a.role + (l > 0 ? 128 : 0) + h0, rr);
#pragma unroll
    for (int j = 0; j < 8; ++j) pr[j] += rr[j];
    float att[M], z[8], mean, rstd;
    fuse128<M>(cx, ws, hl, ba, pr, a.ln_eps, att, z, mean, rstd);
    uint32_t keep = 0xffu;
    if (a.dropout_p > 0.f) keep = dropout_keep8(a.dropout_seed, a.dropout_site, (uint64_t)tc * 128u + (uint64_t)h0, a.dropout_p);
    float y[8], g[8], b[8];  // LayerNorm affine re-read from L1 each token: two CTAs per SM need <= 128 registers
    ld8(a.ln_g + h0, g);
    ld8(a.ln_b + h0, b);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float v = (z[j] - mean) * rstd * g[j] + b[j];
      y[j] = (keep >> j) & 1u ? v * ks : 0.f;
    }
    if (valid) *reinterpret_cast<uint4*>(a.x_out + tok * 128 + h0) = pack8(y);
    l += l_step;
    if (l >= a.L) l -= a.L;
  }
}

// shared memory of the backward kernel, in float4 units: staged w_att, then the private d_w_att rows of the 16
// half-warps, then the CTA's fp32 fold rows (0 d_ln_g, 1 d_ln_b, 2 .. M + 1 d_bias, then L rows of d_pos, then M d_b_att)
template <int M>
__host__ __device__ constexpr int bwd128_w4() { return M * M * 32; }
template <int M>
__host__ __device__ constexpr int bwd128_dw4() { return 16 * (M - 1) * M * 32; }
template <int M>
size_t bwd128_smem(int L) { return (size_t)(bwd128_w4<M>() + bwd128_dw4<M>()) * 16 + ((size_t)(2 + M + L) * 128 + M) * 4; }

template <int M, bool TABLE>
__global__ void __launch_bounds__(kThreads, 1) embed_multi_bwd128_kernel(const pmgt_embed_multi_args a) {
  extern __shared__ float4 sm4[];
  float4* ws = sm4;
  float4* dwp = sm4 + bwd128_w4<M>() + (threadIdx.x >> 4) * ((M - 1) * M * 32);  // this half-warp's rows k < M - 1
  float* red = reinterpret_cast<float*>(sm4 + bwd128_w4<M>() + bwd128_dw4<M>());
  const int L = a.L;
  stage_w128<M>(a.w_att, ws);
  for (int i = threadIdx.x; i < bwd128_dw4<M>(); i += kThreads) sm4[bwd128_w4<M>() + i] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int i = threadIdx.x; i < (2 + M + L) * 128 + M; i += kThreads) red[i] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31, hl = lane & 15, sub = lane >> 4;
  const int h0 = hl * 8;
  float ba[M];
#pragma unroll
  for (int k = 0; k < M; ++k) ba[k] = __ldg(a.b_att + k);
  const float ks = a.dropout_p > 0.f ? 1.f / (1.f - a.dropout_p) : 1.f;
  float acc_g[8], acc_b[8], dbias[M][8], db[M];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    acc_g[j] = acc_b[j] = 0.f;
#pragma unroll
    for (int m = 0; m < M; ++m) dbias[m][j] = 0.f;
  }
#pragma unroll
  for (int k = 0; k < M; ++k) db[k] = 0.f;
  const long long stride = (long long)gridDim.x * (kThreads / 32) * 2;
  const long long first = ((long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5)) * 2;
  // position-major order: all rows of position l, then l + 1, so the position gradient accumulates in registers
  for (int l = 0; l < L; ++l) {
    float pr[8], rr[8], dpos[8];
    ld8(a.pos + (long long)l * 128 + h0, pr);
    ld8(a.role + (l > 0 ? 128 : 0) + h0, rr);
#pragma unroll
    for (int j = 0; j < 8; ++j) { pr[j] += rr[j]; dpos[j] = 0.f; }
    long long base = first;
    uint4 nx[M], nd = make_uint4(0, 0, 0, 0), nb = nd;
#pragma unroll
    for (int m = 0; m < M; ++m) nx[m] = nd;
    long long ner = 0;
    if (base < a.rows) {
      const long long t0 = min(base + sub, (long long)a.rows - 1) * L + l;
      ner = a.row_idx ? __ldg(a.row_idx + t0) : t0;
#pragma unroll
      for (int m = 0; m < M; ++m) nx[m] = ldg16(a.e[m] + ner * 128 + h0);
      nd = ldg16(a.dx + t0 * 128 + h0);
      if (a.dx_b) nb = ldg16(a.dx_b + t0 * 128 + h0);
    }
    for (; base < a.rows; base += stride) {
      const long long row = base + sub;
      const bool valid = row < a.rows;
      const long long tok = (valid ? row : a.rows - 1) * L + l;
      uint4 cx[M];
#pragma unroll
      for (int m = 0; m < M; ++m) cx[m] = nx[m];
      const uint4 cd = nd, cb = nb;
      const long long er = ner;
      if (base + stride < a.rows) {
        const long long t1 = min(base + stride + sub, (long long)a.rows - 1) * L + l;
        ner = a.row_idx ? __ldg(a.row_idx + t1) : t1;
#pragma unroll
        for (int m = 0; m < M; ++m) nx[m] = ldg16(a.e[m] + ner * 128 + h0);
        nd = ldg16(a.dx + t1 * 128 + h0);
        if (a.dx_b) nb = ldg16(a.dx_b + t1 * 128 + h0);
      }
      float att[M], z[8], mean, rstd;
      fuse128<M>(cx, ws, hl, ba, pr, a.ln_eps, att, z, mean, rstd);
      float d[8];
      unpack8(cd, d);
      if (a.dx_b) {
        float e[8];
        unpack8(cb, e);
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] += e[j];
      }
      uint32_t keep = valid ? 0xffu : 0u;  // an out-of-range half contributes exact zeros everywhere below
      if (a.dropout_p > 0.f) keep &= dropout_keep8(a.dropout_seed, a.dropout_site, (uint64_t)tok * 128u + (uint64_t)h0, a.dropout_p);
      // LayerNorm backward (gamma re-read from L1: registers are the scarce resource here)
      float g[8];
      ld8(a.ln_g + h0, g);
      float s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float dj = (keep >> j) & 1u ? d[j] * ks : 0.f;
        const float xh = (z[j] - mean) * rstd;
        acc_g[j] = fmaf(dj, xh, acc_g[j]);
        acc_b[j] += dj;
        const float dg = dj * g[j];
        s1 += dg;
        s2 = fmaf(dg, xh, s2);
        d[j] = dg;   // d now holds dy * gamma
        z[j] = xh;   // z now holds xhat
      }
      s1 = half_sum(s1) * (1.f / 128.f);
      s2 = half_sum(s2) * (1.f / 128.f);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        d[j] = rstd * (d[j] - s1 - z[j] * s2);   // d now holds dz
        dpos[j] += d[j];
      }
      // softmax over the M modality logits
      float ds[M];
      if constexpr (M == 1) {
        ds[0] = 0.f;
      } else {
        float da[M], dot = 0.f;
#pragma unroll
        for (int m = 0; m < M; ++m) {
          float e[8];
          unpack8(cx[m], e);
          float v = 0.f;
#pragma unroll
          for (int j = 0; j < 8; ++j) v = fmaf(d[j], e[j], v);
          da[m] = half_sum(v);
          dot = fmaf(da[m], att[m], dot);
        }
#pragma unroll
        for (int k = 0; k < M; ++k) {
          ds[k] = att[k] * (da[k] - dot);
          db[k] += ds[k];
        }
      }
#pragma unroll
      for (int m = 0; m < M; ++m) {
        float t[8], de[8];
        if constexpr (M == 1) {
#pragma unroll
          for (int j = 0; j < 8; ++j) de[j] = d[j];
        } else {
          tanh8(cx[m], t);
          float w[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) w[j] = 0.f;
#pragma unroll
          for (int k = 0; k < M; ++k) {
            const float4 w0 = lds4(ws + il(k * M + m, 0, hl)), w1 = lds4(ws + il(k * M + m, 1, hl));
            w[0] = fmaf(ds[k], w0.x, w[0]); w[1] = fmaf(ds[k], w0.y, w[1]);
            w[2] = fmaf(ds[k], w0.z, w[2]); w[3] = fmaf(ds[k], w0.w, w[3]);
            w[4] = fmaf(ds[k], w1.x, w[4]); w[5] = fmaf(ds[k], w1.y, w[5]);
            w[6] = fmaf(ds[k], w1.z, w[6]); w[7] = fmaf(ds[k], w1.w, w[7]);
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) de[j] = att[m] * d[j] + w[j] * (1.f - t[j] * t[j]);
#pragma unroll
          for (int k = 0; k < M - 1; ++k) {
            float4* p = dwp + il(k * M + m, 0, hl);
            float4 u = p[0], v = p[16];
            u.x = fmaf(ds[k], t[0], u.x); u.y = fmaf(ds[k], t[1], u.y); u.z = fmaf(ds[k], t[2], u.z); u.w = fmaf(ds[k], t[3], u.w);
            v.x = fmaf(ds[k], t[4], v.x); v.y = fmaf(ds[k], t[5], v.y); v.z = fmaf(ds[k], t[6], v.z); v.w = fmaf(ds[k], t[7], v.w);
            p[0] = u;
            p[16] = v;
          }
        }
        // bias gradient of the projections = column sums of the bf16-rounded d e_m
#pragma unroll
        for (int j = 0; j < 8; ++j) dbias[m][j] += bf16_bits_to_float(float_to_bf16_bits(de[j]));
        if (valid) {
          if (TABLE) {
            if (!(a.skip_row0 && er == 0)) {
              float* p = a.de_acc[m] + er * 128 + h0;
              red_v4(p, de[0], de[1], de[2], de[3]);
              red_v4(p + 4, de[4], de[5], de[6], de[7]);
            }
          } else {
            *reinterpret_cast<uint4*>(a.de[m] + tok * 128 + h0) = pack8(de);
          }
        }
      }
    }
    // position gradient of this l: fold the two halves, then into the CTA's shared row
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float v = dpos[j] + __shfl_xor_sync(0xffffffffu, dpos[j], 16);
      if (sub == 0 && v != 0.f) atomicAdd(&red[(2 + M + l) * 128 + h0 + j], v);
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float v = acc_g[j] + __shfl_xor_sync(0xffffffffu, acc_g[j], 16);
    if (sub == 0 && v != 0.f) atomicAdd(&red[0 * 128 + h0 + j], v);
    v = acc_b[j] + __shfl_xor_sync(0xffffffffu, acc_b[j], 16);
    if (sub == 0 && v != 0.f) atomicAdd(&red[1 * 128 + h0 + j], v);
#pragma unroll
    for (int m = 0; m < M; ++m) {
      v = dbias[m][j] + __shfl_xor_sync(0xffffffffu, dbias[m][j], 16);
      if (sub == 0 && v != 0.f) atomicAdd(&red[(2 + m) * 128 + h0 + j], v);
    }
  }
  if (hl == 0) {  // every lane of a half-warp holds the same per-token scalars
#pragma unroll
    for (int k = 0; k < M; ++k)
      if (db[k] != 0.f) atomicAdd(&red[(2 + M + L) * 128 + k], db[k]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < (2 + M) * 128; i += kThreads) {
    const float v = red[i];
    if (v == 0.f) continue;
    const int r = i >> 7, h = i & 127;
    atomicAdd((r == 0 ? a.d_ln_g : r == 1 ? a.d_ln_b : a.d_bias[r - 2]) + h, v);
  }
  for (int i = threadIdx.x; i < L * 128; i += kThreads) {
    const float v = red[(2 + M) * 128 + i];
    if (v == 0.f) continue;
    const int l = i >> 7, h = i & 127;
    atomicAdd(a.d_pos + (long long)l * 128 + h, v);
    atomicAdd(a.d_role + (l > 0 ? 128 : 0) + h, v);
  }
  if (threadIdx.x < M) {
    const float v = red[(2 + M + L) * 128 + threadIdx.x];
    if (v != 0.f) atomicAdd(a.d_b_att + threadIdx.x, v);
  }
  if constexpr (M > 1) {
    // d_w_att: fold the 16 private copies; row M - 1 = -(sum of the others)
    const float* dw0 = reinterpret_cast<const float*>(sm4 + bwd128_w4<M>());
    for (int i = threadIdx.x; i < M * 128; i += kThreads) {
      const int m = i >> 7, h = i & 127;
      const int off = il(0, (h >> 2) & 1, h >> 3) * 4 + (h & 3);  // offset of column h within an il() row
      float last = 0.f;
#pragma unroll
      for (int k = 0; k < M - 1; ++k) {
        float v = 0.f;
        for (int hw = 0; hw < 16; ++hw) v += dw0[hw * (M - 1) * M * 128 + (k * M + m) * 128 + off];
        last -= v;
        if (v != 0.f) atomicAdd(a.d_w_att + (k * M + m) * 128 + h, v);
      }
      if (last != 0.f) atomicAdd(a.d_w_att + ((M - 1) * M + m) * 128 + h, last);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// generic H: a warp per token, lane owns column quads h = 4 (lane + 32 i), i < G.  Only z and the incoming gradient
// stay in registers; the M projected rows are re-read (L1) in each pass, which keeps the register count independent of M.
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void ld4_bf16(const uint16_t* __restrict__ p, float (&v)[4]) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  unpack_bf16x2(u.x, v[0], v[1]);
  unpack_bf16x2(u.y, v[2], v[3]);
}

__device__ __forceinline__ float4 ld4_f32(const float* __restrict__ p) { return __ldg(reinterpret_cast<const float4*>(p)); }

__device__ __forceinline__ uint32_t keep4(const pmgt_embed_multi_args& a, uint64_t idx) {  // idx a multiple of 4
  if (a.dropout_p <= 0.f) return 0xfu;
  return dropout_keep8(a.dropout_seed, a.dropout_site, idx & ~(uint64_t)7, a.dropout_p) >> (uint32_t)(idx & 7);
}

// softmax weights, z (pre-LayerNorm) in registers, mean, rstd of token `tok` (projected row `er`, position l)
template <int M, int G>
__device__ __forceinline__ void fuse_row(const pmgt_embed_multi_args& a, long long er, int l, int lane, float (&att)[M],
                                         float (&z)[G][4], float& mean, float& rstd) {
  const int H = a.H;
  if constexpr (M == 1) {
    att[0] = 1.f;
  } else {
    float s[M];
#pragma unroll
    for (int k = 0; k < M; ++k) s[k] = 0.f;
#pragma unroll
    for (int i = 0; i < G; ++i) {
      const int h = (lane + 32 * i) * 4;
      if (h >= H) continue;
#pragma unroll
      for (int m = 0; m < M; ++m) {
        float t[4];
        ld4_bf16(a.e[m] + er * H + h, t);
#pragma unroll
        for (int j = 0; j < 4; ++j) t[j] = tanhf(t[j]);
#pragma unroll
        for (int k = 0; k < M; ++k) {
          const float4 w = ld4_f32(a.w_att + (long long)(k * M + m) * H + h);
          s[k] += w.x * t[0] + w.y * t[1] + w.z * t[2] + w.w * t[3];
        }
      }
    }
    float mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < M; ++k) {
      s[k] = warp_sum(s[k]) + __ldg(a.b_att + k);
      mx = fmaxf(mx, s[k]);
    }
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < M; ++k) {
      s[k] = __expf(s[k] - mx);
      sum += s[k];
    }
    const float inv = 1.f / sum;
#pragma unroll
    for (int k = 0; k < M; ++k) att[k] = s[k] * inv;
  }
  const float* pos = a.pos + (long long)l * H;
  const float* role = a.role + (l > 0 ? H : 0);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < G; ++i) {
    const int h = (lane + 32 * i) * 4;
    if (h >= H) {
      z[i][0] = z[i][1] = z[i][2] = z[i][3] = 0.f;
      continue;
    }
    const float4 p = ld4_f32(pos + h), r = ld4_f32(role + h);
    z[i][0] = p.x + r.x; z[i][1] = p.y + r.y; z[i][2] = p.z + r.z; z[i][3] = p.w + r.w;
#pragma unroll
    for (int m = 0; m < M; ++m) {
      float e[4];
      ld4_bf16(a.e[m] + er * H + h, e);
#pragma unroll
      for (int j = 0; j < 4; ++j) z[i][j] = fmaf(att[m], e[j], z[i][j]);
    }
    s += z[i][0] + z[i][1] + z[i][2] + z[i][3];
  }
  mean = warp_sum(s) / (float)H;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < G; ++i)
    if ((lane + 32 * i) * 4 < H) {
#pragma unroll
      for (int j = 0; j < 4; ++j) { const float d = z[i][j] - mean; q = fmaf(d, d, q); }
    }
  rstd = rsqrtf(warp_sum(q) / (float)H + a.ln_eps);
}

template <int M, int G>
__global__ void __launch_bounds__(kThreads, 1) embed_multi_fwd_kernel(const pmgt_embed_multi_args a) {
  const int lane = threadIdx.x & 31;
  const int H = a.H;
  const long long T = a.rows * a.L;
  const long long nwarps = (long long)gridDim.x * (kThreads / 32);
  const float ks = a.dropout_p > 0.f ? 1.f / (1.f - a.dropout_p) : 1.f;
  for (long long tok = (long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); tok < T; tok += nwarps) {
    const int l = (int)(tok % a.L);
    const long long er = a.row_idx ? a.row_idx[tok] : tok;
    float att[M], z[G][4], mean, rstd;
    fuse_row<M, G>(a, er, l, lane, att, z, mean, rstd);
#pragma unroll
    for (int i = 0; i < G; ++i) {
      const int h = (lane + 32 * i) * 4;
      if (h >= H) continue;
      const float4 g = ld4_f32(a.ln_g + h), b = ld4_f32(a.ln_b + h);
      const float ga[4] = {g.x, g.y, g.z, g.w}, bb[4] = {b.x, b.y, b.z, b.w};
      const uint32_t keep = keep4(a, (uint64_t)tok * H + h);
      float y[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float v = (z[i][j] - mean) * rstd * ga[j] + bb[j];
        y[j] = (keep >> j) & 1u ? v * ks : 0.f;
      }
      uint2 u;
      u.x = pack_bf16x2(y[0], y[1]);
      u.y = pack_bf16x2(y[2], y[3]);
      *reinterpret_cast<uint2*>(a.x_out + tok * H + h) = u;
    }
  }
}

// per-CTA shared accumulators, rows of H floats: 0 d_ln_g, 1 d_ln_b, 2 d_pos (current l), 3 .. 2 + M d_bias,
// 3 + M .. 2 + M + M^2 d_w_att
template <int M, int G>
__global__ void __launch_bounds__(kThreads, 1) embed_multi_bwd_kernel(const pmgt_embed_multi_args a) {
  extern __shared__ float acc[];
  const int lane = threadIdx.x & 31;
  const int H = a.H;
  for (int i = threadIdx.x; i < (3 + M + M * M) * H; i += kThreads) acc[i] = 0.f;
  __syncthreads();
  const long long nwarps = (long long)gridDim.x * (kThreads / 32);
  const long long warp0 = (long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5);
  const float ks = a.dropout_p > 0.f ? 1.f / (1.f - a.dropout_p) : 1.f;
  float db[M];
#pragma unroll
  for (int k = 0; k < M; ++k) db[k] = 0.f;
  for (int l = 0; l < a.L; ++l) {
    for (long long row = warp0; row < a.rows; row += nwarps) {
      const long long tok = row * a.L + l;
      const long long er = a.row_idx ? a.row_idx[tok] : tok;
      float att[M], z[G][4], d[G][4], mean, rstd;
      fuse_row<M, G>(a, er, l, lane, att, z, mean, rstd);
      // LayerNorm backward
      float s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int i = 0; i < G; ++i) {
        const int h = (lane + 32 * i) * 4;
        if (h >= H) continue;
        ld4_bf16(a.dx + tok * H + h, d[i]);
        if (a.dx_b) {
          float e[4];
          ld4_bf16(a.dx_b + tok * H + h, e);
#pragma unroll
          for (int j = 0; j < 4; ++j) d[i][j] += e[j];
        }
        const uint32_t keep = keep4(a, (uint64_t)tok * H + h);
        const float4 g = ld4_f32(a.ln_g + h);
        const float ga[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float dj = (keep >> j) & 1u ? d[i][j] * ks : 0.f;
          const float xh = (z[i][j] - mean) * rstd;
          atomicAdd(&acc[0 * H + h + j], dj * xh);
          atomicAdd(&acc[1 * H + h + j], dj);
          const float dg = dj * ga[j];
          s1 += dg;
          s2 = fmaf(dg, xh, s2);
          d[i][j] = dg;   // d now holds dy * gamma
          z[i][j] = xh;   // z now holds xhat
        }
      }
      s1 = warp_sum(s1) / (float)H;
      s2 = warp_sum(s2) / (float)H;
      float da[M];
#pragma unroll
      for (int m = 0; m < M; ++m) da[m] = 0.f;
#pragma unroll
      for (int i = 0; i < G; ++i) {
        const int h = (lane + 32 * i) * 4;
        if (h >= H) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          d[i][j] = rstd * (d[i][j] - s1 - z[i][j] * s2);   // d now holds dz
          atomicAdd(&acc[2 * H + h + j], d[i][j]);
        }
        if constexpr (M > 1) {
#pragma unroll
          for (int m = 0; m < M; ++m) {
            float e[4];
            ld4_bf16(a.e[m] + er * H + h, e);
#pragma unroll
            for (int j = 0; j < 4; ++j) da[m] = fmaf(d[i][j], e[j], da[m]);
          }
        }
      }
      float ds[M];
      if constexpr (M == 1) {
        ds[0] = 0.f;
      } else {
        float dot = 0.f;
#pragma unroll
        for (int m = 0; m < M; ++m) {
          da[m] = warp_sum(da[m]);
          dot = fmaf(da[m], att[m], dot);
        }
#pragma unroll
        for (int k = 0; k < M; ++k) {
          ds[k] = att[k] * (da[k] - dot);
          db[k] += ds[k];
        }
      }
      const bool skip = a.row_idx && a.skip_row0 && er == 0;
#pragma unroll
      for (int i = 0; i < G; ++i) {
        const int h = (lane + 32 * i) * 4;
        if (h >= H) continue;
#pragma unroll
        for (int m = 0; m < M; ++m) {
          float de[4];
          if constexpr (M == 1) {
#pragma unroll
            for (int j = 0; j < 4; ++j) de[j] = d[i][j];
          } else {
            float t[4], w[4] = {0.f, 0.f, 0.f, 0.f};
            ld4_bf16(a.e[m] + er * H + h, t);
#pragma unroll
            for (int j = 0; j < 4; ++j) t[j] = tanhf(t[j]);
#pragma unroll
            for (int k = 0; k < M; ++k) {
              const float4 wk = ld4_f32(a.w_att + (long long)(k * M + m) * H + h);
              w[0] = fmaf(ds[k], wk.x, w[0]); w[1] = fmaf(ds[k], wk.y, w[1]);
              w[2] = fmaf(ds[k], wk.z, w[2]); w[3] = fmaf(ds[k], wk.w, w[3]);
              float* p = &acc[(3 + M + k * M + m) * H + h];
#pragma unroll
              for (int j = 0; j < 4; ++j) atomicAdd(p + j, ds[k] * t[j]);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) de[j] = att[m] * d[i][j] + w[j] * (1.f - t[j] * t[j]);
          }
          // bias gradient of the projections = column sums of the bf16-rounded d e_m
#pragma unroll
          for (int j = 0; j < 4; ++j) atomicAdd(&acc[(3 + m) * H + h + j], bf16_bits_to_float(float_to_bf16_bits(de[j])));
          if (a.row_idx) {
            if (!skip) red_v4(a.de_acc[m] + er * H + h, de[0], de[1], de[2], de[3]);
          } else {
            uint2 u;
            u.x = pack_bf16x2(de[0], de[1]);
            u.y = pack_bf16x2(de[2], de[3]);
            *reinterpret_cast<uint2*>(a.de[m] + tok * H + h) = u;
          }
        }
      }
    }
    // flush the position / role gradient of this l
    __syncthreads();
    for (int h = threadIdx.x; h < H; h += kThreads) {
      const float v = acc[2 * H + h];
      if (v != 0.f) {
        atomicAdd(a.d_pos + (long long)l * H + h, v);
        atomicAdd(a.d_role + (l > 0 ? H : 0) + h, v);
      }
      acc[2 * H + h] = 0.f;
    }
    __syncthreads();
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < M; ++k)
      if (db[k] != 0.f) atomicAdd(a.d_b_att + k, db[k]);
  }
  for (int i = threadIdx.x; i < (3 + M + M * M) * H; i += kThreads) {
    const int r = i / H, h = i - r * H;
    if (r == 2) continue;
    const float v = acc[i];
    if (v == 0.f) continue;
    float* dst = r == 0 ? a.d_ln_g + h : r == 1 ? a.d_ln_b + h : r < 3 + M ? a.d_bias[r - 3] + h : a.d_w_att + (r - 3 - M) * H + h;
    atomicAdd(dst, v);
  }
}

int grid_for(long long half_warp_units, int ctas_per_sm) {  // half-warp-per-token kernels: 16 units per CTA
  long long need = (half_warp_units + (kThreads / 16) - 1) / (kThreads / 16);
  const long long cap = (long long)num_sms() * ctas_per_sm;
  if (need > cap) need = cap;
  if (need < 1) need = 1;
  return (int)need;
}

int persistent_grid(long long warp_units, int ctas_per_sm) {
  long long need = (warp_units + (kThreads / 32) - 1) / (kThreads / 32);
  const long long cap = (long long)num_sms() * ctas_per_sm;
  if (need > cap) need = cap;
  if (need < 1) need = 1;
  return (int)need;
}

// CTAs per SM the occupancy calculator allows for `kern` at `smem` bytes (after raising its dynamic shared-memory
// limit once per device); at least 1
template <typename K>
int resident_ctas(K kern, size_t smem, unsigned long long& cfg_mask) {
  if (first_use_on_device(cfg_mask)) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) return -1;
  }
  int n = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, kThreads, smem) != cudaSuccess) return -1;
  return n < 1 ? 1 : n;
}

template <int M>
int fwd_m(const pmgt_embed_multi_args* a, cudaStream_t st) {
  const long long T = a->rows * a->L;
  if (a->H == 128) {
    const size_t smem = (size_t)M * M * 128 * sizeof(float);
    static unsigned long long cfg = 0;
    const int occ = resident_ctas(embed_multi_fwd128_kernel<M>, smem, cfg);
    PMGT_REQUIRE(occ > 0, "pmgt_embed_multi_fwd: kernel configuration failed");
    embed_multi_fwd128_kernel<M><<<grid_for(T, occ < 4 ? occ : 4), kThreads, smem, st>>>(*a);
  } else {
    const int grid = persistent_grid(T, 8);
    if (a->H <= 128) embed_multi_fwd_kernel<M, 1><<<grid, kThreads, 0, st>>>(*a);
    else if (a->H <= 256) embed_multi_fwd_kernel<M, 2><<<grid, kThreads, 0, st>>>(*a);
    else if (a->H <= 512) embed_multi_fwd_kernel<M, 4><<<grid, kThreads, 0, st>>>(*a);
    else if (a->H <= 768) embed_multi_fwd_kernel<M, 6><<<grid, kThreads, 0, st>>>(*a);
    else embed_multi_fwd_kernel<M, 8><<<grid, kThreads, 0, st>>>(*a);
  }
  PMGT_LAUNCH_CHECK();
  return PMGT_OK;
}

template <int M, int G>
int bwd_generic(const pmgt_embed_multi_args* a, cudaStream_t st) {
  const size_t smem = (size_t)(3 + M + M * M) * a->H * sizeof(float);
  static unsigned long long cfg = 0;
  const int occ = resident_ctas(embed_multi_bwd_kernel<M, G>, smem, cfg);
  PMGT_REQUIRE(occ > 0, "pmgt_embed_multi_bwd: kernel configuration failed");
  embed_multi_bwd_kernel<M, G><<<persistent_grid(a->rows, occ < 2 ? occ : 2), kThreads, smem, st>>>(*a);
  PMGT_LAUNCH_CHECK();
  return PMGT_OK;
}

template <int M>
int bwd_m(const pmgt_embed_multi_args* a, cudaStream_t st) {
  if (a->H == 128 && bwd128_smem<M>(a->L) <= 227 * 1024) {
    const size_t smem = bwd128_smem<M>(a->L);
    static unsigned long long cfg_t = 0, cfg_d = 0;
    const int occ = a->row_idx ? resident_ctas(embed_multi_bwd128_kernel<M, true>, smem, cfg_t)
                               : resident_ctas(embed_multi_bwd128_kernel<M, false>, smem, cfg_d);
    PMGT_REQUIRE(occ > 0, "pmgt_embed_multi_bwd: kernel configuration failed");
    const int grid = grid_for(a->rows, occ < 2 ? occ : 2);
    if (a->row_idx)
      embed_multi_bwd128_kernel<M, true><<<grid, kThreads, smem, st>>>(*a);
    else
      embed_multi_bwd128_kernel<M, false><<<grid, kThreads, smem, st>>>(*a);
    PMGT_LAUNCH_CHECK();
    return PMGT_OK;
  }
  if (a->H <= 128) return bwd_generic<M, 1>(a, st);
  if (a->H <= 256) return bwd_generic<M, 2>(a, st);
  if (a->H <= 512) return bwd_generic<M, 4>(a, st);
  if (a->H <= 768) return bwd_generic<M, 6>(a, st);
  return bwd_generic<M, 8>(a, st);
}

// the two-modality argument block of the same call (M = 2 runs the kernels of pmgt_embed_fuse_fwd / _bwd)
pmgt_embed_args to_pair(const pmgt_embed_multi_args* m) {
  pmgt_embed_args p = {};
  p.rows = m->rows; p.L = m->L; p.H = m->H;
  p.ev = m->e[0]; p.et = m->e[1];
  p.w_att = m->w_att; p.b_att = m->b_att; p.pos = m->pos; p.role = m->role;
  p.ln_g = m->ln_g; p.ln_b = m->ln_b; p.ln_eps = m->ln_eps;
  p.dropout_p = m->dropout_p; p.dropout_seed = m->dropout_seed; p.dropout_site = m->dropout_site;
  p.x_out = m->x_out;
  p.dx = m->dx;
  p.dev = m->de[0]; p.det = m->de[1];
  p.d_w_att = m->d_w_att; p.d_b_att = m->d_b_att; p.d_pos = m->d_pos; p.d_role = m->d_role;
  p.d_ln_g = m->d_ln_g; p.d_ln_b = m->d_ln_b;
  p.d_bias_v = m->d_bias[0]; p.d_bias_t = m->d_bias[1];
  p.dx_b = m->dx_b;
  p.row_idx = m->row_idx; p.dev_acc = m->de_acc[0]; p.det_acc = m->de_acc[1]; p.skip_row0 = m->skip_row0;
  return p;
}

bool misaligned(const void* p) { return ((uintptr_t)p & 15) != 0; }

// checks shared by forward and backward for n_mod != 2
int check_common(const pmgt_embed_multi_args* a, const char* fn) {
  PMGT_REQUIRE(a->w_att && a->b_att && a->pos && a->role && a->ln_g && a->ln_b, "%s: null argument", fn);
  for (int m = 0; m < a->n_mod; ++m) PMGT_REQUIRE(a->e[m], "%s: null argument e[%d]", fn, m);
  PMGT_REQUIRE(a->H % 8 == 0 && a->H >= 8 && a->H <= 1024, "%s: H must be a multiple of 8 in [8,1024]", fn);
  PMGT_REQUIRE(a->L >= 1 && a->rows >= 0, "%s: bad sizes", fn);
  bool bad = misaligned(a->w_att) || misaligned(a->pos) || misaligned(a->role) || misaligned(a->ln_g) ||
             misaligned(a->ln_b) || misaligned(a->x_out) || misaligned(a->dx) || misaligned(a->dx_b);
  for (int m = 0; m < a->n_mod; ++m)
    bad = bad || misaligned(a->e[m]) || misaligned(a->de[m]) || misaligned(a->de_acc[m]);
  PMGT_REQUIRE(!bad, "%s: every matrix must be 16-byte aligned", fn);
  return PMGT_OK;
}

}  // namespace
}  // namespace pmgt

using namespace pmgt;

extern "C" {

int pmgt_embed_multi_fwd(const pmgt_embed_multi_args* a, void* stream) {
  PMGT_REQUIRE(a, "pmgt_embed_multi_fwd: null argument");
  PMGT_REQUIRE(a->n_mod >= 1 && a->n_mod <= PMGT_MAX_MODALITIES, "pmgt_embed_multi_fwd: n_mod must be in [1,%d]",
               PMGT_MAX_MODALITIES);
  if (a->n_mod == 2) {
    const pmgt_embed_args p = to_pair(a);
    return pmgt_embed_fuse_fwd(&p, stream);
  }
  const int rc = check_common(a, "pmgt_embed_multi_fwd");
  if (rc != PMGT_OK) return rc;
  PMGT_REQUIRE(a->x_out, "pmgt_embed_multi_fwd: null argument x_out");
  if (a->rows == 0) return PMGT_OK;
  const cudaStream_t st = (cudaStream_t)stream;
  return a->n_mod == 1 ? fwd_m<1>(a, st) : a->n_mod == 3 ? fwd_m<3>(a, st) : fwd_m<4>(a, st);
}

int pmgt_embed_multi_bwd(const pmgt_embed_multi_args* a, void* stream) {
  PMGT_REQUIRE(a, "pmgt_embed_multi_bwd: null argument");
  PMGT_REQUIRE(a->n_mod >= 1 && a->n_mod <= PMGT_MAX_MODALITIES, "pmgt_embed_multi_bwd: n_mod must be in [1,%d]",
               PMGT_MAX_MODALITIES);
  if (a->n_mod == 2) {
    const pmgt_embed_args p = to_pair(a);
    return pmgt_embed_fuse_bwd(&p, stream);
  }
  const int rc = check_common(a, "pmgt_embed_multi_bwd");
  if (rc != PMGT_OK) return rc;
  PMGT_REQUIRE(a->dx && a->d_w_att && a->d_b_att && a->d_pos && a->d_role && a->d_ln_g && a->d_ln_b,
               "pmgt_embed_multi_bwd: null argument");
  for (int m = 0; m < a->n_mod; ++m)
    PMGT_REQUIRE(a->d_bias[m] && (a->row_idx ? a->de_acc[m] != nullptr : a->de[m] != nullptr),
                 "pmgt_embed_multi_bwd: null gradient output of modality %d", m);
  if (a->rows == 0) return PMGT_OK;
  const cudaStream_t st = (cudaStream_t)stream;
  return a->n_mod == 1 ? bwd_m<1>(a, st) : a->n_mod == 3 ? bwd_m<3>(a, st) : bwd_m<4>(a, st);
}

}  // extern "C"
