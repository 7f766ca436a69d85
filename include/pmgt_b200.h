/*
 * pmgt_b200.h -- C ABI of libpmgt_b200.so: the B200 (sm_100a) implementation of
 * the PMGT pre-training hot path (uoo723/PMGT).
 *
 * The reference is pure Python and has no FFI of its own; the boundary a
 * maintainer binds is therefore this header, loaded with ctypes from the
 * host-side mirror of the reference's Python API (pmgt_b200/*.py).  Every entry
 * point cites the reference code it replaces (paths relative to the reference
 * repository root).
 *
 * Conventions
 *  - plain C: raw pointers, explicit sizes, no torch types;
 *  - every pointer is a DEVICE pointer unless its name ends in `_host`;
 *  - the caller owns every buffer; the library allocates nothing persistent
 *    except the opaque pmgt_graph handle (and small per-device scratch);
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and
 *    no entry point synchronises the device unless stated;
 *  - return value: 0 on success, negative pmgt_status on failure, and
 *    pmgt_last_error() then describes the failure (thread-local);
 *  - bf16 buffers are `uint16_t` bit patterns (torch.bfloat16 storage);
 *  - there is NO CPU fallback: without a CUDA device every compute entry point
 *    fails with PMGT_ERR_CUDA.
 */
#ifndef PMGT_B200_H_
#define PMGT_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum pmgt_status {
  PMGT_OK = 0,
  PMGT_ERR_INVALID = -1, /* bad argument (shape / alignment / range)            */
  PMGT_ERR_CUDA = -2,    /* CUDA runtime / driver error or no device            */
  PMGT_ERR_UNSUPPORTED = -3
} pmgt_status;

/* ABI version of this header; bumped on any signature change. */
#define PMGT_B200_ABI_VERSION 14
int pmgt_abi_version(void);
const char* pmgt_last_error(void);

/*
 * Programmatic dependent launch of the encoder's kernel chain (token-tile GEMMs, dW, LayerNorm backward, attention
 * core): on by default (environment PMGT_PDL=0 turns it off at load time).  Returns the previous setting.  Timing
 * single kernels with events is only meaningful with it off, because a dependent kernel's prologue then overlaps
 * its predecessor's tail.
 */
int pmgt_set_pdl(int enabled);

/*
 * Alternating traversal order of the encoder's persistent kernels (token-tile GEMMs, LayerNorm backward, attention
 * core): consecutive launches walk the token tiles in opposite directions, so each kernel starts on the rows its
 * predecessor wrote last, which are still in L2.  Results do not depend on the order.  On by default
 * (PMGT_ALTERNATE=0 at load time turns it off); returns the previous setting.
 */
int pmgt_set_alternate_order(int enabled);

/* ------------------------------------------------------------------------ */
/* Item graph (CSR)                                                          */
/* ------------------------------------------------------------------------ */
/*
 * Replaces the weighted nx.Graph the reference keeps on the host
 * (pmgt/pmgt/trainer.py:34-41, used at pmgt/pmgt/datasets.py:27-32,167-180).
 * Node-id space is the reference's: 0 = <pad>, 1 = <mask>, real nodes
 * 2..num_nodes+1 (datasets.py:96-102).  indptr has num_nodes+3 entries and is
 * indexed by node id (rows 0 and 1 are empty).  indices keeps the adjacency
 * INSERTION order of the nx.Graph so that inverse-CDF positions mean the same
 * neighbours as in the reference.  cdf[e] is the running softmax CDF of the
 * edge weights of the row e belongs to (datasets.py:27-29 + numpy's legacy
 * RandomState.choice: p.cumsum(), normalised, last entry forced to 1).
 * The arrays are COPIED to the device; the host buffers may be freed.
 */
typedef struct pmgt_graph pmgt_graph;

int pmgt_graph_create(pmgt_graph** out, int device, int64_t num_nodes, int64_t num_edges_directed,
                      const int64_t* indptr_host, const int32_t* indices_host,
                      const float* cdf_host);
/*
 * The same handle built ON the device from device-resident arrays: `indptr_dev` / `indices_dev` as above (rows already
 * in adjacency insertion order) and the fp64 edge weights; the per-row softmax CDF (fp64 math, stored fp32, last entry 1)
 * and the sampler's lookup structures are computed by kernels (replaces the networkx ingestion of
 * pmgt/pmgt/trainer.py:34-41 for graphs whose host-side construction is the start-up bottleneck).  Synchronises `stream`.
 */
int pmgt_graph_create_device(pmgt_graph** out, int device, int64_t num_nodes, int64_t num_edges_directed,
                             const int64_t* indptr_dev, const int32_t* indices_dev, const double* weights_dev,
                             void* stream);
int pmgt_graph_destroy(pmgt_graph* g);
int64_t pmgt_graph_num_nodes(const pmgt_graph* g);
int64_t pmgt_graph_num_edges(const pmgt_graph* g);
/* device pointers of the resident CSR (for tests / roofline byte accounting) */
const int64_t* pmgt_graph_indptr(const pmgt_graph* g);
const int32_t* pmgt_graph_indices(const pmgt_graph* g);
const float* pmgt_graph_cdf(const pmgt_graph* g);

/* ------------------------------------------------------------------------ */
/* K1  MCNSampling: context sampler + pair selection (Philox4x32-10)          */
/* ------------------------------------------------------------------------ */
/*
 * pmgt_sample_contexts replaces _sample_context_neigh + _get_attention_mask +
 * get_input_tensor (pmgt/pmgt/datasets.py:14-79) for a whole batch of roots.
 *
 *   roots[n]     node id of the n-th context's target node
 *   ctx_keys[n]  64-bit RNG sub-stream id of that context (counter words 2,3)
 *   hops_host    hop sampling sizes (depth entries, host memory), e.g. {16,8,4}
 *   out_ids      [n_ctx][max_ctx+1] int64: root, then the top-`max_ctx`
 *                neighbours by score (frequency x hop weight, ties broken by
 *                first appearance), right-padded with 0
 *   out_mask     [n_ctx][max_ctx+1] float32: 1 for root + real neighbours
 *   out_visited_deg (optional, may be NULL) [n_ctx] int64: sum of the degrees
 *                of every row the context visited (roofline byte accounting)
 *
 * Draw d of a context uses Philox counter (d/4, PMGT_STREAM_CTX, key_lo, key_hi)
 * word d%4 under key (seed_lo, seed_hi); u = (word >> 8) * 2^-24; the neighbour
 * is row[upper_bound(cdf_row, u)].  d enumerates hop 1 first, then hop 2 in
 * parent order, ...  oracle/philox_sampler.c replays exactly this on the CPU.
 */
#define PMGT_STREAM_CTX 0u
#define PMGT_STREAM_POS 1u
#define PMGT_STREAM_NEG 2u
#define PMGT_MAX_NEG_ATTEMPTS 64

int pmgt_sample_contexts(const pmgt_graph* g, const int64_t* roots, const int64_t* ctx_keys,
                         int64_t n_ctx, const int32_t* hops_host, int depth, int max_ctx,
                         uint64_t seed, int64_t* out_ids, float* out_mask,
                         int64_t* out_visited_deg, void* stream);

/*
 * pmgt_sample_pairs replaces PMGTDataset._sample_neigh / _sample_neg /
 * _get_label_tensor (pmgt/pmgt/datasets.py:125-146,159,167-183).
 * For target b: n_pos = min(max_pos, deg) distinct neighbours (partial
 * Fisher-Yates on stream PMGT_STREAM_POS), then n_neg = max(min_neg,
 * max_total - n_pos) uniform node ids in [2, N+2) rejected while adjacent to
 * the target (stream PMGT_STREAM_NEG, at most PMGT_MAX_NEG_ATTEMPTS attempts
 * per negative).  Rows are written at a fixed stride `pair_stride`
 * (>= max_pos + max(min_neg, max_total)); unused slots are 0.
 *   out_pairs [n_tgt][pair_stride] int64, out_labels [n_tgt][pair_stride] f32,
 *   out_num_pairs [n_tgt] int64.
 */
int pmgt_sample_pairs(const pmgt_graph* g, const int64_t* targets, const int64_t* tgt_keys,
                      int64_t n_tgt, int max_pos, int min_neg, int max_total, int pair_stride,
                      uint64_t seed, int64_t* out_pairs, float* out_labels,
                      int64_t* out_num_pairs, void* stream);

/* ------------------------------------------------------------------------ */
/* GEMM on tcgen05 tensor cores (building block of K2 / K3 / K5)              */
/* ------------------------------------------------------------------------ */
/*
 * D[M,N] (+)= op(A)[M,K] * op(B)[K,N], bf16 operands, fp32 accumulation in
 * TMEM, TMA- or cp.async-gather-staged operands.  Replaces the cuBLAS GEMMs
 * behind nn.Linear in PMGTEmbeddings / PMGTSelfAttention / BertSelfOutput /
 * BertIntermediate / BertOutput / PMGTNodeConstructLoss
 * (pmgt/pmgt/modeling_pmgt.py:195-198,429-433,371,322-325,566-569) and their
 * autograd backward GEMMs.
 *
 * Operand storage ("major"):
 *   a_mn = 0: A stored row-major [M][K] (lda = row pitch in elements)
 *   a_mn = 1: A stored row-major [K][M]  (i.e. A^T is what is in memory)
 *   b_mn = 0: B stored row-major [N][K]  (nn.Linear weight layout)
 *   b_mn = 1: B stored row-major [K][N]
 * Gather: if a_rows != NULL the stored rows of A (a_mn=0: the M rows; a_mn=1:
 * the K rows) are fetched through the index vector, row r of the operand is
 * a + a_rows[r]*lda.  Same for b_rows.  Indices are int64; index < 0 or row
 * beyond the logical extent reads as zeros.
 *
 * Epilogue (flags in `epi`): v = acc * alpha; +bias[n]; GELU(erf) with the
 * pre-activation stored to `aux`; or multiply by gelu'(aux[m][n]); + addend;
 * store as bf16 (out_bf16), fp32 (out_f32) or atomically accumulate into fp32
 * (PMGT_EPI_ATOMIC, used with split_k > 1 for weight gradients).
 */
#define PMGT_EPI_BIAS 1u
#define PMGT_EPI_GELU 2u      /* out = gelu(v); aux_out (bf16) = v            */
#define PMGT_EPI_GELU_BWD 4u  /* out = v * gelu'(aux_in[m][n])                */
#define PMGT_EPI_ADDEND 8u    /* out += addend[m][n] (bf16)                   */
#define PMGT_EPI_OUT_F32 16u  /* store fp32 instead of bf16                   */
#define PMGT_EPI_ATOMIC 32u   /* fp32 atomicAdd into out (implies OUT_F32)    */

typedef struct pmgt_gemm_args {
  int64_t M, N, K;
  const uint16_t* a; int64_t lda; int a_mn; const int64_t* a_rows; int64_t a_src_rows;
  const uint16_t* b; int64_t ldb; int b_mn; const int64_t* b_rows; int64_t b_src_rows;
  void* out; int64_t ldo;
  const float* bias;            /* [N] fp32                                   */
  const uint16_t* addend; int64_t ld_addend;
  uint16_t* aux; int64_t ld_aux; /* GELU: written; GELU_BWD: read             */
  float alpha;
  uint32_t epi;
  int split_k;                  /* >= 1                                        */
} pmgt_gemm_args;

int pmgt_gemm_bf16(const pmgt_gemm_args* args, void* stream);

/* ------------------------------------------------------------------------ */
/* K2  multimodal feature path                                               */
/* ------------------------------------------------------------------------ */
/*
 * The gather + per-modality projection GEMMs go through pmgt_gemm_bf16 with
 * a_rows = node ids (replaces get_input_feat_embeds, pmgt/pmgt/utils.py:43-50,
 * and feat_linear, modeling_pmgt.py:195-198).  pmgt_embed_fuse_fwd/bwd are the
 * rest of PMGTEmbeddings.forward (modeling_pmgt.py:199-208): modality
 * attention softmax(Linear(tanh([e_v;e_t]))), weighted sum, + position + role
 * embedding, LayerNorm, dropout.
 *   ev, et      [T][H] bf16 projected features (T = rows * L tokens)
 *   w_att [2][2H], b_att [2], pos [max_pos][H], role [2][H], ln_g/ln_b [H] fp32
 *   x_out       [T][H] bf16
 * Backward recomputes the forward from ev/et and produces dev/det (bf16) and
 * fp32 gradients ACCUMULATED (atomicAdd) into d_w_att, d_b_att, d_pos, d_role,
 * d_ln_g, d_ln_b, d_bias_v, d_bias_t (column sums of dev/det).
 */
typedef struct pmgt_embed_args {
  int64_t rows; int L; int H;
  const uint16_t* ev; const uint16_t* et;
  const float* w_att; const float* b_att; const float* pos; const float* role;
  const float* ln_g; const float* ln_b; float ln_eps;
  float dropout_p; uint64_t dropout_seed; uint32_t dropout_site;
  uint16_t* x_out;            /* fwd */
  const uint16_t* dx;         /* bwd: [T][H] bf16 */
  uint16_t* dev; uint16_t* det;
  float* d_w_att; float* d_b_att; float* d_pos; float* d_role; float* d_ln_g; float* d_ln_b;
  float* d_bias_v; float* d_bias_t;
  const uint16_t* dx_b;       /* bwd, optional: second gradient term, summed with dx */
  /* Projected-table mode (small graphs: project every table row once, gather the PROJECTED rows): when
   * `row_idx` != NULL, ev / et are [table_rows][H] and token t reads row row_idx[t]; backward then accumulates the
   * per-row gradients into dev_acc / det_acc ([table_rows][H] fp32, red.add) instead of writing dev / det.
   * skip_row0: row 0 (<pad>) of the feature tables is all zero, so its gradient rows are never used. */
  const int64_t* row_idx; float* dev_acc; float* det_acc; int skip_row0;
} pmgt_embed_args;

int pmgt_embed_fuse_fwd(const pmgt_embed_args* a, void* stream);
int pmgt_embed_fuse_bwd(const pmgt_embed_args* a, void* stream);

/*
 * The same fusion for any number of feature modalities M = n_mod in [1, PMGT_MAX_MODALITIES] (the reference's
 * PMGTEmbeddings takes one feat_linear per entry of feat_hidden_sizes and a Linear(M*H -> M) modality attention):
 * pmgt_embed_args with every per-modality pair turned into an array indexed by modality.
 *   e[m]        [T][H] (or [table_rows][H] with row_idx) bf16 projected features of modality m
 *   w_att [M][M*H], b_att [M] fp32; d_w_att / d_b_att the same shapes
 *   de[m]       bwd: [T][H] bf16 gradient of e[m];  de_acc[m]: projected-table mode, [table_rows][H] fp32, red.add
 *   d_bias[m]   bwd: [H] fp32 column sums of de[m], accumulated
 * Entries m >= n_mod are ignored.  n_mod == 2 runs pmgt_embed_fuse_fwd / _bwd with the equivalent pmgt_embed_args.
 * Otherwise H is a multiple of 8 in [8, 1024] and every matrix is 16-byte aligned.  The dropout mask is the one of
 * pmgt_embed_fuse_fwd (element tok * H + h under dropout_seed / dropout_site), whatever M is.  At n_mod == 1 the
 * softmax weight is exactly 1 and d_w_att / d_b_att receive exact zeros.
 */
#define PMGT_MAX_MODALITIES 4

typedef struct pmgt_embed_multi_args {
  int64_t rows; int L; int H; int n_mod;
  const uint16_t* e[PMGT_MAX_MODALITIES];
  const float* w_att; const float* b_att; const float* pos; const float* role;
  const float* ln_g; const float* ln_b; float ln_eps;
  float dropout_p; uint64_t dropout_seed; uint32_t dropout_site;
  uint16_t* x_out;            /* fwd */
  const uint16_t* dx;         /* bwd: [T][H] bf16 */
  uint16_t* de[PMGT_MAX_MODALITIES];
  float* d_w_att; float* d_b_att; float* d_pos; float* d_role; float* d_ln_g; float* d_ln_b;
  float* d_bias[PMGT_MAX_MODALITIES];
  const uint16_t* dx_b;       /* bwd, optional: second gradient term, summed with dx */
  const int64_t* row_idx; float* de_acc[PMGT_MAX_MODALITIES]; int skip_row0;
} pmgt_embed_multi_args;

int pmgt_embed_multi_fwd(const pmgt_embed_multi_args* a, void* stream);
int pmgt_embed_multi_bwd(const pmgt_embed_multi_args* a, void* stream);

/*
 * Gather-fused feature projection for large graphs, H = 128 (csrc/gather_proj.cu): persistent tcgen05 kernels whose
 * shared-memory ring belongs to the gathered operand (~160 KB in flight per SM); table rows are fetched by TMA
 * tile::gather4 (environment PMGT_GATHER_TMA: bit 0 forward, bit 1 weight gradient; 0 selects the 16-byte cp.async
 * gather kept for comparison; default 3).  Same contract as pmgt_gemm_bf16 with a_rows / b_rows (get_input_feat_embeds, pmgt/pmgt/utils.py:43-50,
 * + feat_linear, pmgt/pmgt/modeling_pmgt.py:195-198):
 *   pmgt_gather_proj_fwd  out[T][128] (bf16) = table[rows[t]][0:K] . w[128][K]^T + bias
 *   pmgt_gather_proj_dw   dw[128][K] (fp32) += dy[T][128]^T . table[rows[t]][0:K]
 * rows[t] outside [0, table_rows) reads as a zero row.  pmgt_gather_proj_supported(N, K): N == 128, K a multiple of
 * 128 and of 256, 384 or 512.
 */
typedef struct pmgt_gather_proj_args {
  int64_t T, K;
  const uint16_t* table; int64_t ld; int64_t table_rows;   /* [table_rows][K] bf16, row pitch ld elements */
  const int64_t* rows;                                      /* [T] node ids */
  const uint16_t* w; int64_t ldw; const float* bias;        /* fwd: [128][K] bf16, [128] fp32 (may be NULL) */
  uint16_t* out; int64_t ldo;                               /* fwd: [T][128] bf16, 32-byte aligned rows */
  const uint16_t* dy; int64_t ld_dy;                        /* dw: [T][128] bf16 */
  float* dw; int64_t ld_dw;                                 /* dw: [128][K] fp32, accumulated */
} pmgt_gather_proj_args;

int pmgt_gather_proj_supported(int64_t N, int64_t K);
int pmgt_gather_proj_fwd(const pmgt_gather_proj_args* a, void* stream);
int pmgt_gather_proj_dw(const pmgt_gather_proj_args* a, void* stream);

/* ------------------------------------------------------------------------ */
/* K3  encoder layer pieces                                                  */
/* ------------------------------------------------------------------------ */
/*
 * Dual-softmax "diversity promoting" attention core of PMGTSelfAttention
 * (modeling_pmgt.py:435-526), per (sequence, head):
 *   S1 = 1 - C C^T / (|C||C|^T) + I + mask ; P1 = dropout(softmax(S1))
 *   S2 = Q K^T / sqrt(dh) + mask           ; P2 = dropout(softmax(S2))
 *   ctx = (beta P1 + (1-beta) P2) V
 * qkvc is [T][4H] bf16 with column blocks [Q | K | V | C]; mask is the
 * reference's 0/1 attention mask [rows][L] fp32 (the additive -10000 key mask
 * of transformers 4.11.2 get_extended_attention_mask is applied inside).
 * Backward recomputes P1/P2 and writes dqkvc [T][4H] bf16 and accumulates the
 * bias gradient d_bias_qkvc [4H] (fp32 atomicAdd) when non-NULL.
 * qkvc, ctx (forward), dctx and dqkvc (backward) must be 16-byte aligned;
 * otherwise the call returns PMGT_ERR_INVALID.  1 <= L <= 128, even head size.
 * The kernel, and with it the dropout stream, depends only on the shape
 * (L, H, heads, rows * heads), so a forward / backward pair with the same
 * dropout_seed and dropout_site always sees the same mask.
 */
typedef struct pmgt_attn_args {
  int64_t rows; int L; int H; int heads; float beta;
  const uint16_t* qkvc; const float* mask;
  float dropout_p; uint64_t dropout_seed; uint32_t dropout_site;
  uint16_t* ctx;               /* fwd out [T][H] */
  const uint16_t* dctx;        /* bwd in  [T][H] */
  uint16_t* dqkvc;             /* bwd out [T][4H] */
  float* d_bias_qkvc;          /* bwd out [4H], accumulated */
} pmgt_attn_args;

int pmgt_attn_core_fwd(const pmgt_attn_args* a, void* stream);
int pmgt_attn_core_bwd(const pmgt_attn_args* a, void* stream);

/*
 * Attention maps: maps [rows][heads][L][L] fp32 receives, per (sequence, head),
 * the matrix pmgt_attn_core_fwd multiplies V with for the same arguments,
 *   A = beta * dropout(P1) + (1 - beta) * dropout(P2),
 * with the very dropout mask the core applies for that shape, seed and site
 * (ctx = A V).  Reads qkvc, mask, beta, dropout_*, rows, L, H and heads; ctx,
 * dctx, dqkvc and d_bias_qkvc are ignored.  qkvc and maps must be 16-byte
 * aligned; the shape limits are those of pmgt_attn_core_fwd.  Every check is
 * made before any CUDA call.
 */
int pmgt_attn_maps_fwd(const pmgt_attn_args* a, float* maps, void* stream);

/*
 * y = LayerNorm(dropout(o) + res) -- BertSelfOutput / BertOutput after their
 * dense layer (transformers BertSelfOutput/BertOutput, called at
 * modeling_pmgt.py:371,324).  o already contains the dense bias.
 * Backward: given dy, recomputes z = dropout(o)+res and writes dz (bf16, the
 * gradient wrt `res`; the gradient wrt `o` is dz with the dropout mask applied,
 * written to d_o when dropout_p > 0, else d_o may alias dz) and accumulates
 * d_g, d_b (LayerNorm) and d_bias (column sums of d_o) in fp32.
 */
typedef struct pmgt_resln_args {
  int64_t T; int H;
  const uint16_t* o; const uint16_t* res;
  const float* ln_g; const float* ln_b; float ln_eps;
  float dropout_p; uint64_t dropout_seed; uint32_t dropout_site;
  uint16_t* y; float* y_f32;   /* fwd out; y_f32 optional */
  const uint16_t* dy; const float* dy_f32; /* bwd in: dy (bf16) and/or dy_f32 are summed */
  uint16_t* dz; uint16_t* d_o;
  float* d_g; float* d_b; float* d_bias;
} pmgt_resln_args;

int pmgt_res_ln_fwd(const pmgt_resln_args* a, void* stream);
int pmgt_res_ln_bwd(const pmgt_resln_args* a, void* stream);

/*
 * Persistent tcgen05 "token-tile" kernels: the fast path of the nn.Linear layers of the encoder when every
 * dimension is a multiple of 128 and the weight fits in shared memory (the default PMGT encoder, H = I = 128;
 * modeling_pmgt.py:429-433,371,322-325 forward, and their autograd backward).  A CTA per SM loops over tiles of
 * 128 tokens; activations arrive by TMA, weights stay resident, accumulators live in TMEM, results leave by
 * TMA store.  Shapes outside pmgt_linear_tile_supported() go through pmgt_gemm_bf16.
 *
 *   epi PMGT_LT_BIAS      out = x w^T + bias                                   (w_mn = 0)
 *       PMGT_LT_GELU      aux_out = x w^T + bias ; out = gelu_erf(aux_out)      (w_mn = 0; BertIntermediate)
 *       PMGT_LT_RES_LN    z = dropout(x w^T + bias) + e_in ; aux_out = z ; out = LayerNorm(z)
 *                         (w_mn = 0; BertSelfOutput / BertOutput; N == 128; out_f32 optional fp32 copy)
 *       PMGT_LT_PLAIN     out = x w                                             (w_mn = 1; dX of a Linear)
 *       PMGT_LT_GELU_BWD  out = (x w) * gelu_erf'(e_in)                          (w_mn = 1)
 *   w_mn = 0: w is [N][K] (nn.Linear weight, y = x w^T); w_mn = 1: w is [K][N] (dx = dy w, same storage).
 *   Dropout element index = token * N + column (the same stream pmgt_ln_bwd regenerates).
 *   With programmatic dependent launch on (default, see pmgt_set_pdl) the weight tiles are fetched while the preceding
 *   kernel of the stream may still be running: `w` must not be written by the kernels launched immediately before
 *   this call (activations x / e_in are read only after the predecessor has completed).
 */
#define PMGT_LT_BIAS 0
#define PMGT_LT_GELU 1
#define PMGT_LT_RES_LN 2
#define PMGT_LT_PLAIN 3
#define PMGT_LT_GELU_BWD 4

typedef struct pmgt_linear_tile_args {
  int64_t T; int K; int N;
  const uint16_t* x; int64_t ldx;          /* [T][K] bf16 */
  const uint16_t* w; int64_t ldw; int w_mn;
  int epi;
  const float* bias;                        /* [N] fp32 */
  uint16_t* out; int64_t ldo;               /* [T][N] bf16 */
  uint16_t* aux_out; int64_t ld_aux_out;    /* GELU: pre-activation; RES_LN: z */
  const uint16_t* e_in; int64_t ld_e;       /* RES_LN: residual; GELU_BWD: pre-activation */
  const float* ln_g; const float* ln_b; float ln_eps;
  float dropout_p; uint64_t dropout_seed; uint32_t dropout_site;
  float* out_f32;                           /* RES_LN only, optional, [T][N] fp32 */
  /* Fused weight gradient of the SAME Linear (dX calls only: PLAIN / GELU_BWD with w_mn = 1, K = N = 128): when dw is
   * non-NULL the call also accumulates dw[K][ld_dw] += x^T dw_x  (x = the dY operand of this call, dw_x = the
   * Linear's forward input, [T][128] bf16) and dbias[K] += column sums of x (optional).  One pass over dY serves
   * dX, dW and dbias. */
  const uint16_t* dw_x; int64_t ld_dw_x;
  float* dw; int64_t ld_dw; float* dbias;
} pmgt_linear_tile_args;

int pmgt_linear_tile_supported(int64_t K, int64_t N, int w_mn, int epi);
int pmgt_linear_tile(const pmgt_linear_tile_args* a, void* stream);

/*
 * dw[N][K] += dy^T x and dbias[N] += column sums of dy (fp32, accumulated): the weight / bias gradient of a
 * Linear.  Accumulators stay in TMEM over all token tiles of a CTA and are flushed once.  K == 128,
 * N in {128, 512}; other shapes: pmgt_gemm_bf16 (split-K) + pmgt_colsum_bf16.
 */
typedef struct pmgt_dw_tile_args {
  int64_t T; int N; int K;
  const uint16_t* dy; int64_t ld_dy;        /* [T][N] bf16 */
  const uint16_t* x; int64_t ldx;           /* [T][K] bf16 */
  float* dw; int64_t ld_dw;                 /* [N][K] fp32 */
  float* dbias;                             /* [N] fp32, may be NULL */
} pmgt_dw_tile_args;

int pmgt_dw_tile_supported(int64_t N, int64_t K);
int pmgt_dw_tile(const pmgt_dw_tile_args* a, void* stream);
/* n independent problems of one (N, K) shape in one launch: the CTAs are dealt round-robin to the problems, so every dw
 * receives ~SMs / n partial sums instead of SMs and the fixed cost of the accumulator flush is paid once (used for the
 * Q/K/V/C weight gradients of all encoder layers, deferred to the end of the backward pass). */
int pmgt_dw_tile_batch(const pmgt_dw_tile_args* a, int n, void* stream);

/*
 * Fused post-attention blocks of one encoder layer, H = I = 128 (one persistent tcgen05 kernel per call):
 *   ffn = 0  BertSelfOutput as composed by PMGTAttention (pmgt/pmgt/modeling_pmgt.py:358-375):
 *              out = LayerNorm(dropout(in w2^T + b2) + res)
 *   ffn = 1  BertIntermediate + BertOutput as composed by PMGTLayer.feed_forward_chunk (modeling_pmgt.py:296-325):
 *              out = LayerNorm(dropout(gelu(in w1^T + b1) w2^T + b2) + in)
 * pmgt_block_fwd  writes out (optional fp32 copy out_f32) and, when xhat != NULL, what pmgt_block_bwd reads back:
 *                 xhat (normalised pre-affine LayerNorm value, bf16), rstd (fp32 per row) and -- ffn -- h = gelu(h_pre)
 *                 and gp = gelu'(h_pre).  The dropout mask is regenerated from (seed, site) in the backward call.
 * pmgt_block_bwd  dy (+ dy_b) = d(loss)/d(out).  dx = d(loss)/d(in): for ffn = 1 it includes the residual branch
 *                 (in IS the residual); for ffn = 0 the residual-branch gradient is written to dz instead.
 *                 dw1, dw2, db1, db2, d_ln_g, d_ln_b are ACCUMULATED (fp32).
 * All [T][128] bf16 matrices: 32-byte aligned, pitch a multiple of 16 elements.
 */
typedef struct pmgt_block_args {
  int64_t T;
  int ffn;
  const uint16_t* in; int64_t ld_in;        /* [T][128] bf16 */
  const uint16_t* res; int64_t ld_res;      /* ffn = 0: residual rows [T][128] bf16 (ffn = 1: ignored, the residual is `in`) */
  const uint16_t* w1; const float* b1;      /* ffn = 1: intermediate.dense  [128][128] bf16 contiguous, [128] fp32 */
  const uint16_t* w2; const float* b2;      /* the dense layer in front of the LayerNorm */
  const float* ln_g; const float* ln_b; float ln_eps;
  float dropout_p; uint64_t dropout_seed; uint32_t dropout_site;
  uint16_t* out; int64_t ld_out;            /* fwd: [T][128] bf16 */
  float* out_f32;                           /* fwd, optional: [T][128] fp32 contiguous */
  uint16_t* h; uint16_t* gp; uint16_t* xhat; int64_t ld_save;   /* saved activations, [T][128] bf16 each, same pitch */
  float* rstd;                              /* [T] fp32 */
  const uint16_t* dy; int64_t ld_dy;        /* bwd: [T][128] bf16 */
  const uint16_t* dy_b; int64_t ld_dy_b;    /* bwd, optional second term of the incoming gradient */
  uint16_t* dx; int64_t ld_dx;              /* bwd: [T][128] bf16 */
  uint16_t* dz; int64_t ld_dz;              /* bwd, ffn = 0: [T][128] bf16 gradient of the residual branch */
  float* dw1; float* dw2;                   /* bwd: [128][128] fp32 */
  float* db1; float* db2; float* d_ln_g; float* d_ln_b;   /* bwd: [128] fp32, each may be NULL */
} pmgt_block_args;

int pmgt_block_fwd(const pmgt_block_args* a, void* stream);
int pmgt_block_bwd(const pmgt_block_args* a, void* stream);
/* Diagnostics: `buf` = device buffer of 8 * 32 * 4 uint64 (or NULL to stop).  While set, CTA 0 of every block kernel
 * stamps clock64() at its stage boundaries ([role][tile][event]; roles: 0 MMA issuer, then the epilogue groups) --
 * tools/blk_timeline.py prints the per-stage durations. */
int pmgt_block_set_trace(void* buf);

/*
 * LayerNorm backward from the saved pre-LayerNorm input z (PMGT_LT_RES_LN's aux_out): dy = dy_a + dy_b +
 * dy_f32 (any subset), dz = gradient wrt z (and wrt the residual), d_o = dz with the dropout mask of the
 * forward re-applied (gradient wrt the dense output; may alias dz when dropout_p == 0), d_g / d_b fp32
 * accumulated.  H == 128.
 */
typedef struct pmgt_lnbwd_args {
  int64_t T; int H;
  const uint16_t* z;
  const uint16_t* dy_a; const uint16_t* dy_b; const float* dy_f32;
  const float* ln_g; float ln_eps;
  float dropout_p; uint64_t dropout_seed; uint32_t dropout_site;
  uint16_t* dz; uint16_t* d_o;
  float* d_g; float* d_b;
} pmgt_lnbwd_args;

int pmgt_ln_bwd(const pmgt_lnbwd_args* a, void* stream);

/* column sums: out[n] += sum_t x[t][n]  (bias gradients), x bf16 [T][N] */
int pmgt_colsum_bf16(const uint16_t* x, int64_t T, int64_t N, int64_t ldx, float* out, void* stream);

/* ------------------------------------------------------------------------ */
/* K4  graph-structure reconstruction loss                                   */
/* ------------------------------------------------------------------------ */
/*
 * PMGTGraphConstructLoss + the per-target loop of PMGT.forward
 * (modeling_pmgt.py:537-546, models.py:104-127) for the whole batch at once.
 *   tgt_h   [B][ld_t] fp32 : position-0 hidden state of each target row
 *   pair_h  [SP][ld_p] fp32: position-0 hidden state of each pair row
 *   pair_off[B+1] int64    : prefix sum of num_pairs
 *   labels  [SP] fp32
 * fwd: logits [SP] fp32, loss_out[0] = mean_b mean_p BCEWithLogits.
 * bwd: d_tgt / d_pair (same layout as the inputs, overwritten) scaled by
 *      *grad_out (device scalar).
 */
typedef struct pmgt_gsr_args {
  int64_t B; int64_t SP; int H;
  const float* tgt_h; int64_t ld_t; const float* pair_h; int64_t ld_p;
  const int64_t* pair_off; const float* labels;
  float* logits; float* loss_out;
  const float* grad_out; float* d_tgt; float* d_pair;
} pmgt_gsr_args;

int pmgt_gsr_fwd(const pmgt_gsr_args* a, void* stream);
int pmgt_gsr_bwd(const pmgt_gsr_args* a, void* stream);

/* ------------------------------------------------------------------------ */
/* K5  node-feature reconstruction loss                                      */
/* ------------------------------------------------------------------------ */
/*
 * MSE part of PMGTNodeConstructLoss (modeling_pmgt.py:566-569) for ONE
 * modality: proj [Mm][D] bf16 (= Linear(h_masked), produced by pmgt_gemm_bf16)
 * against rows of the frozen feature table gathered by target_ids
 * (models.py:150,159).  fwd accumulates  weight * mean((proj-tgt)^2)  into
 * loss_out[0]; bwd writes dproj = *grad_out * weight * 2/(Mm*D) * (proj-tgt).
 * Mm == 0 contributes NaN like nn.MSELoss over an empty tensor.
 */
typedef struct pmgt_nfr_args {
  int64_t Mm; int64_t D;
  const uint16_t* proj; int64_t ld_proj;
  const uint16_t* table; int64_t ld_table; const int64_t* target_ids;
  float weight;
  float* loss_out;
  const float* grad_out; uint16_t* dproj;
} pmgt_nfr_args;

int pmgt_nfr_mse_fwd(const pmgt_nfr_args* a, void* stream);
int pmgt_nfr_mse_bwd(const pmgt_nfr_args* a, void* stream);

/* ------------------------------------------------------------------------ */
/* K6  optimizer + utility                                                   */
/* ------------------------------------------------------------------------ */
/*
 * Dense branch of DenseSparseAdamW.step (pmgt/optimizers.py:256-270) over a
 * flat fp32 parameter buffer: p *= 1 - lr*wd[i]; m = b1 m + (1-b1) g;
 * v = b2 v + (1-b2) g^2; p -= (lr/bc1) * m / (sqrt(v)/sqrt(bc2) + eps).
 * `decay_mask` (uint8, per element) selects the weight-decay group
 * (base_trainer.py:35-59: no decay for names containing "bias" or
 * "LayerNorm.weight").  grad_scale multiplies g first (1/world_size after an
 * allreduce-sum, gradient clipping coefficient, ...); if grad_scale_dev is
 * non-NULL the device scalar is used instead.
 */
int pmgt_adamw_step(float* p, const float* g, float* m, float* v, const uint8_t* decay_mask,
                    int64_t n, float lr, float beta1, float beta2, float eps, float weight_decay,
                    int64_t step, float grad_scale, const float* grad_scale_dev, void* stream);

/* fp32 -> bf16 cast of a flat buffer (weights shadow / feature tables) */
int pmgt_cast_f32_bf16(const float* src, uint16_t* dst, int64_t n, void* stream);
/* sum of squares of a flat fp32 buffer accumulated into out[0] (clip_grad_norm_) */
int pmgt_sumsq_f32(const float* x, int64_t n, float* out, void* stream);
/* torch.nn.utils.clip_grad_norm_ (pmgt/base_trainer.py:314 gradient_clip_val) folded with the gradient scale:
 * out[0] = scale * min(1, max_norm / (sqrt(sumsq[0]) * scale + 1e-6)); sumsq[0] is reset to 0 for the next step */
int pmgt_clip_coef(float* sumsq, float scale, float max_norm, float* out, void* stream);
/* In-place sum of a flat fp32 vector over the ranks of one NVSwitch domain (replaces the gradient all-reduce of the
 * reference's implicit DDP, pmgt/base_trainer.py:309-322).  peer_ptrs[r] = device address of rank r's copy as mapped into
 * THIS process (symmetric memory / CUDA IPC; 16-byte aligned; peer_ptrs[rank] is the local copy).  Rank `rank` reduces
 * slice `rank` of the vector and stores the sum into every copy.  The caller brackets the call with barriers over all
 * ranks: every copy complete before it, every slice written after it.  world_size <= 8. */
int pmgt_peer_reduce_f32(const uint64_t* peer_ptrs, int world_size, int rank, int64_t n, void* stream);
/* out[r][:] = src[idx[r]][:]   (bf16 rows, D elements, D % 8 == 0) */
int pmgt_gather_rows_bf16(const uint16_t* src, int64_t ld_src, const int64_t* idx, int64_t n_rows,
                          int64_t D, uint16_t* out, int64_t ld_out, void* stream);
/* dst[idx[r]][:] = src[r][:]   (the inverse: idx unique, other rows of dst untouched) -- with pmgt_gather_rows_bf16 this
 * is how the LAST encoder layer runs its post-attention half only on the token rows whose hidden state is consumed */
int pmgt_scatter_rows_bf16(const uint16_t* src, int64_t ld_src, const int64_t* idx, int64_t n_rows, int64_t D,
                           uint16_t* dst, int64_t ld_dst, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PMGT_B200_H_ */
