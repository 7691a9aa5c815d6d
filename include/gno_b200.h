/*
 * gno_b200.h — C-ABI of the B200-native GNN aggregation path.
 *
 * This is the drop-in boundary: plain C, raw device pointers and sizes, a
 * cudaStream_t passed as void*.  No torch types.  Every buffer (inputs,
 * outputs, workspaces, plan arrays) is OWNED BY THE CALLER; the library never
 * allocates device memory and never synchronises the device, so it composes
 * with any allocator (torch's caching allocator in the Python host) and with
 * CUDA-graph capture.  All functions return 0 on success or a gno_status
 * code; gno_last_error() gives the thread-local message.
 *
 * The reference (ryienh/gnn-ops-benchmark) holds no native code: its kernels
 * live in torch-scatter 2.0.9 / torch-sparse 0.6.12 / ATen 1.11.  Each entry
 * point below names the reference call site whose work it replaces
 * (file:line relative to the reference root).
 */
#ifndef GNO_B200_H
#define GNO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GNO_ABI_VERSION 3

typedef void* gno_stream_t; /* a cudaStream_t */

typedef enum gno_status {
  GNO_OK = 0,
  GNO_ERR_INVALID = 1,     /* bad argument (shape, alignment, enum) */
  GNO_ERR_UNSUPPORTED = 2, /* valid request this build does not cover */
  GNO_ERR_CUDA = 3,        /* a CUDA runtime call or launch failed */
  GNO_ERR_WORKSPACE = 4    /* workspace pointer NULL or too small */
} gno_status;

typedef enum gno_dtype { GNO_F32 = 0, GNO_F16 = 1, GNO_BF16 = 2 } gno_dtype;

/* Reductions of torch_scatter.scatter(..., reduce=) — the five the reference
 * times: op_bm_scripts/benchmark_scatter_add.py:18, _mean.py:17, _max.py:17,
 * _min.py:17, benchmark_scatter_multiply.py:44. */
typedef enum gno_reduce {
  GNO_SUM = 0,
  GNO_MEAN = 1,
  GNO_MUL = 2,
  GNO_MIN = 3,
  GNO_MAX = 4
} gno_reduce;

/* ---------------------------------------------------------------- info -- */

int gno_abi_version(void);
const char* gno_last_error(void);
/* Number of kernels this library has launched in this process (monotonic;
 * bench.py differences it around the timed region for "gpu_launches"). */
int64_t gno_launch_count(void);

/* ---------------------------------------------------------------- sort -- */
/*
 * Stable LSD radix sort of unsigned keys (4 or 8 bytes) with an optional
 * payload (0, 4 or 8 bytes), ascending, over key bits [begin_bit, end_bit).
 * On-chip ranking: warp match + shared-memory exchange; 8 bits per pass.
 * keys_in/vals_in are not modified; results land in keys_out/vals_out.
 * Replaces the CUB radix sort under torch.sort / argsort that the reference
 * reaches through op_bm_scripts/benchmark_native_sort.py:29 and through
 * torch_sparse.coalesce (op_bm_scripts/benchmark_sparse_coalesce.py:36).
 */
int gno_sort_pairs_workspace(int64_t n, int key_bytes, int val_bytes,
                             size_t* bytes);
int gno_sort_pairs(const void* keys_in, void* keys_out, const void* vals_in,
                   void* vals_out, int64_t n, int key_bytes, int val_bytes,
                   int begin_bit, int end_bit, void* ws, size_t ws_bytes,
                   gno_stream_t stream);

/*
 * torch.sort(input, dim, stable=True) for fp32: input viewed as
 * [outer, len, inner] (row-major), sorted along `len`.  Writes sorted values
 * and int64 positions along `len`.  NaNs sort last, -0.0 == +0.0 (ties keep
 * input order), matching torch's comparison semantics.
 * Reference call site: op_bm_scripts/benchmark_native_sort.py:28-30.
 */
int gno_sort_f32_workspace(int64_t outer, int64_t len, int64_t inner,
                           size_t* bytes);
int gno_sort_f32(const float* in, float* out_values, int64_t* out_index,
                 int64_t outer, int64_t len, int64_t inner, int descending,
                 void* ws, size_t ws_bytes, gno_stream_t stream);

/* ---------------------------------------------------------------- plan -- */
/*
 * Build the dst-sorted plan of a 1-D int64 index vector (the
 * "index"/edge_index[1] argument of torch_scatter.scatter,
 * op_bm_scripts/benchmark_scatter_add.py:18 in its message-passing form):
 *   perm   [E]   int32  stable argsort of index  (perm[k] = original edge id)
 *   erow   [E]   int32  destination row of sorted edge k (the sorted keys;
 *                        N for entries that were outside [0,N))
 *   rowptr [N+1] int64  rowptr[i] = first sorted position with index >= i
 *   info   [4]   int64  device scalars: [0] #entries outside [0,N) (they sort
 *                        to the tail and belong to no row), [1] max row
 *                        length, [2] #rows that span more than one
 *                        chunk_len-edge chunk, [3] #empty rows
 * The aggregation kernel gives every worker one chunk of `chunk_len`
 * consecutive sorted edges (edge-balanced, so power-law rows cost nothing
 * extra); rows cut by a chunk boundary are finished by a second pass.
 * gno_plan_lists then materialises those rows (srow, ascending) and the
 * empty rows (zrow) once the host has read info[2], info[3].
 * Requires N < 2^31 - 1, E < 2^31, chunk_len a multiple of 32.
 */
int gno_plan_workspace(int64_t E, int64_t N, size_t* bytes);
int gno_plan_build(const int64_t* index, int64_t E, int64_t N,
                   int64_t chunk_len, int64_t* rowptr, int32_t* perm,
                   int32_t* erow, int64_t* info, void* ws, size_t ws_bytes,
                   gno_stream_t stream);
/* Same for a caller-supplied CSR rowptr (torch_sparse SparseTensor /
 * segment_csr inputs): expands erow and fills info[1..3]. */
int gno_plan_from_rowptr(const int64_t* rowptr, int64_t N, int64_t E,
                         int64_t chunk_len, int32_t* erow, int64_t* info,
                         gno_stream_t stream);
int gno_plan_lists_workspace(int64_t N, size_t* bytes);
int gno_plan_lists(const int64_t* rowptr, int64_t N, int64_t chunk_len,
                   int32_t* srow, int32_t* zrow, void* ws, size_t ws_bytes,
                   gno_stream_t stream);

/* out[k] = (int32) src[perm[k]]  — builds the sorted source-id array of the
 * fused gather→scatter form (edge_index[0] reordered by the plan). */
int gno_permute_i64_to_i32(const int64_t* src, const int32_t* perm,
                           int32_t* out, int64_t E, gno_stream_t stream);
/* out[k] = (int32) src[k] */
int gno_narrow_i64_to_i32(const int64_t* src, int32_t* out, int64_t E,
                          gno_stream_t stream);
/* out[k, :] = src[perm[k], :] for rows of row_bytes bytes (value reorder). */
int gno_permute_rows(const void* src, const int32_t* perm, void* out,
                     int64_t E, int64_t row_bytes, gno_stream_t stream);

/* ------------------------------------------------------ segment reduce -- */
/*
 * A dst-sorted graph as the kernels see it.  All pointers are device
 * pointers owned by the caller.
 */
typedef struct gno_csr {
  int64_t N;             /* destination rows */
  int64_t E;             /* sorted edges that belong to a row (= rowptr[N]) */
  const int64_t* rowptr; /* [N+1] */
  const int32_t* erow;   /* [E] destination row of sorted edge k */
  const int32_t* gidx;   /* [E] row of x to gather for sorted edge k;
                            NULL = k itself (segment_csr form) */
  const int32_t* eid;    /* [E] value reported by arg outputs for edge k
                            (original edge position); NULL = k */
  int64_t chunk_len;     /* edges per worker chunk the lists were built for */
  int64_t n_span;        /* info[2] */
  const int32_t* srow;   /* [n_span] rows cut by a chunk boundary */
  int64_t n_empty;       /* info[3] */
  const int32_t* zrow;   /* [n_empty] rows without edges */
} gno_csr;

/*
 * out[i, :] = reduce over sorted edges k in row i of  w[k] * x[gidx[k], :]
 * — the one kernel family behind scatter sum/mean/mul/min/max (+arg), the
 * fused index_select→scatter_add / index_add_ gather-reduce, segment_csr and
 * CSR spmm.  Edge-balanced segmented reduction (one chunk of sorted edges per
 * lane group), atomic-free and deterministic; fp32 accumulation for every
 * dtype, one rounding at the end.
 *
 *   x        [x_rows, F] with row stride ldx elements; x_rows*ldx elements
 *            must be readable (a padded stride is read in whole vectors)
 *   w        [E] per-sorted-edge weights in x's dtype, or NULL (spmm value)
 *   out      [N, F] with row stride ldo elements
 *   arg      [N, F] int64 (contiguous) or NULL; MIN/MAX only.  Winner =
 *            lowest eid among equal values; rows with no winner get
 *            arg_fill and out 0 (torch_scatter semantics)
 *   accumulate  non-zero: combine with the values already in out
 *            (index_add_ / out= forms; SUM and MUL only)
 *   ws       >= gno_segment_reduce_workspace(...) bytes (chunk-boundary partials)
 *
 * Replaces: scatter_add/mean/max/min (op_bm_scripts/benchmark_scatter_add.py:18,
 * _mean.py:17, _max.py:17, _min.py:17), scatter_(reduce="multiply")
 * (benchmark_scatter_multiply.py:44), index_select→sum and
 * index_add→index_select→sum (benchmark_fused_index_select_reduce.py:12-15,
 * benchmark_fused_index_add_reduce.py:12-15), index_add_
 * (benchmark_native_index_add_.py:13-16), torch.sparse.mm
 * (benchmark_sparse_spmm.py:12-14).
 */
int gno_segment_reduce_workspace(const gno_csr* g, int64_t F, int dtype,
                                 int reduce, int with_arg, size_t* bytes);
int gno_segment_reduce(const gno_csr* g, const void* x, int64_t x_rows,
                       int64_t ldx, const void* w, void* out, int64_t ldo,
                       int64_t* arg, int64_t arg_fill, int64_t F, int dtype,
                       int reduce, int accumulate, void* ws, size_t ws_bytes,
                       gno_stream_t stream);

/*
 * The same reduction with the gather source in TWO buffers of the same row
 * stride and dtype: gather ids below x_rows read x, ids x_rows + j read row j
 * of x2 (j < x2_rows).  The partitioned aggregation uses it to reduce the
 * edges whose source row the rank owns (its own feature shard) and the edges
 * whose source arrived over NVLink (the receive buffer) in ONE pass over the
 * output instead of two accumulating ones (new work, no reference
 * counterpart: the reference is single-GPU, SURVEY §2.4).
 */
int gno_segment_reduce_two(const gno_csr* g, const void* x, int64_t x_rows, int64_t ldx,
                           const void* x2, int64_t x2_rows, const void* w, void* out,
                           int64_t ldo, int64_t* arg, int64_t arg_fill, int64_t F,
                           int dtype, int reduce, int accumulate, void* ws,
                           size_t ws_bytes, gno_stream_t stream);

/*
 * Multi-head attention aggregation (GATv2's message passing, PyG
 * GATv2Conv.message + aggregate):
 *   out[i, h*C + c] = sum over sorted edges k in row i of
 *                     alpha[eid[k] * H + h] * x[gidx[k], h*C + c]
 * x [x_rows, F] and out [N, F] contiguous, F = H*C; alpha [*, H] in x's dtype,
 * read through the ORIGINAL edge id eid[k] (NULL = k), so a dst-sorted plan and
 * the src-sorted plan of the transposed aggregation (the backward w.r.t. x)
 * read the same tensor.  The segment-reduce kernel with a per-head weight: a
 * gathered vector covers columns of one head only.  With H = 1 the arithmetic
 * is gno_segment_reduce's with w[k] = alpha[eid[k]], in the same order.
 * ws >= gno_segment_reduce_workspace(g, F, dtype, GNO_SUM, 0) bytes.
 */
int gno_segment_reduce_heads(const gno_csr* g, const void* x, int64_t x_rows,
                             const void* alpha, int64_t H, void* out, int64_t F,
                             int dtype, void* ws, size_t ws_bytes,
                             gno_stream_t stream);

/*
 * Per-edge, per-head dot product (the gradient w.r.t. alpha of
 * gno_segment_reduce_heads), over a dst-sorted plan:
 *   grad_alpha[eid[k] * H + h] = sum_c grad_out[erow[k], h*C + c] * x[gidx[k], h*C + c]
 * x [x_rows, F], grad_out [N, F] contiguous, F = H*C; fp32 accumulation.  Edges
 * the plan dropped are not written.
 */
int gno_edge_head_dot(const gno_csr* g, const void* x, int64_t x_rows,
                      const void* grad_out, int64_t H, int64_t F,
                      void* grad_alpha, int dtype, gno_stream_t stream);

/*
 * Segment softmax over destination rows (torch_geometric.utils.softmax of PyG
 * 2.0.2, GATv2REG's attention normalisation), H heads per edge:
 *   m[i, h] = max of the row's logits (torch_scatter rule: start at the dtype's
 *             lowest finite value, strictly greater wins, NaN never wins, no
 *             winner -> 0)
 *   out[e, h] = exp(src[e, h] - m[dst[e], h]) / (sum over the row of exp(src - m) + eps)
 * src / out [E, H] are in ORIGINAL edge order.  dst[e] = index[e] (int64, the
 * index the plan was built from; edges outside [0, N) get 0), or index = NULL
 * for a plan made by gno_plan_from_rowptr (original order = sorted order,
 * E = g->E).  The plan's eid must be its perm (NULL with a rowptr plan).  fp32
 * math, one rounding; atomic-free and bit-reproducible.  The backward writes
 *   grad_src[e, h] = out[e, h] * (grad_out[e, h] - sum over the row of grad_out * out).
 * ws >= gno_segment_softmax_workspace(g, H) bytes (both directions).
 */
int gno_segment_softmax_workspace(const gno_csr* g, int64_t H, size_t* bytes);
int gno_segment_softmax(const gno_csr* g, const void* src, const int64_t* index,
                        int64_t E, int64_t H, double eps, void* out, int dtype,
                        void* ws, size_t ws_bytes, gno_stream_t stream);
int gno_segment_softmax_backward(const gno_csr* g, const void* out,
                                 const void* grad_out, const int64_t* index,
                                 int64_t E, int64_t H, void* grad_src, int dtype,
                                 void* ws, size_t ws_bytes, gno_stream_t stream);

/*
 * GATv2 attention logits (PyG 2.0.2 GATv2Conv.message: leaky_relu(x_i + x_j),
 * then (. * att).sum(-1)), over the dst-sorted plan of dst with gidx = src[perm]:
 *   out[eid[k] * H + h] = sum_c att[h*C + c] *
 *       leaky_relu(x_l[gidx[k], h*C + c] + x_r[erow[k], h*C + c], negative_slope)
 * x_l [xl_rows, F], x_r [N, F], att [F] contiguous in `dtype`, F = H*C; out [E, H]
 * in original edge order.  The sum z is formed in fp32 from the stored values;
 * fp32 accumulation, one rounding.  E = 0 touches nothing.
 */
int gno_gatv2_logits(const gno_csr* g, const void* x_l, int64_t xl_rows,
                     const void* x_r, const void* att, int64_t H, int64_t F,
                     double negative_slope, void* out, int dtype,
                     gno_stream_t stream);

/*
 * Backward of gno_gatv2_logits along one plan (grad_logits [E, H], original order):
 *   grad_own[i, f] = att[f] * sum_{k in row i} grad_logits[eid[k]*H + h] * (z > 0 ? 1 : slope)
 *   grad_att[f]    = sum over the plan's edges of grad_logits[eid[k]*H + h] * leaky_relu(z)
 * with z = other[gidx[k], f] + own[i, f] in fp32 and h = f / C.  Run on the dst
 * plan with own = x_r, other = x_l (gidx = src[perm]) for grad_x_r and grad_att, and
 * on the src plan with own = x_l, other = x_r (gidx = dst[perm]) for grad_x_l.
 * grad_own [N, F] in `dtype` (empty rows get 0) and grad_att fp32 [F] may each be
 * NULL, not both.  No atomics: bit-reproducible.
 * ws >= gno_gatv2_logits_backward_workspace(g, H, F, grad_own != NULL,
 * grad_att != NULL) bytes: the chunk partials of grad_own and the per-CTA
 * partials of grad_att are reserved only for the outputs requested.
 */
int gno_gatv2_logits_backward_workspace(const gno_csr* g, int64_t H, int64_t F,
                                        int with_grad_own, int with_grad_att,
                                        size_t* bytes);
int gno_gatv2_logits_backward(const gno_csr* g, const void* own, const void* other,
                              int64_t other_rows, const void* att,
                              const void* grad_logits, int64_t H, int64_t F,
                              double negative_slope, void* grad_own, float* grad_att,
                              int dtype, void* ws, size_t ws_bytes,
                              gno_stream_t stream);

/*
 * A GATv2 layer's whole message passing in one pass over the dst-sorted plan of
 * dst (gidx = src[perm], eid = perm): gno_gatv2_logits, gno_segment_softmax and
 * gno_segment_reduce_heads fused, the way flash attention fuses score, softmax
 * and weighted sum:
 *   a[e, h]      = sum_c att[h*C + c] * leaky_relu(x_l[src, h*C + c] + x_r[dst, h*C + c])
 *   alpha[e, h]  = exp(a - m[dst, h]) / s[dst, h]   (gno_segment_softmax's max rule)
 *   out[i, h*C + c] = sum over the row's edges of alpha[e, h] * x_l[src, h*C + c]
 * Each gathered x_l vector is loaded once and serves the logit and the weighted
 * sum (online max / sum-of-exp rescaling).  Neither a nor alpha is written:
 * out [N, F] in `dtype` (empty rows get 0) and the fp32 row statistics m [N, H]
 * (the max after the empty-value rule) and s [N, H] (sum of exp(a - m) + eps)
 * are, for the backward.  x_l [xl_rows, F], x_r [N, F], att [F] contiguous,
 * F = H*C; a head may span at most 128 vectors of the widest load that divides
 * it.  fp32 math, one rounding per output; atomic-free, bit-reproducible.
 * E = 0 touches nothing.  ws >= gno_gatv2_attention_workspace(g, H, F) bytes.
 */
int gno_gatv2_attention_workspace(const gno_csr* g, int64_t H, int64_t F, size_t* bytes);
int gno_gatv2_attention(const gno_csr* g, const void* x_l, int64_t xl_rows,
                        const void* x_r, const void* att, int64_t H, int64_t F,
                        double negative_slope, double eps, void* out, float* m,
                        float* s, int dtype, void* ws, size_t ws_bytes,
                        gno_stream_t stream);

/*
 * The destination pass of gno_gatv2_attention's backward, on the same plan.
 * With D[i, h] = sum_c grad_out[i, h*C + c] * out[i, h*C + c], it recomputes a
 * and alpha from m and s and forms
 *   da[e, h]       = alpha * (sum_c grad_out[dst, h*C + c] * x_l[src, h*C + c] - D[dst, h])
 *   grad_x_r[i, f] = att[f] * sum over the row's edges of da * leaky_relu'(z)   (empty rows 0)
 *   grad_att[f]    = sum_e da * leaky_relu(z)                                  (fp32)
 * and writes grad_logits = da and alpha [E, H] in original edge order, the
 * inputs of the source pass: gno_gatv2_logits_backward (own = x_l, other = x_r,
 * grad_logits = da) on the src plan gives the logit part of grad_x_l, and
 * gno_segment_reduce_heads (x = grad_out, alpha) the rest.  grad_x_r, grad_att
 * and the pair (grad_logits, alpha) may each be NULL, not all three.  No
 * atomics: bit-reproducible.  ws >= gno_gatv2_attention_backward_workspace(g,
 * H, F, grad_x_r != NULL, grad_att != NULL) bytes.
 */
int gno_gatv2_attention_backward_workspace(const gno_csr* g, int64_t H, int64_t F,
                                           int with_grad_x_r, int with_grad_att,
                                           size_t* bytes);
int gno_gatv2_attention_backward(const gno_csr* g, const void* x_l, int64_t xl_rows,
                                 const void* x_r, const void* att, const void* out,
                                 const float* m, const float* s, const void* grad_out,
                                 int64_t H, int64_t F, double negative_slope,
                                 void* grad_x_r, float* grad_att, void* grad_logits,
                                 void* alpha, int dtype, void* ws, size_t ws_bytes,
                                 gno_stream_t stream);

/*
 * Several aggregators over one neighbourhood in one pass (PNAConv.aggregate of PyG: a list of
 * aggregators concatenated, then copies scaled by degree scalers; Corso et al., "Principal
 * Neighbourhood Aggregation").  Codes of the aggregators and scalers, in output order:
 */
typedef enum gno_aggregator {
  GNO_AGG_SUM = 0,
  GNO_AGG_MEAN = 1,
  GNO_AGG_MIN = 2,
  GNO_AGG_MAX = 3,
  GNO_AGG_VAR = 4,
  GNO_AGG_STD = 5
} gno_aggregator;
typedef enum gno_scaler {
  GNO_SCALE_IDENTITY = 0,
  GNO_SCALE_AMPLIFICATION = 1,  /* log(d + 1) / avg_log */
  GNO_SCALE_ATTENUATION = 2,    /* avg_log / log(d + 1) */
  GNO_SCALE_LINEAR = 3,         /* d / avg_lin */
  GNO_SCALE_INVERSE_LINEAR = 4  /* avg_lin / d */
} gno_scaler;

/*
 * Forward over the dst-sorted plan: message m_e = x[gidx[k], :] of sorted edge k (edge id
 * eid[k]); x [x_rows, T*F] contiguous (T towers of F columns).  With d = max(row length, 1):
 *   sum = Σ m, mean = sum / d, var = Σ m² / d − mean², std = sqrt(relu(var) + 1e-5),
 *   min / max with torch_scatter's rule (lowest edge wins a tie, NaN never wins, empty -> 0),
 *   out[i, t*S*A*F + (s*A + a)*F + f] = agg_a · scale_s(d)      (out [N, T*S*A*F])
 * aggs [n_aggs] and scalers [n_scalers] are host arrays of the codes above (1..8 each,
 * duplicates allowed).  Σm and Σm² accumulate in fp32; rows cut by a chunk boundary combine
 * their chunk partials in chunk order in fp64; the scale is applied in fp32 and each output is
 * rounded once.  For the backward, optionally: int32 winners arg_min / arg_max [N, T*F]
 * (original edge ids, arg_fill where nothing won; need min or max among aggs) and fp32 mean /
 * var [N, T*F] (var before relu; both or neither).  No atomics: bit-reproducible.
 * ws >= gno_multi_aggregate_workspace(g, T, F, aggs, n_aggs) bytes.
 */
int gno_multi_aggregate_workspace(const gno_csr* g, int64_t T, int64_t F,
                                  const int* aggs, int n_aggs, size_t* bytes);
int gno_multi_aggregate(const gno_csr* g, const void* x, int64_t x_rows, int64_t T,
                        int64_t F, const int* aggs, int n_aggs, const int* scalers,
                        int n_scalers, double avg_lin, double avg_log, void* out,
                        int32_t* arg_min, int32_t* arg_max, float* mean, float* var,
                        int64_t arg_fill, int dtype, void* ws, size_t ws_bytes,
                        gno_stream_t stream);

/*
 * Backward of gno_multi_aggregate w.r.t. the messages (message form: gidx = eid = the plan's
 * perm, x [E, T*F] in original edge order).  grad_out [N, T*S*A*F] in `dtype`; the winners
 * and mean / var saved by the forward (winners of each requested extreme, mean / var when var or
 * std is requested).  Per row, c_a = Σ_s scale_s · grad_out block (s, a),
 * cv = c_var + c_std · [var > 0] / (2 std), and every edge e of the row gets
 *   grad_x[e] = c_sum + c_mean / d + 2 cv (m_e − mean) / d + [e = argmin] c_min + [e = argmax] c_max
 * Each element of grad_x [x_rows, T*F] that a kept edge owns is written once (no atomics); edges
 * the plan dropped are not written.
 */
int gno_multi_aggregate_backward(const gno_csr* g, const void* x, int64_t x_rows,
                                 int64_t T, int64_t F, const int* aggs, int n_aggs,
                                 const int* scalers, int n_scalers, double avg_lin,
                                 double avg_log, const void* grad_out,
                                 const int32_t* arg_min, const int32_t* arg_max,
                                 const float* mean, const float* var, void* grad_x,
                                 int dtype, gno_stream_t stream);

/*
 * Node-level coefficients of the same backward (gather form, where grad_x[j] sums over the
 * edges with source j): fp32 pq [N + 1, 2*T*F] gets rows [P | Q] for rows 0..N-1 with
 *   P = c_sum + c_mean / d − 2 cv · mean / d,  Q = 2 cv / d
 * (row N is left to the caller), and c_min / c_max [N, T*F] fp32 are written when non-NULL.
 */
int gno_multi_aggregate_coeffs(const gno_csr* g, int64_t T, int64_t F, const int* aggs,
                               int n_aggs, const int* scalers, int n_scalers,
                               double avg_lin, double avg_log, const void* grad_out,
                               const int32_t* arg_min, const int32_t* arg_max,
                               const float* mean, const float* var, float* pq,
                               float* c_min, float* c_max, int dtype, gno_stream_t stream);

/*
 * Integer form (int32 / int64 values, exact int64 accumulation): torch_scatter.scatter on
 * integer tensors — PyG's TopKPooling / to_dense_batch count nodes per graph with
 * scatter_add(batch.new_ones(n), batch, dim=0) (graph_benchmark/models/ptg_models.py:165-172).
 * x [rows, K] with row stride ldx elements, out [N, K]; MEAN is the floor division upstream
 * applies to integer tensors; MIN/MAX report the lowest edge position among equal values.
 */
int gno_segment_reduce_int(const gno_csr* g, const void* x, int64_t ldx,
                           void* out, int64_t ldo, int64_t* arg,
                           int64_t arg_fill, int64_t K, int elem_bytes,
                           int reduce, int accumulate, gno_stream_t stream);

/*
 * Last-dim form: out[b, i] = reduce_{k in row i} x[b, gidx[k]] for x [B, L]
 * (dim == last, 1-D index): index_select / index_add_ along dim 1
 * (benchmark_native_index_add_.py:62, benchmark_fused_*_reduce.py dim=1).
 * Source rows are staged through shared memory.
 */
int gno_segment_reduce_lastdim(const gno_csr* g, const void* x, int64_t B,
                               int64_t L, int64_t ldx, void* out, int64_t ldo,
                               int64_t* arg, int64_t arg_fill, int dtype,
                               int reduce, int accumulate,
                               gno_stream_t stream);

/* Re-stride a row-major matrix: dst[r, :row_bytes] = src[r, :row_bytes] with
 * independent row strides.  Used to give feature rows a 16-byte-multiple
 * stride (F=602: 2408 B fp32 / 1204 B bf16 rows) so the gather kernel can use
 * 128-bit loads; gno_segment_reduce reads whole vectors when ldx leaves room. */
int gno_pad_rows(const void* src, int64_t rows, int64_t row_bytes,
                 int64_t src_stride_bytes, void* dst, int64_t dst_stride_bytes,
                 gno_stream_t stream);

/* Batched 2-D transpose out[o, c, r] = in[o, r, c] of 4- or 8-byte elements
 * (32x32 shared-memory tiles).  Used by gno_b200.sort to move an inner sorted
 * dim last and back: torch.sort(input, dim=0) of
 * op_bm_scripts/benchmark_native_sort.py:28-30. */
int gno_transpose_batched(const void* in, void* out, int64_t outer,
                          int64_t rows, int64_t cols, int elem_bytes,
                          gno_stream_t stream);

/* out[k, :] = x[index[k], :]  (row gather with 128-bit accesses): the
 * un-fused index_select of benchmark_native_index_select.py:12-15. */
int gno_gather_rows(const void* x, int64_t x_rows, int64_t row_bytes,
                    const int64_t* index, int64_t n_index, void* out,
                    gno_stream_t stream);

/*
 * Multi-GPU needed-rows exchange, fused with NVLink delivery: for every row a
 * peer requested (slots seg[q]..seg[q+1] belong to peer q, HOST arrays of
 * n_peers+1 / n_peers entries), read x[serve_rows[slot]] once from local HBM
 * and store it directly into that peer's receive buffer through its mapped
 * peer pointer (peer_bufs[q], e.g. from torch symmetric memory / CUDA IPC) at
 * row row_off[q] + slot - seg[q].  serve_rows == NULL sends row slot - seg[q]
 * (every peer receives all local rows: an all-gather by peer stores).  Slots are served in rotated order starting
 * at start_slot (pass seg[(rank+1) % n_peers]) so that at any moment the ranks
 * push to different receivers.  max_blocks > 0 caps the grid: posted peer
 * stores keep NVLink busy from a few warps per SM, and a small grid leaves the
 * SM slots to a reduction running beside it on another stream (0 = fill the
 * chip).  Replaces "gather into a send buffer, then all-to-all"; the caller
 * provides the cross-rank barrier (new work, no reference counterpart: the
 * reference is single-GPU, SURVEY §2.4).
 */
/* Ring slot size of the TMA-staged form of gno_push_rows (4096..16384 bytes, four slots per
 * CTA; 0 = the GNO_PUSH_CHUNK environment variable, else 8192): small slots leave shared memory to
 * a reduction running beside the push, large ones keep more bytes in flight. */
int gno_push_set_chunk(int bytes);
int gno_push_rows(const void* x, int64_t row_bytes, int64_t src_stride_bytes,
                  const int64_t* serve_rows, int64_t n_serve, int n_peers,
                  void* const* peer_bufs, const int64_t* seg,
                  const int64_t* row_off, int64_t dst_stride_bytes,
                  int64_t start_slot, int max_blocks, gno_stream_t stream);

/* -------------------------------------------- element-wise index form -- */
/*
 * torch_scatter.scatter with a FULL-SHAPE index (same shape as src) — what
 * op_bm_scripts/benchmark_scatter_{add,max,min,mean}.py:60-84 pass: src and
 * index viewed as [B, E, K], out as [B, N, K]:
 *   out[b, index[b,e,k], k] = reduce(src[b,e,k]).
 * One launch when the N bins of up to 16 adjacent columns fit in shared
 * memory (every script shape): the input is streamed once, every update is a
 * shared-memory atomic, no global atomics and no workspace
 * (gno_scatter_elementwise_workspace then returns 0).  MIN/MAX values and arg
 * are deterministic (lowest e among ties, like the sequential upstream loop);
 * fp16 SUM/MEAN accumulate exactly in 64-bit fixed point (order-independent,
 * one rounding); fp32/bf16 SUM/MEAN and MUL accumulate in fp32 and round once.
 * Larger N falls back to fp32 L2 atomics in `ws`.
 *   accumulate  non-zero = torch_scatter's out= form: combine with the values
 *               already in out (on-chip path only)
 */
int gno_scatter_elementwise_workspace(int64_t B, int64_t E, int64_t N,
                                      int64_t K, int dtype, int reduce,
                                      size_t* bytes);
int gno_scatter_elementwise(const void* src, const int64_t* index, int64_t B,
                            int64_t E, int64_t K, void* out, int64_t* arg,
                            int64_t N, int dtype, int reduce, int accumulate,
                            void* ws, size_t ws_bytes, gno_stream_t stream);

/*
 * The same op on a cached plan of the index (atomic-free, deterministic for
 * every dtype): the host sorts the index once (gno_sort_pairs, stable) and
 * reuses the plan for every call on that index tensor (the reference scripts
 * time 100 calls on one index, op_bm_scripts/benchmark_scatter_add.py:97-118).
 * The plan is BLOCKED by the CTA that consumes it: a CTA owns KB = 1 << kb_shift
 * adjacent columns (gno_scatter_planned_layout), ncb = ceil(K / KB), and the
 * blocked id of output (b, n, k = cb*KB + kk) is
 *   ob = (((b*ncb + cb)*N + n) << kb_shift) + kk
 *   ptr   [B*ncb*N*KB + 1] int32  output ob owns order[ptr[ob]:ptr[ob+1])
 *   order [B*E*K] int16 (order_bytes = 2, E <= 32768) or int32: position e along
 *         the scatter dim of each element, elements in ascending (ob, e)
 * so every CTA reads one contiguous slice of each.  It stages its KB source
 * columns in shared memory and reduces each output's segment sequentially
 * (ascending e: upstream's CPU loop order; ties of MIN/MAX keep the lowest
 * position).  gno_scatter_planned_layout returns 1 and the layout parameters
 * when a source column fits in shared memory and the plan indexes with 32 bits,
 * else 0 (gno_scatter_planned_ok: the same test without the outputs).
 */
int gno_scatter_planned_layout(int64_t B, int64_t E, int64_t K, int64_t N, int dtype,
                               int* kb_shift, int* order_bytes);
int gno_scatter_planned_ok(int64_t B, int64_t E, int64_t K, int64_t N, int dtype);
int gno_scatter_planned(const void* src, const void* order, const int32_t* ptr,
                        int64_t B, int64_t E, int64_t K, void* out, int64_t* arg,
                        int64_t N, int dtype, int reduce, int accumulate,
                        gno_stream_t stream);

/* ------------------------------------------------- coalesce / transpose -- */
/*
 * torch_sparse.coalesce(index, value, m, n, op): sort COO entries by
 * (row, col), merge duplicates (op = SUM/MEAN/MIN/MAX/MUL over `value`
 * rows of K elements).  Outputs are sized for E entries; *nnz_out (device
 * int64) receives the merged count.  Passing (col,row,n,m) gives
 * torch_sparse.transpose.  flags: bit0 = input known sorted by `row`
 * (sort only the low key bits); bit1 = sort only, duplicate (row, col) entries
 * stay separate (torch_sparse.SparseStorage's construction order: it sorts by
 * row*n+col and never merges).
 * Reference call site: op_bm_scripts/benchmark_sparse_coalesce.py:35-37;
 * transpose: data/sparse_transpose.csv rows (torch_sparse.transpose).
 */
int gno_coalesce_workspace(int64_t E, int64_t m, int64_t n, int64_t K,
                           int dtype, size_t* bytes);
int gno_coalesce(const int64_t* row, const int64_t* col, const void* value,
                 int64_t K, int dtype, int64_t E, int64_t m, int64_t n,
                 int reduce, int flags, int64_t* out_row, int64_t* out_col,
                 void* out_value, int64_t* nnz_out, void* ws, size_t ws_bytes,
                 gno_stream_t stream);
/* Device check used for torch_sparse's early exit: status[0] = #inversions
 * of key=row*n+col, status[1] = #adjacent duplicates. */
int gno_coo_order_check(const int64_t* row, const int64_t* col, int64_t E,
                        int64_t n, int64_t* status, gno_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GNO_B200_H */
