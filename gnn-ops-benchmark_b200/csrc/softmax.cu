// Segment softmax over a dst-sorted plan (torch_geometric.utils.softmax, PyG 2.0.2), forward and
// backward, for logits of H heads per edge:
//
//   m[i, h]   = max of the row's logits, torch_scatter rule: start at the dtype's finite lowest(),
//               take strictly greater values (a NaN never wins), still lowest() at the end -> 0
//   y[e, h]   = exp(a[e, h] - m[dst[e], h]) / (sum_{row} exp(a - m) + eps)
//   grad_a    = y * (g - sum_{row} g * y)            (exact for any eps: the shift is a constant)
//
// Logits, outputs and gradients are [E, H] in ORIGINAL edge order, the order PyG produces and
// consumes.  Two passes per direction:
//   1. softmax_stats_kernel, edge-balanced like the segment reduce: one thread per (chunk of
//      chunk_len sorted edges, head) walks its chunk in sorted order, reading a[perm[k], h], and
//      keeps the running (max, sum of exp relative to the max) of the current row (online form:
//      one exp per logit).  Rows that end inside the chunk are finished in place; rows cut by a
//      chunk boundary leave partials (two slots per chunk, as in segreduce.cu) that
//      softmax_finish_kernel combines IN CHUNK ORDER in fp64: m = max(m1, m2),
//      s = s1 e^(m1-m) + s2 e^(m2-m).  The backward pass reuses both kernels for the row dot
//      product sum g*y (partials are added).
//   2. softmax_apply_kernel, one thread per (edge, head) in original order: read the edge's
//      logit and destination (the caller's int64 index, or erow when the plan came from a rowptr),
//      look up the row's statistics, write the result coalesced.  Edges whose destination lies
//      outside [0, N) get 0.
// fp32 math for every dtype, one rounding per output.  No atomics: bit-reproducible.
//
// Roofline: HBM.  Bytes per (edge, head) = forward: s (logit, read via perm in pass 1) + s (logit,
// pass 2) + s (y) ; backward: 2s (y, g in pass 1) + 2s (pass 2) + s (grad); per edge 4 (perm) +
// 4 (erow) + 8 (int64 index, or 4 erow); the [N, H] statistics are 8 bytes per (row, head).
#include <climits>

#include "common.cuh"

namespace gno {

constexpr int kSmThreads = 256;
constexpr int kSmBatch = 8;  // sorted edges whose records and logits are loaded before use

struct SmParams {
  const int32_t* erow;
  const int32_t* eid;      // original edge id of sorted edge k (NULL = k)
  const int32_t* srow;
  const int64_t* rowptr;
  const int64_t* index;    // original-order destinations (NULL: erow, original order = sorted order)
  const void* a;           // forward: logits; backward: y
  const void* b;           // backward: g (unused forward)
  void* out;
  float2* stats;           // [N, H]: (m, sum + eps) forward, (0, sum g*y) backward
  float2* part;            // [2 * n_chunks, H] partials of rows cut by a chunk boundary
  int64_t N, E, E_total, n_chunks, n_span;
  float eps;
  int H;
  int chunk_len;
  bool narrow;             // (edges * H) < 2^32: 32-bit division splits thread ids
};

__device__ __forceinline__ int64_t split_heads(int64_t t, int H, bool narrow) {
  return narrow ? (int64_t)((uint32_t)t / (uint32_t)H) : t / H;
}

// Row statistics -> what the apply pass reads.
template <typename T, bool BWD>
__device__ __forceinline__ float2 sm_final(float m, float s, float eps) {
  if constexpr (BWD) {
    return make_float2(0.f, s);
  } else {
    const float mf = (m == DType<T>::lowest()) ? 0.f : m;  // no logit won: torch_scatter's empty value
    if (mf != m) s *= expf(m - mf);
    return make_float2(mf, s + eps);
  }
}

template <typename T, bool BWD>
__global__ void __launch_bounds__(kSmThreads) softmax_stats_kernel(const SmParams p) {
  const int64_t t = (int64_t)blockIdx.x * kSmThreads + threadIdx.x;
  const int H = p.H;
  const int64_t c = split_heads(t, H, p.narrow);
  if (c >= p.n_chunks) return;
  const int h = (int)(t - c * H);
  const int64_t k0 = c * p.chunk_len;
  const int nv = (int)imin64(p.chunk_len, p.E - k0);
  const T* a = static_cast<const T*>(p.a) + h;
  const T* b = static_cast<const T*>(p.b) + h;
  const float lowest = DType<T>::lowest();

  int cur = __ldg(p.erow + k0);
  bool head = k0 > 0 && __ldg(p.erow + k0 - 1) == cur;
  float m = BWD ? 0.f : lowest, s = 0.f;
  auto flush = [&](bool tail) {
    if (head || tail) {  // a chunk inside one row is both: it uses the head slot
      p.part[(2 * c + (head ? 0 : 1)) * H + h] = make_float2(m, s);
    } else {
      p.stats[(int64_t)cur * H + h] = sm_final<T, BWD>(m, s, p.eps);
    }
  };
  auto step = [&](int row, float v, float w) {
    if (row != cur) {
      flush(false);
      head = false;
      cur = row;
      m = BWD ? 0.f : lowest;
      s = 0.f;
    }
    if constexpr (BWD) {
      s = fmaf(v, w, s);
    } else if (v > m) {  // strict: NaN never wins, and its exp makes the row's sum NaN below
      // the winner's own term is exp(v - v): 1, or NaN for +inf (PyG's exp(inf - inf) makes the
      // whole row NaN)
      s = s * expf(m - v) + (v == INFINITY ? __int_as_float(0x7fffffff) : 1.f);
      m = v;
    } else {
      s += expf(v - m);
    }
  };
  int i = 0;
  for (; i + kSmBatch <= nv; i += kSmBatch) {
    int row[kSmBatch];
    float v[kSmBatch], w[kSmBatch];
#pragma unroll
    for (int u = 0; u < kSmBatch; ++u) {
      const int64_t k = k0 + i + u;
      row[u] = __ldg(p.erow + k);
      const int64_t e = p.eid ? (int64_t)__ldg(p.eid + k) : k;
      v[u] = DType<T>::to_f(a[e * H]);
      w[u] = BWD ? DType<T>::to_f(b[e * H]) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < kSmBatch; ++u) step(row[u], v[u], w[u]);
  }
  for (; i < nv; ++i) {
    const int64_t k = k0 + i;
    const int64_t e = p.eid ? (int64_t)__ldg(p.eid + k) : k;
    step(__ldg(p.erow + k), DType<T>::to_f(a[e * H]), BWD ? DType<T>::to_f(b[e * H]) : 0.f);
  }
  flush(k0 + nv < p.E && __ldg(p.erow + k0 + nv) == cur);
}

// Rows cut by a chunk boundary: the tail slot of the first chunk, then the head slot of every
// later chunk, combined in chunk order in fp64 (a hub row has thousands of partials).
template <typename T, bool BWD>
__global__ void __launch_bounds__(kSmThreads) softmax_finish_kernel(const SmParams p) {
  const int64_t t = (int64_t)blockIdx.x * kSmThreads + threadIdx.x;
  const int H = p.H;
  const int64_t i = split_heads(t, H, p.narrow);
  if (i >= p.n_span) return;
  const int h = (int)(t - i * H);
  const int64_t row = p.srow[i];
  const int64_t kb = p.rowptr[row], ke = p.rowptr[row + 1];
  const int64_t ca = kb / p.chunk_len, cb = (ke - 1) / p.chunk_len;
  const float2 first = p.part[(2 * ca + 1) * H + h];
  double m = first.x, s = first.y;
  for (int64_t c = ca + 1; c <= cb; ++c) {
    const float2 q = p.part[2 * c * H + h];
    if constexpr (BWD) {
      s += (double)q.y;
    } else {
      const double mn = q.x > m ? (double)q.x : m;
      s = s * exp(m - mn) + (double)q.y * exp((double)q.x - mn);
      m = mn;
    }
  }
  p.stats[row * H + h] = sm_final<T, BWD>((float)m, (float)s, p.eps);
}

template <typename T, bool BWD>
__global__ void __launch_bounds__(kSmThreads) softmax_apply_kernel(const SmParams p) {
  const int64_t t = (int64_t)blockIdx.x * kSmThreads + threadIdx.x;
  if (t >= p.E_total * p.H) return;
  const int64_t e = split_heads(t, p.H, p.narrow);
  const int h = (int)(t - e * p.H);
  const int64_t row = p.index ? __ldg(p.index + e) : (int64_t)__ldg(p.erow + e);
  const float v = DType<T>::to_f(static_cast<const T*>(p.a)[t]);
  float r = 0.f;
  if (row >= 0 && row < p.N) {
    const float2 st = p.stats[row * p.H + h];
    if constexpr (BWD) {
      r = v * (DType<T>::to_f(static_cast<const T*>(p.b)[t]) - st.y);
    } else {
      r = __fdiv_rn(expf(v - st.x), st.y);
    }
  }
  static_cast<T*>(p.out)[t] = DType<T>::from_f(r);
}

template <typename T, bool BWD>
static int launch_softmax(const SmParams& p, cudaStream_t s) {
  const int64_t H = p.H;
  if (p.n_chunks > 0) {
    softmax_stats_kernel<T, BWD><<<(unsigned)ceil_div(p.n_chunks * H, kSmThreads), kSmThreads, 0, s>>>(p);
    GNO_LAUNCHED("softmax_stats_kernel");
  }
  if (p.n_span > 0) {
    softmax_finish_kernel<T, BWD><<<(unsigned)ceil_div(p.n_span * H, kSmThreads), kSmThreads, 0, s>>>(p);
    GNO_LAUNCHED("softmax_finish_kernel");
  }
  if (p.E_total > 0) {
    softmax_apply_kernel<T, BWD><<<(unsigned)ceil_div(p.E_total * H, kSmThreads), kSmThreads, 0, s>>>(p);
    GNO_LAUNCHED("softmax_apply_kernel");
  }
  return GNO_OK;
}

static int softmax_sizes_ok(const gno_csr* g, int64_t H, const char* fn) {
  GNO_CHECK_ARG(g != nullptr, "%s: graph is NULL", fn);
  GNO_CHECK_ARG(H > 0 && H < (int64_t(1) << 20), "%s: bad head count H=%lld", fn, (long long)H);
  GNO_CHECK_ARG(g->N >= 0 && g->E >= 0 && g->E < (int64_t(1) << 31), "%s: bad sizes N=%lld E=%lld", fn,
                (long long)g->N, (long long)g->E);
  GNO_CHECK_ARG(g->chunk_len >= 32 && g->chunk_len % 32 == 0 && g->chunk_len <= (1 << 20),
                "%s: chunk_len must be a multiple of 32", fn);
  return GNO_OK;
}

static int softmax_run(bool bwd, const gno_csr* g, const void* a, const void* b, const int64_t* index,
                       int64_t E, int64_t H, float eps, void* out, int dtype, void* wsp, size_t ws_bytes,
                       gno_stream_t stream) {
  const char* fn = bwd ? "gno_segment_softmax_backward" : "gno_segment_softmax";
  if (int rc = softmax_sizes_ok(g, H, fn)) return rc;
  GNO_CHECK_ARG(dtype == GNO_F32 || dtype == GNO_F16 || dtype == GNO_BF16, "%s: unknown dtype %d", fn, dtype);
  GNO_CHECK_ARG(E >= 0 && E >= g->E && (index != nullptr || E == g->E),
                "%s: E=%lld edges for a plan of %lld (without an index they must be equal)", fn, (long long)E,
                (long long)g->E);
  if (E == 0) return GNO_OK;
  GNO_CHECK_ARG(a && out && (!bwd || b) && (g->E == 0 || (g->erow && g->rowptr)) &&
                    (index || g->erow) && (g->n_span == 0 || g->srow),
                "%s: NULL buffer", fn);
  SmParams p;
  p.erow = g->erow;
  p.eid = g->eid;
  p.srow = g->srow;
  p.rowptr = g->rowptr;
  p.index = index;
  p.a = a;
  p.b = b;
  p.out = out;
  p.N = g->N;
  p.E = g->E;
  p.E_total = E;
  p.n_chunks = ceil_div(g->E, g->chunk_len);
  p.n_span = g->n_span;
  p.eps = eps;
  p.H = (int)H;
  p.chunk_len = (int)g->chunk_len;
  p.narrow = E * H < (int64_t(1) << 32);
  p.stats = nullptr;
  p.part = nullptr;
  if (p.n_chunks > 0) {
    if (wsp == nullptr) return fail(GNO_ERR_WORKSPACE, "%s: workspace is NULL", fn);
    Workspace ws(wsp, ws_bytes);
    p.stats = ws.take<float2>((size_t)(g->N * H));
    p.part = ws.take<float2>((size_t)(2 * p.n_chunks * H));
    if (!ws.ok()) return fail(GNO_ERR_WORKSPACE, "%s: workspace too small (%zu < %zu)", fn, ws_bytes, ws.off);
  }
  cudaStream_t s = (cudaStream_t)stream;
  switch (dtype) {
    case GNO_F32: return bwd ? launch_softmax<float, true>(p, s) : launch_softmax<float, false>(p, s);
    case GNO_F16: return bwd ? launch_softmax<__half, true>(p, s) : launch_softmax<__half, false>(p, s);
    default:
      return bwd ? launch_softmax<__nv_bfloat16, true>(p, s) : launch_softmax<__nv_bfloat16, false>(p, s);
  }
}

}  // namespace gno

using namespace gno;

extern "C" {

int gno_segment_softmax_workspace(const gno_csr* g, int64_t H, size_t* bytes) {
  GNO_CHECK_ARG(bytes != nullptr, "gno_segment_softmax_workspace: NULL argument");
  if (int rc = softmax_sizes_ok(g, H, "gno_segment_softmax_workspace")) return rc;
  WorkspaceSizer sz;
  const int64_t n_chunks = ceil_div(g->E, g->chunk_len);
  if (n_chunks > 0) {
    sz.take<float2>((size_t)(g->N * H));
    sz.take<float2>((size_t)(2 * n_chunks * H));
  }
  *bytes = sz.total();
  return GNO_OK;
}

int gno_segment_softmax(const gno_csr* g, const void* src, const int64_t* index, int64_t E, int64_t H,
                        double eps, void* out, int dtype, void* ws, size_t ws_bytes, gno_stream_t stream) {
  return softmax_run(false, g, src, nullptr, index, E, H, (float)eps, out, dtype, ws, ws_bytes, stream);
}

int gno_segment_softmax_backward(const gno_csr* g, const void* out, const void* grad_out, const int64_t* index,
                                 int64_t E, int64_t H, void* grad_src, int dtype, void* ws, size_t ws_bytes,
                                 gno_stream_t stream) {
  return softmax_run(true, g, out, grad_out, index, E, H, 0.f, grad_src, dtype, ws, ws_bytes, stream);
}

}  // extern "C"
