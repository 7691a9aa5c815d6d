// GATv2 attention logits (PyG 2.0.2 GATv2Conv.message: x_i + x_j, leaky_relu, (x * att).sum(-1))
// without the [E, H, C] messages, forward and backward:
//
//   z[e, h, c]   = x_l[src[e], h*C + c] + x_r[dst[e], h*C + c]          (fp32, from the stored values)
//   logits[e, h] = sum_c att[h*C + c] * leaky_relu(z[e, h, c])
//
//   grad_x_r[i, f] = att[f] * sum_{e: dst[e] = i} g[e, h] * d(z[e, f]),   d(z) = z > 0 ? 1 : slope
//   grad_x_l[j, f] = att[f] * sum_{e: src[e] = j} g[e, h] * d(z[e, f])
//   grad_att[f]    = sum_e g[e, h] * leaky_relu(z[e, f])                    (h = f / C)
//
// d is torch's leaky_relu_backward (z = 0 takes the slope).  The sign of an fp32 sum of two
// representable values is exact, so the branch agrees with an fp64 reference.
//
//   gatv2_logits_kernel: one thread per (dst-sorted edge, head).  The gathered x_l head slice
//   comes from HBM; the edges of a row are consecutive, so the row's x_r slice comes from HBM once
//   and from L1 for the rest of the row.  The logit goes to out[eid * H + h] (original order).
//
//   gatv2_backward_kernel: one pass along a plan (the dst plan with own = x_r, other = x_l, or the
//   src plan with own = x_l, other = x_r).  Edge-balanced like the segment reduce: a slot of L
//   lanes owns a chunk of chunk_len sorted edges; a lane's VB-byte vector stays inside one head, so
//   its g is one scalar gathered through eid per edge.  The own row is loaded when the row changes.
//   Rows that end inside the chunk are written in place; rows cut by a chunk boundary leave fp32
//   partials in segreduce.cu's two-slot layout, and its finish pass combines them in chunk order
//   (fp64) and zero-fills empty rows.  grad_att (dst pass only): each lane keeps its columns' sum
//   over all its chunks, the CTA adds its slots in slot order into a per-CTA partial, and
//   gatv2_att_finish_kernel sums those in CTA order in fp64.  No atomics: bit-reproducible.
//
// Roofline: HBM.  Bytes per edge = forward: F*s (x_l row) + H*s (logits) + 12 (gidx, erow, eid);
// backward, per pass: F*s (other row) + H*s (g, a sector per edge and head in the worst case) +
// 12; per row = 2 F*s (own row, grad row).
#include "segreduce.cuh"

namespace gno {

constexpr int kGatThreads = 256;
constexpr int kGatBatch = 4;  // sorted edges whose records, g values and rows are loaded before use
constexpr int kGatMaxCtasPerSm = 2048 / kGatThreads;  // resident threads per SM / CTA size

__device__ __forceinline__ float leaky(float z, float slope) { return z > 0.f ? z : z * slope; }

template <typename T, int VB>
__global__ void __launch_bounds__(256) gatv2_logits_kernel(const int32_t* __restrict__ erow,
                                                           const int32_t* __restrict__ gidx,
                                                           const int32_t* __restrict__ eid,
                                                           const char* __restrict__ xl,
                                                           const char* __restrict__ xr,
                                                           const char* __restrict__ att, T* __restrict__ out,
                                                           int64_t total, int H, int64_t row_bytes, int nvh,
                                                           float slope, bool narrow) {
  constexpr int EPV = VB / (int)sizeof(T);
  const int64_t t = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (t >= total) return;
  const int64_t k = narrow ? (int64_t)((uint32_t)t / (uint32_t)H) : t / H;
  const int h = (int)(t - k * H);
  const int64_t row = __ldg(erow + k);
  const int64_t s = gidx ? (int64_t)__ldg(gidx + k) : k;
  const int64_t e = eid ? (int64_t)__ldg(eid + k) : k;
  const int64_t hoff = (int64_t)h * nvh * VB;
  const char* lp = xl + s * row_bytes + hoff;
  const char* rp = xr + row * row_bytes + hoff;
  const char* ap = att + hoff;
  float acc = 0.f;
  for (int j = 0; j < nvh; ++j) {
    const Words<VB> a = ld_vec<VB>(lp + j * VB);
    const Words<VB> b = ld_vec<VB>(rp + j * VB);
    const Words<VB> w = ld_vec<VB>(ap + j * VB);
#pragma unroll
    for (int i = 0; i < EPV; ++i)
      acc = fmaf(elem<T, VB>(w, i), leaky(elem<T, VB>(a, i) + elem<T, VB>(b, i), slope), acc);
  }
  out[e * H + h] = DType<T>::from_f(acc);
}

struct GatBwdParams {
  const int32_t* erow;
  const int32_t* gidx;    // row of `other` per sorted edge (NULL = k)
  const int32_t* eid;     // original edge id per sorted edge (NULL = k)
  const char* own;        // [N, F]: the plan's rows
  const char* other;      // [other_rows, F]: the gathered rows
  const char* att;        // [F]
  const void* g;          // grad of the logits, [E, H] in original order
  void* out;              // grad of own [N, F], or NULL
  float* part;            // [2 * n_chunks, Fp] partials of rows cut by a chunk boundary
  float* att_part;        // [gridDim.x, F] per-CTA sums of grad_att, or NULL
  int64_t E, n_chunks, F, Fp, row_bytes;
  int H, head_c, nvec, L, chunk_len;
  float slope;
};

template <typename T, int VB, bool ATT>
__global__ void __launch_bounds__(kGatThreads) gatv2_backward_kernel(const GatBwdParams p) {
  constexpr int EPV = VB / (int)sizeof(T);
  __shared__ float s_att[ATT ? kGatThreads * EPV : 1];
  const int L = p.L, S = kGatThreads / L;
  const int slot = threadIdx.x / L, lane = threadIdx.x - slot * L;
  const int v = blockIdx.y * 32 + lane;
  const bool vact = v < p.nvec;
  const int64_t col = (int64_t)v * VB;
  const int h = vact ? v * EPV / p.head_c : 0;
  float w[EPV];
  {
    const Words<VB> a = vact ? ld_vec<VB>(p.att + col) : Words<VB>{};
#pragma unroll
    for (int i = 0; i < EPV; ++i) w[i] = elem<T, VB>(a, i);
  }
  float ga[ATT ? EPV : 1];
#pragma unroll
  for (int i = 0; i < (ATT ? EPV : 1); ++i) ga[i] = 0.f;
  const T* g = static_cast<const T*>(p.g) + h;
  const float slope = p.slope;

  for (int64_t grp = blockIdx.x; vact && grp * S < p.n_chunks; grp += gridDim.x) {
    const int64_t c = grp * S + slot;
    if (c >= p.n_chunks) break;
    const int64_t k0 = c * p.chunk_len;
    const int nv = (int)imin64(p.chunk_len, p.E - k0);
    int cur = __ldg(p.erow + k0);
    bool head = k0 > 0 && __ldg(p.erow + k0 - 1) == cur;
    float o[EPV], acc[EPV];
    auto load_own = [&](int row) {
      const Words<VB> r = ld_vec<VB>(p.own + (int64_t)row * p.row_bytes + col);
#pragma unroll
      for (int i = 0; i < EPV; ++i) {
        o[i] = elem<T, VB>(r, i);
        acc[i] = 0.f;
      }
    };
    auto flush = [&](bool tail) {
      if (p.out == nullptr) return;
      if (head || tail) {  // a chunk inside one row is both: it uses the head slot
        float* dp = p.part + (2 * c + (head ? 0 : 1)) * p.Fp + (int64_t)v * EPV;
#pragma unroll
        for (int i = 0; i < EPV; ++i) dp[i] = w[i] * acc[i];
      } else {
        Words<VB> r;
#pragma unroll
        for (int i = 0; i < EPV; ++i) set_elem<T, VB>(r, i, w[i] * acc[i]);
        st_vec<VB>(static_cast<char*>(p.out) + (int64_t)cur * p.row_bytes + col, r);
      }
    };
    auto step = [&](int row, float gv, const Words<VB>& x) {
      if (row != cur) {
        flush(false);
        head = false;
        cur = row;
        load_own(row);
      }
#pragma unroll
      for (int i = 0; i < EPV; ++i) {
        const float z = elem<T, VB>(x, i) + o[i];
        acc[i] += z > 0.f ? gv : gv * slope;
        if constexpr (ATT) ga[i] = fmaf(gv, leaky(z, slope), ga[i]);
      }
    };
    load_own(cur);
    int i = 0;
    for (; i + kGatBatch <= nv; i += kGatBatch) {
      int row[kGatBatch];
      float gv[kGatBatch];
      Words<VB> x[kGatBatch];
#pragma unroll
      for (int u = 0; u < kGatBatch; ++u) {
        const int64_t k = k0 + i + u;
        row[u] = __ldg(p.erow + k);
        const int64_t s = p.gidx ? (int64_t)__ldg(p.gidx + k) : k;
        const int64_t e = p.eid ? (int64_t)__ldg(p.eid + k) : k;
        gv[u] = DType<T>::to_f(g[e * p.H]);
        x[u] = ld_vec<VB>(p.other + s * p.row_bytes + col);
      }
#pragma unroll
      for (int u = 0; u < kGatBatch; ++u) step(row[u], gv[u], x[u]);
    }
    for (; i < nv; ++i) {
      const int64_t k = k0 + i;
      const int64_t s = p.gidx ? (int64_t)__ldg(p.gidx + k) : k;
      const int64_t e = p.eid ? (int64_t)__ldg(p.eid + k) : k;
      step(__ldg(p.erow + k), DType<T>::to_f(g[e * p.H]), ld_vec<VB>(p.other + s * p.row_bytes + col));
    }
    flush(k0 + nv < p.E && __ldg(p.erow + k0 + nv) == cur);
  }

  if constexpr (ATT) {
#pragma unroll
    for (int i = 0; i < EPV; ++i) s_att[threadIdx.x * EPV + i] = ga[i];
    __syncthreads();
    if (slot == 0 && vact) {
#pragma unroll
      for (int i = 0; i < EPV; ++i) {
        float sum = 0.f;
        for (int q = 0; q < S; ++q) sum += s_att[(q * L + lane) * EPV + i];
        p.att_part[(int64_t)blockIdx.x * p.F + (int64_t)v * EPV + i] = sum;
      }
    }
  }
}

// grad_att[f] = the per-CTA partials summed in CTA order in fp64.
__global__ void __launch_bounds__(256) gatv2_att_finish_kernel(const float* __restrict__ att_part, int n_parts,
                                                               int64_t F, float* __restrict__ grad_att) {
  const int64_t f = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (f >= F) return;
  double s = 0.0;
#pragma unroll 8
  for (int b = 0; b < n_parts; ++b) s += (double)att_part[(int64_t)b * F + f];
  grad_att[f] = (float)s;
}

static int gat_dtype_size(int dtype) { return dtype == GNO_F32 ? 4 : 2; }

static int gat_sizes_ok(const gno_csr* g, int64_t H, int64_t F, int64_t other_rows, int dtype, const char* fn) {
  GNO_CHECK_ARG(g != nullptr, "%s: graph is NULL", fn);
  GNO_CHECK_ARG(dtype == GNO_F32 || dtype == GNO_F16 || dtype == GNO_BF16, "%s: unknown dtype %d", fn, dtype);
  GNO_CHECK_ARG(H > 0 && H < (int64_t(1) << 20) && F > 0 && F % H == 0 && F < (int64_t(1) << 24) && other_rows >= 0 &&
                    g->N >= 0 && g->E >= 0 && g->E < (int64_t(1) << 31),
                "%s: bad sizes H=%lld F=%lld rows=%lld N=%lld E=%lld", fn, (long long)H, (long long)F,
                (long long)other_rows, (long long)g->N, (long long)g->E);
  GNO_CHECK_ARG(g->chunk_len >= 32 && g->chunk_len % 32 == 0 && g->chunk_len <= (1 << 20),
                "%s: chunk_len must be a multiple of 32", fn);
  return GNO_OK;
}

template <typename T>
static int launch_logits(const gno_csr* g, const void* xl, const void* xr, const void* att, int64_t H, int64_t F,
                         float slope, void* out, cudaStream_t s) {
  const int es = (int)sizeof(T);
  const int64_t total = g->E * H;
  const int vb = head_vector_bytes(F / H * es, (uintptr_t)xl | (uintptr_t)xr | (uintptr_t)att, es);
  const int nvh = (int)(F / H * es / vb);
  const unsigned blocks = (unsigned)ceil_div(total, 256);
  const bool narrow = total < (int64_t(1) << 32);
  const char *l = static_cast<const char*>(xl), *r = static_cast<const char*>(xr), *a = static_cast<const char*>(att);
  T* o = static_cast<T*>(out);
  switch (vb) {
    case 16: gatv2_logits_kernel<T, 16><<<blocks, 256, 0, s>>>(g->erow, g->gidx, g->eid, l, r, a, o, total, (int)H, F * es, nvh, slope, narrow); break;
    case 8: gatv2_logits_kernel<T, 8><<<blocks, 256, 0, s>>>(g->erow, g->gidx, g->eid, l, r, a, o, total, (int)H, F * es, nvh, slope, narrow); break;
    case 4: gatv2_logits_kernel<T, 4><<<blocks, 256, 0, s>>>(g->erow, g->gidx, g->eid, l, r, a, o, total, (int)H, F * es, nvh, slope, narrow); break;
    default:
      if constexpr (sizeof(T) == 2) {
        gatv2_logits_kernel<T, 2><<<blocks, 256, 0, s>>>(g->erow, g->gidx, g->eid, l, r, a, o, total, (int)H, F * es, nvh, slope, narrow);
        break;
      }
      return fail(GNO_ERR_INVALID, "gno_gatv2_logits: bad vector width %d", vb);
  }
  GNO_LAUNCHED("gatv2_logits_kernel");
  return GNO_OK;
}

// Grid: column tiles of 32 vectors in y; in x, as many CTAs as fit on the device at once, each
// walking groups of chunks (so the grad_att partials number at most kNumSMs * kGatMaxCtasPerSm).
template <typename T, int VB, bool ATT>
static int launch_backward_vb(const GatBwdParams& p, int ncoltiles, int* gx, cudaStream_t s) {
  static int per_sm = -1;
  if (per_sm < 0) {
    int n = 0;
    GNO_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, gatv2_backward_kernel<T, VB, ATT>, kGatThreads, 0));
    per_sm = (int)imax64(1, imin64(n, kGatMaxCtasPerSm));
  }
  const int64_t groups = ceil_div(p.n_chunks, kGatThreads / p.L);
  *gx = (int)imin64(groups, imax64(1, (int64_t)kNumSMs * per_sm / ncoltiles));
  gatv2_backward_kernel<T, VB, ATT><<<dim3((unsigned)*gx, (unsigned)ncoltiles), kGatThreads, 0, s>>>(p);
  GNO_LAUNCHED("gatv2_backward_kernel");
  return GNO_OK;
}

template <typename T, bool ATT>
static int launch_backward(const GatBwdParams& p, int vb, int ncoltiles, int* gx, cudaStream_t s) {
  switch (vb) {
    case 16: return launch_backward_vb<T, 16, ATT>(p, ncoltiles, gx, s);
    case 8: return launch_backward_vb<T, 8, ATT>(p, ncoltiles, gx, s);
    case 4: return launch_backward_vb<T, 4, ATT>(p, ncoltiles, gx, s);
    default:
      if constexpr (sizeof(T) == 2) return launch_backward_vb<T, 2, ATT>(p, ncoltiles, gx, s);
  }
  return fail(GNO_ERR_INVALID, "gno_gatv2_logits_backward: bad vector width %d", vb);
}

template <typename T>
static int dispatch_backward(const GatBwdParams& p, int vb, int ncoltiles, int* gx, cudaStream_t s) {
  return p.att_part ? launch_backward<T, true>(p, vb, ncoltiles, gx, s)
                    : launch_backward<T, false>(p, vb, ncoltiles, gx, s);
}

}  // namespace gno

using namespace gno;

extern "C" {

int gno_gatv2_logits(const gno_csr* g, const void* x_l, int64_t xl_rows, const void* x_r, const void* att,
                     int64_t H, int64_t F, double negative_slope, void* out, int dtype, gno_stream_t stream) {
  const char* fn = "gno_gatv2_logits";
  if (int rc = gat_sizes_ok(g, H, F, xl_rows, dtype, fn)) return rc;
  if (g->E == 0) return GNO_OK;
  GNO_CHECK_ARG(g->erow && x_l && x_r && att && out, "%s: NULL buffer", fn);
  const int es = gat_dtype_size(dtype);
  GNO_CHECK_ARG((((uintptr_t)x_l | (uintptr_t)x_r | (uintptr_t)att | (uintptr_t)out) % es) == 0,
                "%s: buffers not aligned to the element size", fn);
  cudaStream_t s = (cudaStream_t)stream;
  const float slope = (float)negative_slope;
  switch (dtype) {
    case GNO_F32: return launch_logits<float>(g, x_l, x_r, att, H, F, slope, out, s);
    case GNO_F16: return launch_logits<__half>(g, x_l, x_r, att, H, F, slope, out, s);
    default: return launch_logits<__nv_bfloat16>(g, x_l, x_r, att, H, F, slope, out, s);
  }
}

int gno_gatv2_logits_backward_workspace(const gno_csr* g, int64_t H, int64_t F, int with_grad_own,
                                        int with_grad_att, size_t* bytes) {
  const char* fn = "gno_gatv2_logits_backward_workspace";
  GNO_CHECK_ARG(bytes != nullptr, "%s: NULL argument", fn);
  if (int rc = gat_sizes_ok(g, H, F, 0, GNO_F32, fn)) return rc;
  WorkspaceSizer sz;
  const int64_t n_chunks = ceil_div(g->E, g->chunk_len);
  if (n_chunks > 0) {
    if (with_grad_own) sz.take<float>((size_t)(2 * n_chunks * ((F + 7) / 8 * 8)));
    if (with_grad_att) sz.take<float>((size_t)((int64_t)kNumSMs * kGatMaxCtasPerSm * F));
  }
  *bytes = sz.total();
  return GNO_OK;
}

int gno_gatv2_logits_backward(const gno_csr* g, const void* own, const void* other, int64_t other_rows,
                              const void* att, const void* grad_logits, int64_t H, int64_t F,
                              double negative_slope, void* grad_own, float* grad_att, int dtype, void* wsp,
                              size_t ws_bytes, gno_stream_t stream) {
  const char* fn = "gno_gatv2_logits_backward";
  if (int rc = gat_sizes_ok(g, H, F, other_rows, dtype, fn)) return rc;
  if (g->E == 0) return GNO_OK;
  GNO_CHECK_ARG(g->erow && g->rowptr && own && other && att && grad_logits && (grad_own || grad_att),
                "%s: NULL buffer", fn);
  GNO_CHECK_ARG(grad_own == nullptr || ((g->n_span == 0 || g->srow) && (g->n_empty == 0 || g->zrow)),
                "%s: row lists missing", fn);
  const int es = gat_dtype_size(dtype);
  const uintptr_t al = (uintptr_t)own | (uintptr_t)other | (uintptr_t)att | (uintptr_t)grad_own;
  GNO_CHECK_ARG(((al | (uintptr_t)grad_logits) % es) == 0, "%s: buffers not aligned to the element size", fn);
  if (wsp == nullptr) return fail(GNO_ERR_WORKSPACE, "%s: workspace is NULL", fn);

  GatBwdParams p;
  p.erow = g->erow;
  p.gidx = g->gidx;
  p.eid = g->eid;
  p.own = static_cast<const char*>(own);
  p.other = static_cast<const char*>(other);
  p.att = static_cast<const char*>(att);
  p.g = grad_logits;
  p.out = grad_own;
  p.E = g->E;
  p.n_chunks = ceil_div(g->E, g->chunk_len);
  p.F = F;
  p.Fp = (F + 7) / 8 * 8;
  p.row_bytes = F * es;
  p.H = (int)H;
  p.head_c = (int)(F / H);
  p.chunk_len = (int)g->chunk_len;
  p.slope = (float)negative_slope;
  Workspace ws(wsp, ws_bytes);
  p.part = grad_own ? ws.take<float>((size_t)(2 * p.n_chunks * p.Fp)) : nullptr;
  p.att_part = grad_att ? ws.take<float>((size_t)((int64_t)kNumSMs * kGatMaxCtasPerSm * F)) : nullptr;
  if (!ws.ok()) return fail(GNO_ERR_WORKSPACE, "%s: workspace too small (%zu < %zu)", fn, ws_bytes, ws.off);

  const int vb = head_vector_bytes(F / H * es, al, es);
  p.nvec = (int)(F * es / vb);
  const int ncoltiles = (p.nvec + 31) / 32;
  int L = 1;
  while (L < p.nvec && L < 32) L <<= 1;
  p.L = L;
  cudaStream_t s = (cudaStream_t)stream;
  int gx = 0;
  int rc;
  switch (dtype) {
    case GNO_F32: rc = dispatch_backward<float>(p, vb, ncoltiles, &gx, s); break;
    case GNO_F16: rc = dispatch_backward<__half>(p, vb, ncoltiles, &gx, s); break;
    default: rc = dispatch_backward<__nv_bfloat16>(p, vb, ncoltiles, &gx, s); break;
  }
  if (rc) return rc;
  if (grad_own) {
    // the finish pass of a SUM over the same partial layout: rows cut by a chunk boundary, empty rows
    SegParams q = {};
    q.out = grad_own;
    q.part_val = p.part;
    q.rowptr = g->rowptr;
    q.srow = g->srow;
    q.zrow = g->zrow;
    q.N = g->N;
    q.E = g->E;
    q.n_chunks = p.n_chunks;
    q.n_span = g->n_span;
    q.n_empty = g->n_empty;
    q.F = F;
    q.Fp = p.Fp;
    q.ldx_bytes = q.ldo_bytes = F * es;
    q.chunk_len = p.chunk_len;
    if (int rf = seg_finish_sum(q, dtype, true, s)) return rf;
  }
  if (grad_att) {
    gatv2_att_finish_kernel<<<(unsigned)ceil_div(F, 256), 256, 0, s>>>(p.att_part, gx, F, grad_att);
    GNO_LAUNCHED("gatv2_att_finish_kernel");
  }
  return GNO_OK;
}

}  // extern "C"
