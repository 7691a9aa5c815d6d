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

// ---- The whole GATv2 message passing in one pass (gno_gatv2_attention) ----------------------
//
//   a[e, h]     = sum_c att[h, c] * leaky_relu(x_l[src[e], h, c] + x_r[dst[e], h, c])
//   alpha[e, h] = exp(a - m[dst, h]) / (sum_{row} exp(a - m) + eps)        (gno_segment_softmax's rule)
//   out[i, h,:] = sum_{e: dst[e] = i} alpha[e, h] * x_l[src[e], h, :]
//
// gatv2_attention_kernel walks the dst plan edge-balanced like gatv2_backward_kernel: a slot of L
// lanes owns a chunk of chunk_len sorted edges.  Within the slot, P lanes (a power of two) cover
// one head, NV vectors of VB bytes each (vector q of lane j is the head's vector j + q*P), and the
// slot covers HT = L / P heads; more heads go to column tiles in blockIdx.y.  Per edge a lane loads
// its x_l[src] vectors once, forms z = x_l + x_r in fp32 (the row's x_r is loaded when the row
// changes), and the head's logit is a butterfly shuffle sum over its P lanes (the same value, bit
// for bit, in every lane).  The head's running (m, s) follows softmax_stats_kernel's online form,
// and the fp32 accumulator of p * x_l is rescaled by exp(m_old - m_new) when the max grows, so the
// loaded vector serves both the logit and the weighted sum.  A row that ends inside the chunk is
// written as acc / (s + eps); rows cut by a chunk boundary leave (m, s) and acc in the two-slot
// layout, and gatv2_attention_finish_kernel combines them in chunk order in fp64 and fills empty
// rows.  Neither the [E, H] logits nor alpha are written; the fp32 row statistics m and
// d = s + eps ([N, H]) are kept for the backward.  No atomics: bit-reproducible.
//
// gatv2_attention_backward_kernel is the dst pass of the backward, on the same walk.  With
// D[i, h] = sum_c g[i, h, c] * out[i, h, c], it recomputes a and alpha from (m, d) and forms
//   da[e, h] = alpha * (g[dst] . x_l[src] - D[dst])  = alpha * sum_c g[dst, h, c] * (x_l[src, h, c] - out[dst, h, c])
// with one shuffle sum per edge (each lane holds its part of D, taken when the row changes):
//   grad_x_r[i, f] = att[f] * sum_{e in row i} da * leaky_relu'(z)   (chunk partials + seg_finish_sum)
//   grad_att[f]    = sum_e da * leaky_relu(z)                        (CTA partials + gatv2_att_finish_kernel)
// and writes da and alpha [E, H] in original edge order for the src pass, which reuses
// gno_gatv2_logits_backward (logit part of grad_x_l) and gno_segment_reduce_heads (alpha * g[dst]).
//
// Roofline: HBM.  Bytes per edge = forward: F*s (x_l row) + 8 (erow, gidx); per row 2 F*s (x_r, out)
// + 8 H (m, d).  Backward dst pass: F*s + 12 per edge + 2 H*s (da, alpha); per row 4 F*s (x_r, g,
// out, grad_x_r) + 8 H.

constexpr int kGaMaxVecs = 4;  // vectors per lane: a head may span at most 32 * 4 vectors

struct GatAttnParams {
  const int32_t* erow;
  const int32_t* gidx;     // src row per sorted edge
  const int32_t* eid;      // original edge id per sorted edge (NULL = k)
  const int64_t* rowptr;
  const int32_t* srow;
  const int32_t* zrow;
  const char* xl;          // [xl_rows, F]
  const char* xr;          // [N, F]
  const char* att;         // [F]
  const char* out_in;      // backward: the forward's out [N, F]
  const void* g;           // backward: grad of out [N, F]
  void* out;               // forward: out [N, F]; backward: grad_x_r [N, F] or NULL
  float* m;                // [N, H] row max (after the empty-row rule)
  float* d;                // [N, H] sum of exp(a - m) + eps
  void* da;                // backward: [E, H] grad of the logits, original order (or NULL)
  void* alpha;             // backward: [E, H] attention weights, original order (or NULL)
  float* part;             // [2 * n_chunks, Fp] chunk partials of acc
  float2* part_ms;         // forward: [2 * n_chunks, H] chunk partials of (m, s)
  float* att_part;         // backward: [gridDim.x, F] per-CTA sums of grad_att, or NULL
  int64_t N, E, n_chunks, n_span, n_empty, F, Fp, row_bytes, head_bytes;
  int H, head_c, nvh, P, L, HT, chunk_len;
  float slope, eps;
};

// Lane geometry shared by both kernels: the slot, the head and the byte / element offsets of the
// lane's vectors.
template <int VB, int NV, typename T>
struct GaLane {
  int slot, lane, h;
  bool act[NV];
  int64_t col[NV];     // byte offset in a row
  int64_t f[NV];       // element offset in a row
  __device__ __forceinline__ GaLane(const GatAttnParams& p) {
    constexpr int EPV = VB / (int)sizeof(T);
    slot = threadIdx.x / p.L;
    lane = threadIdx.x - slot * p.L;
    const int hh = lane / p.P, j = lane - hh * p.P;
    h = blockIdx.y * p.HT + hh;
    const bool hact = h < p.H;
#pragma unroll
    for (int q = 0; q < NV; ++q) {
      const int vi = j + q * p.P;
      act[q] = hact && vi < p.nvh;
      col[q] = act[q] ? (int64_t)h * p.head_bytes + (int64_t)vi * VB : 0;
      f[q] = act[q] ? (int64_t)h * p.head_c + (int64_t)vi * EPV : 0;
    }
    if (!hact) h = 0;
  }
};

// 1/d (MUFU.RCP, within an ulp; d >= eps is never subnormal) and a / d from it with one Newton
// step on a * r: the quotient to within an ulp, inline, where __fdiv_rn and __frcp_rn call a slow
// path whose stack frame the walk would spill.
__device__ __forceinline__ float ga_rcp(float d) {
  float r;
  asm("rcp.approx.f32 %0, %1;" : "=f"(r) : "f"(d));
  return r;
}
__device__ __forceinline__ float ga_div(float a, float d, float r) {
  const float q = a * r;
  return isfinite(q) ? fmaf(fmaf(-q, d, a), r, q) : q;
}

// Sum over the P lanes of a head (butterfly: commutative adds, every lane gets the same bits).
// Every lane of the warp calls it once per step of the walk: the walk of every slot takes
// chunk_len steps, the steps past a chunk's end (only the last chunk, and slots past it) idle.
__device__ __forceinline__ float ga_head_sum(float v, int P) {
  for (int o = 1; o < P; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <typename T, int VB, int NV>
__device__ __forceinline__ void ga_load(const GaLane<VB, NV, T>& ln, const char* base, float (&r)[NV][VB / sizeof(T)],
                                        bool ok = true) {
  constexpr int EPV = VB / (int)sizeof(T);
#pragma unroll
  for (int q = 0; q < NV; ++q) {
    const Words<VB> w = ok && ln.act[q] ? ld_vec<VB>(base + ln.col[q]) : Words<VB>{};
#pragma unroll
    for (int i = 0; i < EPV; ++i) r[q][i] = elem<T, VB>(w, i);
  }
}

// Edges per batch whose records and x_l vectors are loaded before use (the sizes that compile
// spill-free: the backward holds three more row vectors per lane).
template <int NV, bool BWD>
struct GaBatch {
  static constexpr int U = NV == 1 ? 4 : (NV == 2 && !BWD) ? 2 : 1;
};

template <typename T, int VB, int NV>
__global__ void __launch_bounds__(kGatThreads) gatv2_attention_kernel(const GatAttnParams p) {
  constexpr int EPV = VB / (int)sizeof(T);
  constexpr int U = GaBatch<NV, false>::U;
  const GaLane<VB, NV, T> ln(p);
  const int64_t c = (int64_t)blockIdx.x * (kGatThreads / p.L) + ln.slot;
  const bool live = c < p.n_chunks;
  float w[NV][EPV], xr[NV][EPV], acc[NV][EPV];
  ga_load<T, VB, NV>(ln, p.att, w);
  const float slope = p.slope, lowest = DType<T>::lowest();
  const int64_t k0 = c * p.chunk_len;
  const int nv = live ? (int)imin64(p.chunk_len, p.E - k0) : 0;
  int cur = live ? __ldg(p.erow + k0) : 0;
  bool head = live && k0 > 0 && __ldg(p.erow + k0 - 1) == cur;
  const int next = live && k0 + nv < p.E ? __ldg(p.erow + k0 + nv) : -1;  // the row after the chunk
  float m = lowest, s = 0.f;
  auto reset = [&](int row) {
    ga_load<T, VB, NV>(ln, p.xr + (int64_t)row * p.row_bytes, xr, live);
    m = lowest;
    s = 0.f;
#pragma unroll
    for (int q = 0; q < NV; ++q)
#pragma unroll
      for (int i = 0; i < EPV; ++i) acc[q][i] = 0.f;
  };
  auto flush = [&](bool tail) {
    if (head || tail) {  // a chunk inside one row is both: it uses the head slot
      const int64_t sl = 2 * c + (head ? 0 : 1);
      if (ln.lane % p.P == 0 && ln.act[0]) p.part_ms[sl * p.H + ln.h] = make_float2(m, s);
#pragma unroll
      for (int q = 0; q < NV; ++q) {
        if (!ln.act[q]) continue;
        float* dp = p.part + sl * p.Fp + ln.f[q];
#pragma unroll
        for (int i = 0; i < EPV; ++i) dp[i] = acc[q][i];
      }
    } else {
      const float mf = (m == lowest) ? 0.f : m;  // no logit won: torch_scatter's empty value
      const float sc = mf != m ? expf(m - mf) : 1.f;
      const float d = s * sc + p.eps, r = ga_rcp(d);
      if (ln.lane % p.P == 0 && ln.act[0]) {
        p.m[(int64_t)cur * p.H + ln.h] = mf;
        p.d[(int64_t)cur * p.H + ln.h] = d;
      }
#pragma unroll
      for (int q = 0; q < NV; ++q) {
        if (!ln.act[q]) continue;
        Words<VB> o;
#pragma unroll
        for (int i = 0; i < EPV; ++i) set_elem<T, VB>(o, i, ga_div(acc[q][i] * sc, d, r));
        st_vec<VB>(static_cast<char*>(p.out) + (int64_t)cur * p.row_bytes + ln.col[q], o);
      }
    }
  };
  auto step = [&](bool ok, int row, const float (&x)[NV][EPV]) {
    if (ok && row != cur) {
      flush(false);
      head = false;
      cur = row;
      reset(row);
    }
    float a = 0.f;
#pragma unroll
    for (int q = 0; q < NV; ++q)
#pragma unroll
      for (int i = 0; i < EPV; ++i) a = fmaf(w[q][i], leaky(x[q][i] + xr[q][i], slope), a);
    a = ga_head_sum(a, p.P);
    if (!ok) return;
    float pe, sc = 1.f;
    if (a > m) {  // strict: NaN never wins, and its exp makes the row's sum NaN below
      // the winner's own term is exp(a - a): 1, or NaN for +inf (PyG's exp(inf - inf))
      sc = expf(m - a);
      pe = a == INFINITY ? __int_as_float(0x7fffffff) : 1.f;
      m = a;
    } else {
      pe = expf(a - m);
    }
    s = fmaf(s, sc, pe);
#pragma unroll
    for (int q = 0; q < NV; ++q)
#pragma unroll
      for (int i = 0; i < EPV; ++i) acc[q][i] = fmaf(acc[q][i], sc, pe * x[q][i]);
  };
  reset(cur);
  for (int i = 0; i < p.chunk_len; i += U) {
    int row[U];
    float x[U][NV][EPV];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t k = k0 + i + u;
      const bool ok = i + u < nv;
      row[u] = ok ? __ldg(p.erow + k) : cur;
      ga_load<T, VB, NV>(ln, p.xl + (ok ? (int64_t)__ldg(p.gidx + k) * p.row_bytes : 0), x[u], ok);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) step(i + u < nv, row[u], x[u]);
  }
  if (live) flush(next == cur);
}

// Rows cut by a chunk boundary: the tail slot of the first chunk, then the head slot of every
// later chunk, combined in chunk order in fp64 (m = max, s and acc rescaled by e^(m_k - m)); one
// thread per (row, element).  Then empty rows: out 0, m 0, d eps.
template <typename T>
__global__ void __launch_bounds__(256) gatv2_attention_finish_kernel(const GatAttnParams p) {
  const int64_t t = (int64_t)blockIdx.x * 256 + threadIdx.x;
  const int64_t n_a = p.n_span * p.F, n_z = p.n_empty * p.F;
  T* out = static_cast<T*>(p.out);
  if (t < n_a) {
    const int64_t r = t / p.F, f = t - r * p.F;
    const int h = (int)(f / p.head_c);
    const int64_t row = p.srow[r];
    const int64_t kb = p.rowptr[row], ke = p.rowptr[row + 1];
    const int64_t ca = kb / p.chunk_len, cb = (ke - 1) / p.chunk_len;
    const float2 first = p.part_ms[(2 * ca + 1) * p.H + h];
    double m = first.x, s = first.y, a = p.part[(2 * ca + 1) * p.Fp + f];
    for (int64_t c = ca + 1; c <= cb; ++c) {
      const float2 q = p.part_ms[2 * c * p.H + h];
      const double qa = p.part[2 * c * p.Fp + f];
      const double mn = q.x > m ? (double)q.x : m;
      const double e0 = exp(m - mn), e1 = exp((double)q.x - mn);
      s = s * e0 + (double)q.y * e1;
      a = a * e0 + qa * e1;
      m = mn;
    }
    const float lowest = DType<T>::lowest();
    const float mf = ((float)m == lowest) ? 0.f : (float)m;
    const double sc = exp(m - (double)mf);
    const float d = (float)(s * sc) + p.eps;
    out[row * p.F + f] = DType<T>::from_f(__fdiv_rn((float)(a * sc), d));
    if (f % p.head_c == 0) {
      p.m[row * p.H + h] = mf;
      p.d[row * p.H + h] = d;
    }
  } else if (t < n_a + n_z) {
    const int64_t r = (t - n_a) / p.F, f = (t - n_a) - r * p.F;
    const int64_t row = p.zrow[r];
    out[row * p.F + f] = DType<T>::from_f(0.f);
    if (f % p.head_c == 0) {
      p.m[row * p.H + f / p.head_c] = 0.f;
      p.d[row * p.H + f / p.head_c] = p.eps;
    }
  }
}

template <typename T, int VB, int NV, bool ATT>
__global__ void __launch_bounds__(kGatThreads) gatv2_attention_backward_kernel(const GatAttnParams p) {
  constexpr int EPV = VB / (int)sizeof(T);
  constexpr int U = GaBatch<NV, true>::U;
  __shared__ float s_att[ATT ? kGatThreads * NV * EPV : 1];
  const GaLane<VB, NV, T> ln(p);
  const int S = kGatThreads / p.L;
  float w[NV][EPV], xr[NV][EPV], gr[NV][EPV], acc[NV][EPV], ga[ATT ? NV : 1][EPV];
  ga_load<T, VB, NV>(ln, p.att, w);
#pragma unroll
  for (int q = 0; q < (ATT ? NV : 1); ++q)
#pragma unroll
    for (int i = 0; i < EPV; ++i) ga[q][i] = 0.f;
  const float slope = p.slope;
  const int64_t ld_g = p.row_bytes;

  for (int64_t grp = blockIdx.x; grp * S < p.n_chunks; grp += gridDim.x) {
    const int64_t c = grp * S + ln.slot;
    const bool live = c < p.n_chunks;
    const int64_t k0 = c * p.chunk_len;
    const int nv = live ? (int)imin64(p.chunk_len, p.E - k0) : 0;
    int cur = live ? __ldg(p.erow + k0) : 0;
    bool head = live && k0 > 0 && __ldg(p.erow + k0 - 1) == cur;
    const int next = live && k0 + nv < p.E ? __ldg(p.erow + k0 + nv) : -1;
    float rm = 0.f, rd = 1.f, rr = 1.f, pd = 0.f;  // the row's m, d, 1/d and this lane's part of D
    auto load_row = [&](int row) {
      ga_load<T, VB, NV>(ln, p.xr + (int64_t)row * p.row_bytes, xr, live);
      ga_load<T, VB, NV>(ln, static_cast<const char*>(p.g) + (int64_t)row * ld_g, gr, live);
      float o[NV][EPV];
      ga_load<T, VB, NV>(ln, p.out_in + (int64_t)row * p.row_bytes, o, live);
      pd = 0.f;
#pragma unroll
      for (int q = 0; q < NV; ++q)
#pragma unroll
        for (int i = 0; i < EPV; ++i) {
          pd = fmaf(gr[q][i], o[q][i], pd);
          acc[q][i] = 0.f;
        }
      rm = live ? p.m[(int64_t)row * p.H + ln.h] : 0.f;
      rd = live ? p.d[(int64_t)row * p.H + ln.h] : 1.f;
      rr = ga_rcp(rd);
    };
    auto flush = [&](bool tail) {
      if (p.out == nullptr) return;
      if (head || tail) {
        float* dp = p.part + (2 * c + (head ? 0 : 1)) * p.Fp;
#pragma unroll
        for (int q = 0; q < NV; ++q) {
          if (!ln.act[q]) continue;
#pragma unroll
          for (int i = 0; i < EPV; ++i) dp[ln.f[q] + i] = w[q][i] * acc[q][i];
        }
      } else {
#pragma unroll
        for (int q = 0; q < NV; ++q) {
          if (!ln.act[q]) continue;
          Words<VB> r;
#pragma unroll
          for (int i = 0; i < EPV; ++i) set_elem<T, VB>(r, i, w[q][i] * acc[q][i]);
          st_vec<VB>(static_cast<char*>(p.out) + (int64_t)cur * p.row_bytes + ln.col[q], r);
        }
      }
    };
    auto step = [&](bool ok, int row, int64_t e, const float (&x)[NV][EPV]) {
      if (ok && row != cur) {
        flush(false);
        head = false;
        cur = row;
        load_row(row);
      }
      float a = 0.f, gd = -pd;
#pragma unroll
      for (int q = 0; q < NV; ++q)
#pragma unroll
        for (int i = 0; i < EPV; ++i) {
          a = fmaf(w[q][i], leaky(x[q][i] + xr[q][i], slope), a);
          gd = fmaf(gr[q][i], x[q][i], gd);
        }
      a = ga_head_sum(a, p.P);
      gd = ga_head_sum(gd, p.P);
      if (!ok) return;
      const float al = ga_div(expf(a - rm), rd, rr);
      const float da = al * gd;
      if (ln.lane % p.P == 0 && ln.act[0] && p.da) {
        static_cast<T*>(p.da)[e * p.H + ln.h] = DType<T>::from_f(da);
        static_cast<T*>(p.alpha)[e * p.H + ln.h] = DType<T>::from_f(al);
      }
#pragma unroll
      for (int q = 0; q < NV; ++q)
#pragma unroll
        for (int i = 0; i < EPV; ++i) {
          const float z = x[q][i] + xr[q][i];
          acc[q][i] += z > 0.f ? da : da * slope;
          if constexpr (ATT) ga[q][i] = fmaf(da, leaky(z, slope), ga[q][i]);
        }
    };
    load_row(cur);
    for (int i = 0; i < p.chunk_len; i += U) {
      int row[U];
      int64_t e[U];
      float x[U][NV][EPV];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t k = k0 + i + u;
        const bool ok = i + u < nv;
        row[u] = ok ? __ldg(p.erow + k) : cur;
        e[u] = ok && p.eid ? (int64_t)__ldg(p.eid + k) : k;
        ga_load<T, VB, NV>(ln, p.xl + (ok ? (int64_t)__ldg(p.gidx + k) * p.row_bytes : 0), x[u], ok);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) step(i + u < nv, row[u], e[u], x[u]);
    }
    if (live) flush(next == cur);
  }

  if constexpr (ATT) {
#pragma unroll
    for (int q = 0; q < NV; ++q)
#pragma unroll
      for (int i = 0; i < EPV; ++i) s_att[(threadIdx.x * NV + q) * EPV + i] = ga[q][i];
    __syncthreads();
    if (ln.slot == 0) {
#pragma unroll
      for (int q = 0; q < NV; ++q) {
        if (!ln.act[q]) continue;
#pragma unroll
        for (int i = 0; i < EPV; ++i) {
          float sum = 0.f;
          for (int r = 0; r < S; ++r) sum += s_att[((r * p.L + ln.lane) * NV + q) * EPV + i];
          p.att_part[(int64_t)blockIdx.x * p.F + ln.f[q] + i] = sum;
        }
      }
    }
  }
}

// Lane geometry for a head of nvh vectors: P lanes per head, NV vectors per lane, L lanes per slot
// holding HT heads, and the column tiles over the heads.  0 when a head is too wide.
struct GaShape {
  int vb, nvh, P, NV, L, HT, ncoltiles;
};

static int ga_shape(int64_t H, int64_t F, int es, uintptr_t align, GaShape* sh) {
  const int64_t head_bytes = F / H * es;
  sh->vb = head_vector_bytes(head_bytes, align, es);
  const int64_t nvh = head_bytes / sh->vb;
  if (nvh > 32 * kGaMaxVecs) return 0;
  sh->nvh = (int)nvh;
  int P = 1;
  while (P < nvh && P < 32) P <<= 1;
  sh->P = P;
  const int64_t nv = ceil_div(nvh, P);
  sh->NV = nv == 1 ? 1 : nv == 2 ? 2 : 4;
  int hp = 1;
  while (hp < H && hp * P < 32) hp <<= 1;
  sh->L = hp * P;
  sh->HT = hp;
  sh->ncoltiles = (int)ceil_div(H, hp);
  return 1;
}

static void ga_fill(GatAttnParams& p, const gno_csr* g, const GaShape& sh, int64_t H, int64_t F, int es,
                    double slope) {
  p.erow = g->erow;
  p.gidx = g->gidx;
  p.eid = g->eid;
  p.rowptr = g->rowptr;
  p.srow = g->srow;
  p.zrow = g->zrow;
  p.N = g->N;
  p.E = g->E;
  p.n_chunks = ceil_div(g->E, g->chunk_len);
  p.n_span = g->n_span;
  p.n_empty = g->n_empty;
  p.F = F;
  p.Fp = (F + 7) / 8 * 8;
  p.row_bytes = F * es;
  p.head_bytes = F / H * es;
  p.H = (int)H;
  p.head_c = (int)(F / H);
  p.nvh = sh.nvh;
  p.P = sh.P;
  p.L = sh.L;
  p.HT = sh.HT;
  p.chunk_len = (int)g->chunk_len;
  p.slope = (float)slope;
}

template <typename T, int VB, int NV>
static int ga_forward_vb(const GatAttnParams& p, const GaShape& sh, cudaStream_t s) {
  const unsigned gx = (unsigned)ceil_div(p.n_chunks, kGatThreads / p.L);
  gatv2_attention_kernel<T, VB, NV><<<dim3(gx, (unsigned)sh.ncoltiles), kGatThreads, 0, s>>>(p);
  GNO_LAUNCHED("gatv2_attention_kernel");
  return GNO_OK;
}

template <typename T, int VB>
static int ga_forward_nv(const GatAttnParams& p, const GaShape& sh, cudaStream_t s) {
  switch (sh.NV) {
    case 1: return ga_forward_vb<T, VB, 1>(p, sh, s);
    case 2: return ga_forward_vb<T, VB, 2>(p, sh, s);
    default: return ga_forward_vb<T, VB, 4>(p, sh, s);
  }
}

template <typename T>
static int ga_forward(const GatAttnParams& p, const GaShape& sh, cudaStream_t s) {
  int rc;
  switch (sh.vb) {
    case 16: rc = ga_forward_nv<T, 16>(p, sh, s); break;
    case 8: rc = ga_forward_nv<T, 8>(p, sh, s); break;
    case 4: rc = ga_forward_nv<T, 4>(p, sh, s); break;
    default:
      if constexpr (sizeof(T) == 2) {
        rc = ga_forward_nv<T, 2>(p, sh, s);
        break;
      }
      return fail(GNO_ERR_INVALID, "gno_gatv2_attention: bad vector width %d", sh.vb);
  }
  if (rc) return rc;
  const int64_t items = (p.n_span + p.n_empty) * p.F;
  if (items > 0) {
    gatv2_attention_finish_kernel<T><<<(unsigned)ceil_div(items, 256), 256, 0, s>>>(p);
    GNO_LAUNCHED("gatv2_attention_finish_kernel");
  }
  return GNO_OK;
}

// Grid as launch_backward_vb: as many CTAs as fit at once, each walking groups of chunks.
template <typename T, int VB, int NV, bool ATT>
static int ga_backward_vb(const GatAttnParams& p, const GaShape& sh, int* gx, cudaStream_t s) {
  static int per_sm = -1;
  if (per_sm < 0) {
    int n = 0;
    GNO_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, gatv2_attention_backward_kernel<T, VB, NV, ATT>,
                                                           kGatThreads, 0));
    per_sm = (int)imax64(1, imin64(n, kGatMaxCtasPerSm));
  }
  const int64_t groups = ceil_div(p.n_chunks, kGatThreads / p.L);
  *gx = (int)imin64(groups, imax64(1, (int64_t)kNumSMs * per_sm / sh.ncoltiles));
  gatv2_attention_backward_kernel<T, VB, NV, ATT><<<dim3((unsigned)*gx, (unsigned)sh.ncoltiles), kGatThreads, 0, s>>>(p);
  GNO_LAUNCHED("gatv2_attention_backward_kernel");
  return GNO_OK;
}

template <typename T, int VB, bool ATT>
static int ga_backward_nv(const GatAttnParams& p, const GaShape& sh, int* gx, cudaStream_t s) {
  switch (sh.NV) {
    case 1: return ga_backward_vb<T, VB, 1, ATT>(p, sh, gx, s);
    case 2: return ga_backward_vb<T, VB, 2, ATT>(p, sh, gx, s);
    default: return ga_backward_vb<T, VB, 4, ATT>(p, sh, gx, s);
  }
}

template <typename T, bool ATT>
static int ga_backward_att(const GatAttnParams& p, const GaShape& sh, int* gx, cudaStream_t s) {
  switch (sh.vb) {
    case 16: return ga_backward_nv<T, 16, ATT>(p, sh, gx, s);
    case 8: return ga_backward_nv<T, 8, ATT>(p, sh, gx, s);
    case 4: return ga_backward_nv<T, 4, ATT>(p, sh, gx, s);
    default:
      if constexpr (sizeof(T) == 2) return ga_backward_nv<T, 2, ATT>(p, sh, gx, s);
  }
  return fail(GNO_ERR_INVALID, "gno_gatv2_attention_backward: bad vector width %d", sh.vb);
}

template <typename T>
static int ga_backward(const GatAttnParams& p, const GaShape& sh, int* gx, cudaStream_t s) {
  return p.att_part ? ga_backward_att<T, true>(p, sh, gx, s) : ga_backward_att<T, false>(p, sh, gx, s);
}

static int ga_shape_checked(int64_t H, int64_t F, int es, uintptr_t align, GaShape* sh, const char* fn) {
  GNO_CHECK_ARG(ga_shape(H, F, es, align, sh), "%s: a head of %lld bytes spans more than %d vectors", fn,
                (long long)(F / H * es), 32 * kGaMaxVecs);
  return GNO_OK;
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

// Workspace of a pass that writes gatv2_backward_kernel's partials: chunk partials of the row
// gradient and per-CTA partials of grad_att, each only when asked for.
static int gat_backward_workspace(const gno_csr* g, int64_t H, int64_t F, int with_grad_own, int with_grad_att,
                                  size_t* bytes, const char* fn) {
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

int gno_gatv2_logits_backward_workspace(const gno_csr* g, int64_t H, int64_t F, int with_grad_own,
                                        int with_grad_att, size_t* bytes) {
  return gat_backward_workspace(g, H, F, with_grad_own, with_grad_att, bytes,
                                "gno_gatv2_logits_backward_workspace");
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

int gno_gatv2_attention_workspace(const gno_csr* g, int64_t H, int64_t F, size_t* bytes) {
  const char* fn = "gno_gatv2_attention_workspace";
  GNO_CHECK_ARG(bytes != nullptr, "%s: NULL argument", fn);
  if (int rc = gat_sizes_ok(g, H, F, 0, GNO_F32, fn)) return rc;
  WorkspaceSizer sz;
  const int64_t n_chunks = ceil_div(g->E, g->chunk_len);
  if (n_chunks > 0) {
    sz.take<float>((size_t)(2 * n_chunks * ((F + 7) / 8 * 8)));
    sz.take<float2>((size_t)(2 * n_chunks * H));
  }
  *bytes = sz.total();
  return GNO_OK;
}

int gno_gatv2_attention(const gno_csr* g, const void* x_l, int64_t xl_rows, const void* x_r, const void* att,
                        int64_t H, int64_t F, double negative_slope, double eps, void* out, float* m, float* s,
                        int dtype, void* wsp, size_t ws_bytes, gno_stream_t stream) {
  const char* fn = "gno_gatv2_attention";
  if (int rc = gat_sizes_ok(g, H, F, xl_rows, dtype, fn)) return rc;
  if (g->E == 0) return GNO_OK;
  GNO_CHECK_ARG(g->erow && g->gidx && g->rowptr && x_l && x_r && att && out && m && s, "%s: NULL buffer", fn);
  GNO_CHECK_ARG((g->n_span == 0 || g->srow) && (g->n_empty == 0 || g->zrow), "%s: row lists missing", fn);
  const int es = gat_dtype_size(dtype);
  const uintptr_t al = (uintptr_t)x_l | (uintptr_t)x_r | (uintptr_t)att | (uintptr_t)out;
  GNO_CHECK_ARG(al % es == 0, "%s: buffers not aligned to the element size", fn);
  GaShape sh;
  if (int rc = ga_shape_checked(H, F, es, al, &sh, fn)) return rc;
  if (wsp == nullptr) return fail(GNO_ERR_WORKSPACE, "%s: workspace is NULL", fn);

  GatAttnParams p = {};
  ga_fill(p, g, sh, H, F, es, negative_slope);
  p.xl = static_cast<const char*>(x_l);
  p.xr = static_cast<const char*>(x_r);
  p.att = static_cast<const char*>(att);
  p.out = out;
  p.m = m;
  p.d = s;
  p.eps = (float)eps;
  Workspace ws(wsp, ws_bytes);
  p.part = ws.take<float>((size_t)(2 * p.n_chunks * p.Fp));
  p.part_ms = ws.take<float2>((size_t)(2 * p.n_chunks * H));
  if (!ws.ok()) return fail(GNO_ERR_WORKSPACE, "%s: workspace too small (%zu < %zu)", fn, ws_bytes, ws.off);
  cudaStream_t st = (cudaStream_t)stream;
  switch (dtype) {
    case GNO_F32: return ga_forward<float>(p, sh, st);
    case GNO_F16: return ga_forward<__half>(p, sh, st);
    default: return ga_forward<__nv_bfloat16>(p, sh, st);
  }
}

int gno_gatv2_attention_backward_workspace(const gno_csr* g, int64_t H, int64_t F, int with_grad_x_r,
                                           int with_grad_att, size_t* bytes) {
  return gat_backward_workspace(g, H, F, with_grad_x_r, with_grad_att, bytes,
                                "gno_gatv2_attention_backward_workspace");
}

int gno_gatv2_attention_backward(const gno_csr* g, const void* x_l, int64_t xl_rows, const void* x_r,
                                 const void* att, const void* out, const float* m, const float* s,
                                 const void* grad_out, int64_t H, int64_t F, double negative_slope,
                                 void* grad_x_r, float* grad_att, void* grad_logits, void* alpha, int dtype,
                                 void* wsp, size_t ws_bytes, gno_stream_t stream) {
  const char* fn = "gno_gatv2_attention_backward";
  if (int rc = gat_sizes_ok(g, H, F, xl_rows, dtype, fn)) return rc;
  if (g->E == 0) return GNO_OK;
  GNO_CHECK_ARG(g->erow && g->gidx && g->rowptr && x_l && x_r && att && out && m && s && grad_out &&
                    (grad_x_r || grad_att || grad_logits) && (grad_logits == nullptr) == (alpha == nullptr),
                "%s: NULL buffer", fn);
  GNO_CHECK_ARG(grad_x_r == nullptr || ((g->n_span == 0 || g->srow) && (g->n_empty == 0 || g->zrow)),
                "%s: row lists missing", fn);
  const int es = gat_dtype_size(dtype);
  const uintptr_t al = (uintptr_t)x_l | (uintptr_t)x_r | (uintptr_t)att | (uintptr_t)out | (uintptr_t)grad_out |
                       (uintptr_t)grad_x_r;
  GNO_CHECK_ARG(((al | (uintptr_t)grad_logits | (uintptr_t)alpha) % es) == 0,
                "%s: buffers not aligned to the element size", fn);
  GaShape sh;
  if (int rc = ga_shape_checked(H, F, es, al, &sh, fn)) return rc;
  if (wsp == nullptr && (grad_x_r || grad_att)) return fail(GNO_ERR_WORKSPACE, "%s: workspace is NULL", fn);

  GatAttnParams p = {};
  ga_fill(p, g, sh, H, F, es, negative_slope);
  p.xl = static_cast<const char*>(x_l);
  p.xr = static_cast<const char*>(x_r);
  p.att = static_cast<const char*>(att);
  p.out_in = static_cast<const char*>(out);
  p.g = grad_out;
  p.out = grad_x_r;
  p.m = const_cast<float*>(m);
  p.d = const_cast<float*>(s);
  p.da = grad_logits;
  p.alpha = alpha;
  Workspace ws(wsp, ws_bytes);
  p.part = grad_x_r ? ws.take<float>((size_t)(2 * p.n_chunks * p.Fp)) : nullptr;
  p.att_part = grad_att ? ws.take<float>((size_t)((int64_t)kNumSMs * kGatMaxCtasPerSm * F)) : nullptr;
  if (!ws.ok()) return fail(GNO_ERR_WORKSPACE, "%s: workspace too small (%zu < %zu)", fn, ws_bytes, ws.off);
  cudaStream_t st = (cudaStream_t)stream;
  int gx = 0, rc;
  switch (dtype) {
    case GNO_F32: rc = ga_backward<float>(p, sh, &gx, st); break;
    case GNO_F16: rc = ga_backward<__half>(p, sh, &gx, st); break;
    default: rc = ga_backward<__nv_bfloat16>(p, sh, &gx, st); break;
  }
  if (rc) return rc;
  if (grad_x_r) {
    SegParams q = {};
    q.out = grad_x_r;
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
    if (int rf = seg_finish_sum(q, dtype, true, st)) return rf;
  }
  if (grad_att) {
    gatv2_att_finish_kernel<<<(unsigned)ceil_div(F, 256), 256, 0, st>>>(p.att_part, gx, F, grad_att);
    GNO_LAUNCHED("gatv2_att_finish_kernel");
  }
  return GNO_OK;
}

}  // extern "C"
