// Several aggregators over one neighbourhood in one pass (PNAConv.aggregate: a list of aggregators,
// concatenated, then copies scaled by degree scalers), forward and backward:
//
//   m_e = x[gidx[k], :] for the sorted edge k of edge e = eid[k]   (message form: gidx = eid = perm)
//   d_i = max(deg_i, 1)
//   sum = Σ m, mean = sum / d, var = Σ m² / d − mean², std = sqrt(relu(var) + 1e-5)
//   min / max: torch_scatter's rule (ascending edge order, strict compare, NaN never wins, an
//   element nobody beat gives 0)
//   out[i, t, (s·A + a)·F + f] = agg_a(i, t·F + f) · scale_s(d_i)
//
//   multiagg_kernel: the segment reduce's edge-balanced structure on the dst plan (as the GATv2
//   backward walks it).  A slot of L lanes owns a chunk of chunk_len sorted edges; each lane keeps
//   one VB-byte vector of the message row (a vector never straddles a tower) and only the
//   statistics the requested aggregators need: Σm and Σm² (ST_MOMENTS), the min and max with their
//   edge ids (ST_EXTREMES).  A row that ends inside the chunk writes every (s, a) block directly,
//   scaled by factors from its own length, and optionally the backward state (fp32 mean and var,
//   int32 winners).  Rows cut by a chunk boundary leave per-chunk statistics in a two-slot partial
//   layout (the segment reduce's); multiagg_finish_kernel combines them in chunk order (Σ in fp64,
//   extremes by strict compare, so the lowest edge keeps a tie) and writes the empty rows.
//
//   multiagg_backward_kernel (message form): the same walk.  When the row changes, a lane reads
//   the row's S·A gradient vectors and saved state once and reduces them to
//     c_a = Σ_s scale_s · G_{s,a},  cv = c_var + c_std · [var > 0] / (2 std)
//     P = c_sum + c_mean / d − 2 cv · mean / d,  Q = 2 cv / d
//   and every edge of the row writes grad[eid] = P + Q·m + [e = argmin]·c_min + [e = argmax]·c_max.
//   Each element is written once, no atomics.
//
//   multiagg_coeffs_kernel (gather form): the same per-row reduction, written as node-level fp32
//   [P | Q] rows and c_min / c_max for the transposed pass on the src plan.
//
// Roofline: HBM.  Bytes per edge = forward: W*s (message row) + 8 (gidx, erow) [+4 eid with
// extremes]; per row = S*A*W*s (output) [+8 W state].  Backward (message form): per edge 2 W*s
// (message row in, gradient row out) + 12; per row S*A*W*s (incoming gradient) + state.
#include <climits>

#include "segreduce.cuh"

namespace gno {

constexpr int kMaThreads = 256;
constexpr int kMaBatch = 4;  // sorted edges whose records and rows are loaded before use
constexpr int kMaMaxCtasPerSm = 2048 / kMaThreads;
constexpr int kMaMaxList = 8;  // aggregators / scalers per call
constexpr int kMaNoArg = INT_MAX;
constexpr int ST_MOMENTS = 1, ST_EXTREMES = 2, ST_ALL = 3;

struct MaParams {
  const int32_t* erow;
  const int32_t* gidx;  // row of x per sorted edge (NULL = k)
  const int32_t* eid;   // original edge id per sorted edge (NULL = k)
  const int64_t* rowptr;
  const int32_t* srow;
  const int32_t* zrow;
  const char* x;        // [x_rows, W] messages (message form) or node features (gather form)
  const char* g;        // backward: incoming gradient [N, T*S*A*F]
  void* out;            // forward: [N, T*S*A*F]; backward: grad of x [x_rows, W]
  int32_t* amin;        // [N, W] winners (original edge ids, arg_fill = none), or NULL
  int32_t* amax;
  float* mean;          // [N, W] fp32 mean and var (before relu), or NULL
  float* var;
  float *p_sum, *p_sq, *p_mn, *p_mx;  // [2 * n_chunks, W] statistics of rows cut by a chunk boundary
  int32_t *p_amin, *p_amax;
  float* pq;            // coefficients kernel: [N + 1, 2W] rows [P | Q]
  float* cmn;           // coefficients kernel: [N, W] c_min / c_max, or NULL
  float* cmx;
  int64_t N, E, n_chunks, n_span, n_empty;
  int64_t W, F;         // columns of a message row (T*F); columns of one tower
  int64_t ldo;          // elements per output row: T*S*A*F
  int64_t row_bytes;    // W * sizeof(T)
  int arg_fill;
  int nvec, L, chunk_len;
  int A, S;
  int agg[kMaMaxList];
  int scl[kMaMaxList];
  float avg_lin, avg_log;
};

__device__ __forceinline__ float ma_scale(const MaParams& p, int s, float d) {
  switch (p.scl[s]) {
    case GNO_SCALE_AMPLIFICATION: return logf(d + 1.f) / p.avg_log;
    case GNO_SCALE_ATTENUATION: return p.avg_log / logf(d + 1.f);
    case GNO_SCALE_LINEAR: return d / p.avg_lin;
    case GNO_SCALE_INVERSE_LINEAR: return p.avg_lin / d;
    default: return 1.f;
  }
}

// Unscaled aggregate of one element.  relu(var) keeps a NaN variance NaN, as torch's relu does.
__device__ __forceinline__ float ma_value(int code, float sum, float mean, float var, float mn, float mx) {
  switch (code) {
    case GNO_AGG_SUM: return sum;
    case GNO_AGG_MEAN: return mean;
    case GNO_AGG_MIN: return mn;
    case GNO_AGG_MAX: return mx;
    case GNO_AGG_VAR: return var;
    default: return sqrtf((var < 0.f ? 0.f : var) + 1e-5f);
  }
}

// Per-lane statistics of one VB-byte vector.  The extremes start at the storage type's finite
// limits and a strictly better value wins, like the segment reduce's MIN/MAX.
template <typename T, int VB, int ST>
struct MaAcc {
  static constexpr int EPV = VB / (int)sizeof(T);
  static constexpr bool kMom = (ST & ST_MOMENTS) != 0, kExt = (ST & ST_EXTREMES) != 0;
  float s[kMom ? EPV : 1], q[kMom ? EPV : 1], mn[kExt ? EPV : 1], mx[kExt ? EPV : 1];
  int amn[kExt ? EPV : 1], amx[kExt ? EPV : 1];

  __device__ __forceinline__ void reset() {
#pragma unroll
    for (int i = 0; i < EPV; ++i) {
      if constexpr (kMom) s[i] = q[i] = 0.f;
      if constexpr (kExt) {
        mn[i] = DType<T>::highest();
        mx[i] = DType<T>::lowest();
        amn[i] = amx[i] = kMaNoArg;
      }
    }
  }
  __device__ __forceinline__ void add(const Words<VB>& w, int e) {
#pragma unroll
    for (int i = 0; i < EPV; ++i) {
      const float f = elem<T, VB>(w, i);
      if constexpr (kMom) {
        s[i] += f;
        q[i] = fmaf(f, f, q[i]);
      }
      if constexpr (kExt) {
        if (f < mn[i]) { mn[i] = f; amn[i] = e; }
        if (f > mx[i]) { mx[i] = f; amx[i] = e; }
      }
    }
  }
};

// Output address of element column `ce` (= t*F + f) of row `row`, block (0, 0).
template <typename T>
__device__ __forceinline__ T* ma_out_elem(const MaParams& p, int64_t row, int64_t ce) {
  const int64_t t = ce / p.F;
  const int64_t f = ce - t * p.F;
  return static_cast<T*>(p.out) + row * p.ldo + t * (p.ldo / (p.W / p.F)) + f;
}

// A finished row held by one lane: every (s, a) block with vector stores, and the backward state.
template <typename T, int VB, int ST>
__device__ __forceinline__ void ma_store_row(const MaParams& p, int64_t row, int v, const MaAcc<T, VB, ST>& acc,
                                             int deg) {
  constexpr int EPV = VB / (int)sizeof(T);
  const float d = (float)(deg > 1 ? deg : 1);
  float sum[EPV], mean[EPV], var[EPV], mn[EPV], mx[EPV];
#pragma unroll
  for (int i = 0; i < EPV; ++i) {
    sum[i] = mean[i] = var[i] = mn[i] = mx[i] = 0.f;
    if constexpr (MaAcc<T, VB, ST>::kMom) {
      sum[i] = acc.s[i];
      mean[i] = __fdiv_rn(acc.s[i], d);
      var[i] = __fdiv_rn(acc.q[i], d) - mean[i] * mean[i];
    }
    if constexpr (MaAcc<T, VB, ST>::kExt) {
      mn[i] = acc.amn[i] == kMaNoArg ? 0.f : acc.mn[i];
      mx[i] = acc.amx[i] == kMaNoArg ? 0.f : acc.mx[i];
    }
  }
  const int64_t ce = (int64_t)v * EPV;
  char* ob = reinterpret_cast<char*>(ma_out_elem<T>(p, row, ce));
  const int64_t blk = p.F * (int64_t)sizeof(T);
  for (int s = 0; s < p.S; ++s) {
    const float sc = ma_scale(p, s, d);
    for (int a = 0; a < p.A; ++a) {
      const int code = p.agg[a];
      Words<VB> o;
#pragma unroll
      for (int i = 0; i < EPV; ++i) set_elem<T, VB>(o, i, ma_value(code, sum[i], mean[i], var[i], mn[i], mx[i]) * sc);
      st_vec<VB>(ob + (int64_t)(s * p.A + a) * blk, o);
    }
  }
  const int64_t so = row * p.W + ce;
  if constexpr (MaAcc<T, VB, ST>::kMom) {
    if (p.mean) {
#pragma unroll
      for (int i = 0; i < EPV; ++i) {
        p.mean[so + i] = mean[i];
        p.var[so + i] = var[i];
      }
    }
  }
  if constexpr (MaAcc<T, VB, ST>::kExt) {
#pragma unroll
    for (int i = 0; i < EPV; ++i) {
      if (p.amin) p.amin[so + i] = acc.amn[i] == kMaNoArg ? p.arg_fill : acc.amn[i];
      if (p.amax) p.amax[so + i] = acc.amx[i] == kMaNoArg ? p.arg_fill : acc.amx[i];
    }
  }
}

template <typename T, int VB, int ST>
__device__ __forceinline__ void ma_store_partial(const MaParams& p, int64_t slot, int v,
                                                 const MaAcc<T, VB, ST>& acc) {
  constexpr int EPV = VB / (int)sizeof(T);
  const int64_t o = slot * p.W + (int64_t)v * EPV;
#pragma unroll
  for (int i = 0; i < EPV; ++i) {
    if constexpr (MaAcc<T, VB, ST>::kMom) {
      p.p_sum[o + i] = acc.s[i];
      p.p_sq[o + i] = acc.q[i];
    }
    if constexpr (MaAcc<T, VB, ST>::kExt) {
      p.p_mn[o + i] = acc.mn[i];
      p.p_mx[o + i] = acc.mx[i];
      p.p_amin[o + i] = acc.amn[i];
      p.p_amax[o + i] = acc.amx[i];
    }
  }
}

template <typename T, int VB, int ST>
__global__ void __launch_bounds__(kMaThreads, 2) multiagg_kernel(const MaParams p) {
  // programmatic dependent launch: the finish kernel may fill the empty rows while this grid runs
  asm volatile("griddepcontrol.launch_dependents;");
  constexpr bool kExt = (ST & ST_EXTREMES) != 0;
  const int L = p.L, S = kMaThreads / L;
  const int slot = threadIdx.x / L, lane = threadIdx.x - slot * L;
  const int v = blockIdx.y * 32 + lane;
  const bool vact = v < p.nvec;
  const int64_t col = (int64_t)v * VB;
  const bool same_e = p.eid == p.gidx;
  MaAcc<T, VB, ST> acc;

  for (int64_t grp = blockIdx.x; vact && grp * S < p.n_chunks; grp += gridDim.x) {
    const int64_t c = grp * S + slot;
    if (c >= p.n_chunks) break;
    const int64_t k0 = c * p.chunk_len;
    const int nv = (int)imin64(p.chunk_len, p.E - k0);
    int cur = __ldg(p.erow + k0);
    bool head = k0 > 0 && __ldg(p.erow + k0 - 1) == cur;
    int seg_start = 0;
    acc.reset();
    auto gid = [&](int64_t k) { return p.gidx ? (int64_t)__ldg(p.gidx + k) : k; };
    auto eidx = [&](int64_t k, int64_t gk) { return same_e ? (int)gk : p.eid ? __ldg(p.eid + k) : (int)k; };
    int i = 0;
#pragma unroll 1
    while (i < nv) {
      if (i + kMaBatch <= nv) {
        // rows ascend: the batch's last row equal to cur means no boundary inside it
        int64_t gk[kMaBatch];
#pragma unroll
        for (int u = 0; u < kMaBatch; ++u) gk[u] = gid(k0 + i + u);
        if (__ldg(p.erow + k0 + i + kMaBatch - 1) == cur) {
          Words<VB> xv[kMaBatch];
          int ev[kMaBatch];
#pragma unroll
          for (int u = 0; u < kMaBatch; ++u) {
            xv[u] = ld_vec<VB>(p.x + gk[u] * p.row_bytes + col);
            ev[u] = kExt ? eidx(k0 + i + u, gk[u]) : 0;
          }
#pragma unroll
          for (int u = 0; u < kMaBatch; ++u) acc.add(xv[u], ev[u]);
          i += kMaBatch;
          continue;
        }
      }
      // one edge at a time across a row boundary (and the chunk's last edges)
      const int64_t k = k0 + i;
      const int row = __ldg(p.erow + k);
      const int64_t g1 = gid(k);
      const Words<VB> x1 = ld_vec<VB>(p.x + g1 * p.row_bytes + col);
      if (row != cur) {
        if (head) ma_store_partial(p, 2 * c, v, acc);  // a chunk inside one row never gets here
        else ma_store_row(p, cur, v, acc, i - seg_start);
        head = false;
        cur = row;
        seg_start = i;
        acc.reset();
      }
      acc.add(x1, kExt ? eidx(k, g1) : 0);
      ++i;
    }
    const bool tail = k0 + nv < p.E && __ldg(p.erow + k0 + nv) == cur;
    if (head || tail) ma_store_partial(p, 2 * c + (head ? 0 : 1), v, acc);
    else ma_store_row(p, cur, v, acc, nv - seg_start);
  }
}

// One element of a finished row from its (combined) statistics: every (s, a) block and the state.
template <typename T>
__device__ __forceinline__ void ma_write_elem(const MaParams& p, int64_t row, int64_t ce, int64_t deg, float sum,
                                              float mean, float var, float mn, int amn, float mx, int amx) {
  const float d = (float)(deg > 1 ? deg : 1);
  mn = amn == kMaNoArg ? 0.f : mn;
  mx = amx == kMaNoArg ? 0.f : mx;
  T* o = ma_out_elem<T>(p, row, ce);
  for (int s = 0; s < p.S; ++s) {
    const float sc = ma_scale(p, s, d);
    for (int a = 0; a < p.A; ++a)
      o[(int64_t)(s * p.A + a) * p.F] = DType<T>::from_f(ma_value(p.agg[a], sum, mean, var, mn, mx) * sc);
  }
  const int64_t so = row * p.W + ce;
  if (p.mean) {
    p.mean[so] = mean;
    p.var[so] = var;
  }
  if (p.amin) p.amin[so] = amn == kMaNoArg ? p.arg_fill : amn;
  if (p.amax) p.amax[so] = amx == kMaNoArg ? p.arg_fill : amx;
}

// Finish pass: (a) empty rows (sum 0, var 0, extremes 0, winners arg_fill); (b) after the main
// grid, rows cut by a chunk boundary: the tail slot of their first chunk, then the head slot of
// every later chunk, in chunk order.  One thread per (row, element).
template <typename T>
__global__ void __launch_bounds__(256) multiagg_finish_kernel(const MaParams p) {
  const int64_t W = p.W;
  const int64_t tid0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t tstride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t j = tid0; j < p.n_empty * W; j += tstride) {
    const int64_t z = j / W;
    ma_write_elem<T>(p, p.zrow[z], j - z * W, 0, 0.f, 0.f, 0.f, 0.f, kMaNoArg, 0.f, kMaNoArg);
  }
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const bool mom = p.p_sum != nullptr, ext = p.p_mn != nullptr;
  for (int64_t j = tid0; j < p.n_span * W; j += tstride) {
    const int64_t sr = j / W, ce = j - sr * W;
    const int64_t row = p.srow[sr];
    const int64_t kb = p.rowptr[row], ke = p.rowptr[row + 1];
    const int64_t ca = kb / p.chunk_len, cb = (ke - 1) / p.chunk_len;
    double sum = 0.0, sq = 0.0;
    float mn = 0.f, mx = 0.f;
    int amn = kMaNoArg, amx = kMaNoArg;
    for (int64_t c = ca; c <= cb; ++c) {
      const int64_t o = (c == ca ? 2 * c + 1 : 2 * c) * W + ce;
      if (mom) {
        sum += (double)p.p_sum[o];
        sq += (double)p.p_sq[o];
      }
      if (ext) {
        const float a = p.p_mn[o], b = p.p_mx[o];
        if (c == ca || a < mn) { mn = a; amn = p.p_amin[o]; }  // chunks ascend: strict keeps the lowest
        if (c == ca || b > mx) { mx = b; amx = p.p_amax[o]; }
      }
    }
    const double d = (double)imax64(ke - kb, 1);
    const double mean = sum / d;
    ma_write_elem<T>(p, row, ce, ke - kb, (float)sum, (float)mean, (float)(sq / d - mean * mean), mn, amn, mx,
                     amx);
  }
}

// Per-row coefficients of one lane's vector (see the header comment): P, Q, c_min, c_max and the
// winners.  g is the incoming gradient [N, T*S*A*F] in T.
template <typename T, int VB>
__device__ __forceinline__ void ma_coeffs(const MaParams& p, int64_t row, int v, float (&P)[VB / sizeof(T)],
                                          float (&Q)[VB / sizeof(T)], float (&cmn)[VB / sizeof(T)],
                                          float (&cmx)[VB / sizeof(T)], int (&wmn)[VB / sizeof(T)],
                                          int (&wmx)[VB / sizeof(T)]) {
  constexpr int EPV = VB / (int)sizeof(T);
  const int64_t deg = p.rowptr[row + 1] - p.rowptr[row];
  const float d = (float)(deg > 1 ? deg : 1);
  float cv[EPV], cs[EPV];
#pragma unroll
  for (int i = 0; i < EPV; ++i) P[i] = cv[i] = cs[i] = cmn[i] = cmx[i] = 0.f;
  const int64_t ce = (int64_t)v * EPV;
  const int64_t t = ce / p.F;
  const char* gb = p.g + (row * p.ldo + t * (p.ldo / (p.W / p.F)) + (ce - t * p.F)) * (int64_t)sizeof(T);
  const int64_t blk = p.F * (int64_t)sizeof(T);
  for (int s = 0; s < p.S; ++s) {
    const float sc = ma_scale(p, s, d);
    for (int a = 0; a < p.A; ++a) {
      const int code = p.agg[a];
      const Words<VB> gv = ld_vec<VB>(gb + (int64_t)(s * p.A + a) * blk);
#pragma unroll
      for (int i = 0; i < EPV; ++i) {
        const float c = sc * elem<T, VB>(gv, i);
        switch (code) {
          case GNO_AGG_SUM: P[i] += c; break;
          case GNO_AGG_MEAN: P[i] += __fdiv_rn(c, d); break;
          case GNO_AGG_MIN: cmn[i] += c; break;
          case GNO_AGG_MAX: cmx[i] += c; break;
          case GNO_AGG_VAR: cv[i] += c; break;
          default: cs[i] += c; break;
        }
      }
    }
  }
  const int64_t so = row * p.W + ce;
#pragma unroll
  for (int i = 0; i < EPV; ++i) {
    Q[i] = 0.f;
    if (p.mean) {
      const float var = p.var[so + i], mean = p.mean[so + i];
      // torch's relu backward is 0 at 0
      const float c = var > 0.f ? cv[i] + cs[i] / (2.f * sqrtf(var + 1e-5f)) : cv[i];
      Q[i] = __fdiv_rn(2.f * c, d);
      P[i] -= Q[i] * mean;
    }
    wmn[i] = p.amin ? p.amin[so + i] : -1;
    wmx[i] = p.amax ? p.amax[so + i] : -1;
  }
}

// Message-form backward: grad[eid[k]] = P + Q * x[gidx[k]] + routed extremes, row coefficients
// computed when the row changes.
template <typename T, int VB>
__global__ void __launch_bounds__(kMaThreads, 2) multiagg_backward_kernel(const MaParams p) {
  constexpr int EPV = VB / (int)sizeof(T);
  const int L = p.L, S = kMaThreads / L;
  const int slot = threadIdx.x / L, lane = threadIdx.x - slot * L;
  const int v = blockIdx.y * 32 + lane;
  const bool vact = v < p.nvec;
  const int64_t col = (int64_t)v * VB;
  char* gout = static_cast<char*>(p.out);

  for (int64_t grp = blockIdx.x; vact && grp * S < p.n_chunks; grp += gridDim.x) {
    const int64_t c = grp * S + slot;
    if (c >= p.n_chunks) break;
    const int64_t k0 = c * p.chunk_len;
    const int nv = (int)imin64(p.chunk_len, p.E - k0);
    int cur = __ldg(p.erow + k0);
    float P[EPV], Q[EPV], cmn[EPV], cmx[EPV];
    int wmn[EPV], wmx[EPV];
    ma_coeffs<T, VB>(p, cur, v, P, Q, cmn, cmx, wmn, wmx);
    auto edge = [&](const Words<VB>& x, int64_t e) {
      Words<VB> r;
#pragma unroll
      for (int j = 0; j < EPV; ++j) {
        float gsum = fmaf(Q[j], elem<T, VB>(x, j), P[j]);
        if (wmn[j] == (int)e) gsum += cmn[j];
        if (wmx[j] == (int)e) gsum += cmx[j];
        set_elem<T, VB>(r, j, gsum);
      }
      st_vec<VB>(gout + e * p.row_bytes + col, r);
    };
    auto gid = [&](int64_t k) { return p.gidx ? (int64_t)__ldg(p.gidx + k) : k; };
    auto eidx = [&](int64_t k, int64_t gk) { return p.eid == p.gidx ? gk : p.eid ? (int64_t)__ldg(p.eid + k) : k; };
    int i = 0;
#pragma unroll 1
    while (i < nv) {
      if (i + kMaBatch <= nv) {
        int64_t gk[kMaBatch];
#pragma unroll
        for (int u = 0; u < kMaBatch; ++u) gk[u] = gid(k0 + i + u);
        if (__ldg(p.erow + k0 + i + kMaBatch - 1) == cur) {
          Words<VB> xv[kMaBatch];
#pragma unroll
          for (int u = 0; u < kMaBatch; ++u) xv[u] = ld_vec<VB>(p.x + gk[u] * p.row_bytes + col);
#pragma unroll
          for (int u = 0; u < kMaBatch; ++u) edge(xv[u], eidx(k0 + i + u, gk[u]));
          i += kMaBatch;
          continue;
        }
      }
      const int64_t k = k0 + i;
      const int row = __ldg(p.erow + k);
      if (row != cur) {
        cur = row;
        ma_coeffs<T, VB>(p, cur, v, P, Q, cmn, cmx, wmn, wmx);
      }
      const int64_t g1 = gid(k);
      edge(ld_vec<VB>(p.x + g1 * p.row_bytes + col), eidx(k, g1));
      ++i;
    }
  }
}

// Gather-form coefficients: pq[i] = [P | Q] (fp32, row stride 2W), c_min / c_max [N, W] when
// requested.  One thread per (row, element).
template <typename T>
__global__ void __launch_bounds__(256) multiagg_coeffs_kernel(const MaParams p) {
  const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (j >= p.N * p.W) return;
  const int64_t row = j / p.W;
  const int v = (int)(j - row * p.W);
  float P[1], Q[1], cmn[1], cmx[1];
  int wmn[1], wmx[1];
  ma_coeffs<T, (int)sizeof(T)>(p, row, v, P, Q, cmn, cmx, wmn, wmx);
  p.pq[row * 2 * p.W + v] = P[0];
  p.pq[row * 2 * p.W + p.W + v] = Q[0];
  if (p.cmn) p.cmn[j] = cmn[0];
  if (p.cmx) p.cmx[j] = cmx[0];
}

// ------------------------------------------------------------------------------ host side --
static int ma_es(int dtype) { return dtype == GNO_F32 ? 4 : 2; }

struct MaInfo {
  bool mom, ext, second;  // moments, extremes, var/std requested
};

static int ma_check(const gno_csr* g, int64_t T, int64_t F, const int* aggs, int n_aggs, const int* scalers,
                    int n_scalers, int dtype, const char* fn, MaInfo* info) {
  GNO_CHECK_ARG(g != nullptr, "%s: graph is NULL", fn);
  GNO_CHECK_ARG(dtype == GNO_F32 || dtype == GNO_F16 || dtype == GNO_BF16, "%s: unknown dtype %d", fn, dtype);
  GNO_CHECK_ARG(T >= 1 && F >= 0 && T * F < (int64_t(1) << 24) && g->N >= 0 && g->E >= 0 &&
                    g->E < (int64_t(1) << 31),
                "%s: bad sizes T=%lld F=%lld N=%lld E=%lld", fn, (long long)T, (long long)F, (long long)g->N,
                (long long)g->E);
  GNO_CHECK_ARG(g->chunk_len >= 32 && g->chunk_len % 32 == 0 && g->chunk_len <= (1 << 20),
                "%s: chunk_len must be a multiple of 32", fn);
  GNO_CHECK_ARG(aggs != nullptr && n_aggs >= 1 && n_aggs <= kMaMaxList, "%s: need 1..%d aggregators", fn,
                kMaMaxList);
  GNO_CHECK_ARG(scalers != nullptr && n_scalers >= 1 && n_scalers <= kMaMaxList, "%s: need 1..%d scalers", fn,
                kMaMaxList);
  MaInfo in = {false, false, false};
  for (int a = 0; a < n_aggs; ++a) {
    GNO_CHECK_ARG(aggs[a] >= GNO_AGG_SUM && aggs[a] <= GNO_AGG_STD, "%s: unknown aggregator %d", fn, aggs[a]);
    if (aggs[a] == GNO_AGG_MIN || aggs[a] == GNO_AGG_MAX) in.ext = true;
    else in.mom = true;
    if (aggs[a] == GNO_AGG_VAR || aggs[a] == GNO_AGG_STD) in.second = true;
  }
  for (int s = 0; s < n_scalers; ++s)
    GNO_CHECK_ARG(scalers[s] >= GNO_SCALE_IDENTITY && scalers[s] <= GNO_SCALE_INVERSE_LINEAR,
                  "%s: unknown scaler %d", fn, scalers[s]);
  if (info) *info = in;
  return GNO_OK;
}

static void ma_fill(MaParams& p, const gno_csr* g, int64_t T, int64_t F, const int* aggs, int n_aggs,
                    const int* scalers, int n_scalers, double avg_lin, double avg_log, int es) {
  p = MaParams{};
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
  p.W = T * F;
  p.F = F;
  p.ldo = T * F * n_scalers * n_aggs;
  p.row_bytes = T * F * es;
  p.chunk_len = (int)g->chunk_len;
  p.A = n_aggs;
  p.S = n_scalers;
  for (int a = 0; a < n_aggs; ++a) p.agg[a] = aggs[a];
  for (int s = 0; s < n_scalers; ++s) p.scl[s] = scalers[s];
  p.avg_lin = (float)avg_lin;
  p.avg_log = (float)avg_log;
}


// Widest vector inside one tower and the alignment; an 8-byte vector is read as two 4-byte ones,
// which keeps the vector widths at {16, 4} bytes (fp32) and {16, 4, 2} (16-bit).
static int ma_vectors(MaParams& p, uintptr_t al, int es) {
  int vb = head_vector_bytes(p.F * es, al, es);
  if (vb == 8) vb = 4;
  p.nvec = (int)(p.W * es / vb);
  int L = 1;
  while (L < p.nvec && L < 32) L <<= 1;
  p.L = L;
  return vb;
}

// Grid: column tiles of 32 vectors in y; in x, as many CTAs as are resident at once, each walking
// groups of chunks.
template <typename K>
static dim3 ma_grid(K kernel, const MaParams& p, int* per_sm) {
  if (*per_sm < 0) {
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, kMaThreads, 0) != cudaSuccess) n = 1;
    *per_sm = (int)imax64(1, imin64(n, kMaMaxCtasPerSm));
  }
  const int ncoltiles = (p.nvec + 31) / 32;
  const int64_t groups = ceil_div(p.n_chunks, kMaThreads / p.L);
  return dim3((unsigned)imin64(groups, imax64(1, (int64_t)kNumSMs * *per_sm / ncoltiles)), (unsigned)ncoltiles);
}

template <typename T, int VB, int ST>
static int ma_launch_fwd(const MaParams& p, cudaStream_t s) {
  static int per_sm = -1;
  const dim3 grid = ma_grid(multiagg_kernel<T, VB, ST>, p, &per_sm);
  multiagg_kernel<T, VB, ST><<<grid, kMaThreads, 0, s>>>(p);
  GNO_LAUNCHED("multiagg_kernel");
  return GNO_OK;
}

template <typename T, int VB>
static int ma_fwd_st(const MaParams& p, int st, cudaStream_t s) {
  switch (st) {
    case ST_MOMENTS: return ma_launch_fwd<T, VB, ST_MOMENTS>(p, s);
    case ST_EXTREMES: return ma_launch_fwd<T, VB, ST_EXTREMES>(p, s);
    default: return ma_launch_fwd<T, VB, ST_ALL>(p, s);
  }
}

template <typename T>
static int ma_fwd(const MaParams& p, int vb, int st, bool after_kernel, cudaStream_t s) {
  if (p.n_chunks > 0) {
    int rc;
    switch (vb) {
      case 16: rc = ma_fwd_st<T, 16>(p, st, s); break;
      case 4: rc = ma_fwd_st<T, 4>(p, st, s); break;
      default:
        if constexpr (sizeof(T) == 2) {
          rc = ma_fwd_st<T, 2>(p, st, s);
          break;
        }
        return fail(GNO_ERR_INVALID, "gno_multi_aggregate: bad vector width %d", vb);
    }
    if (rc) return rc;
  }
  const int64_t items = (p.n_span + p.n_empty) * p.W;
  if (items == 0) return GNO_OK;
  const int grid = (int)imin64(ceil_div(items, 256), (int64_t)kNumSMs * 16);
  if (after_kernel && p.n_chunks > 0) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(256);
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    GNO_CUDA(cudaLaunchKernelEx(&cfg, multiagg_finish_kernel<T>, p));
  } else {
    multiagg_finish_kernel<T><<<grid, 256, 0, s>>>(p);
  }
  GNO_LAUNCHED("multiagg_finish_kernel");
  return GNO_OK;
}

template <typename T, int VB>
static int ma_launch_bwd(const MaParams& p, cudaStream_t s) {
  static int per_sm = -1;
  const dim3 grid = ma_grid(multiagg_backward_kernel<T, VB>, p, &per_sm);
  multiagg_backward_kernel<T, VB><<<grid, kMaThreads, 0, s>>>(p);
  GNO_LAUNCHED("multiagg_backward_kernel");
  return GNO_OK;
}

template <typename T>
static int ma_bwd(const MaParams& p, int vb, cudaStream_t s) {
  switch (vb) {
    case 16: return ma_launch_bwd<T, 16>(p, s);
    case 4: return ma_launch_bwd<T, 4>(p, s);
    default:
      if constexpr (sizeof(T) == 2) return ma_launch_bwd<T, 2>(p, s);
  }
  return fail(GNO_ERR_INVALID, "gno_multi_aggregate_backward: bad vector width %d", vb);
}

template <typename T>
static int ma_coeffs_launch(const MaParams& p, cudaStream_t s) {
  const int64_t items = p.N * p.W;
  if (items == 0) return GNO_OK;
  multiagg_coeffs_kernel<T><<<(unsigned)ceil_div(items, 256), 256, 0, s>>>(p);
  GNO_LAUNCHED("multiagg_coeffs_kernel");
  return GNO_OK;
}

}  // namespace gno

using namespace gno;

extern "C" {

int gno_multi_aggregate_workspace(const gno_csr* g, int64_t T, int64_t F, const int* aggs, int n_aggs,
                                  size_t* bytes) {
  const char* fn = "gno_multi_aggregate_workspace";
  GNO_CHECK_ARG(bytes != nullptr, "%s: NULL argument", fn);
  static const int identity = GNO_SCALE_IDENTITY;
  MaInfo in;
  if (int rc = ma_check(g, T, F, aggs, n_aggs, &identity, 1, GNO_F32, fn, &in)) return rc;
  WorkspaceSizer sz;
  const int64_t n_chunks = ceil_div(g->E, g->chunk_len);
  const size_t n = (size_t)(2 * n_chunks * T * F);
  if (n > 0) {
    if (in.mom) {
      sz.take<float>(n);
      sz.take<float>(n);
    }
    if (in.ext) {
      sz.take<float>(n);
      sz.take<float>(n);
      sz.take<int32_t>(n);
      sz.take<int32_t>(n);
    }
  }
  *bytes = sz.total();
  return GNO_OK;
}

int gno_multi_aggregate(const gno_csr* g, const void* x, int64_t x_rows, int64_t T, int64_t F, const int* aggs,
                        int n_aggs, const int* scalers, int n_scalers, double avg_lin, double avg_log, void* out,
                        int32_t* arg_min, int32_t* arg_max, float* mean, float* var, int64_t arg_fill, int dtype,
                        void* wsp, size_t ws_bytes, gno_stream_t stream) {
  const char* fn = "gno_multi_aggregate";
  MaInfo in;
  if (int rc = ma_check(g, T, F, aggs, n_aggs, scalers, n_scalers, dtype, fn, &in)) return rc;
  GNO_CHECK_ARG(x_rows >= 0 && arg_fill >= 0 && arg_fill < (int64_t(1) << 31), "%s: bad sizes x_rows=%lld arg_fill=%lld",
                fn, (long long)x_rows, (long long)arg_fill);
  GNO_CHECK_ARG((mean == nullptr) == (var == nullptr) && (mean == nullptr || in.mom),
                "%s: mean and var go together, and need a moment aggregator", fn);
  GNO_CHECK_ARG((arg_min == nullptr && arg_max == nullptr) || in.ext, "%s: winners need min or max", fn);
  if (g->N == 0 || F == 0) return GNO_OK;
  GNO_CHECK_ARG(g->rowptr && out && (g->E == 0 || (x && g->erow)), "%s: NULL buffer", fn);
  GNO_CHECK_ARG((g->n_span == 0 || g->srow) && (g->n_empty == 0 || g->zrow), "%s: row lists missing", fn);
  const int es = ma_es(dtype);
  GNO_CHECK_ARG((((uintptr_t)x | (uintptr_t)out) % es) == 0, "%s: buffers not aligned to the element size", fn);
  MaParams p;
  ma_fill(p, g, T, F, aggs, n_aggs, scalers, n_scalers, avg_lin, avg_log, es);
  p.x = static_cast<const char*>(x);
  p.out = out;
  p.amin = arg_min;
  p.amax = arg_max;
  p.mean = mean;
  p.var = var;
  p.arg_fill = (int)arg_fill;
  if (p.n_chunks > 0) {
    if (wsp == nullptr) return fail(GNO_ERR_WORKSPACE, "%s: workspace is NULL", fn);
    Workspace ws(wsp, ws_bytes);
    const size_t n = (size_t)(2 * p.n_chunks * p.W);
    if (in.mom) {
      p.p_sum = ws.take<float>(n);
      p.p_sq = ws.take<float>(n);
    }
    if (in.ext) {
      p.p_mn = ws.take<float>(n);
      p.p_mx = ws.take<float>(n);
      p.p_amin = ws.take<int32_t>(n);
      p.p_amax = ws.take<int32_t>(n);
    }
    if (!ws.ok()) return fail(GNO_ERR_WORKSPACE, "%s: workspace too small (%zu < %zu)", fn, ws_bytes, ws.off);
  }
  const int vb = ma_vectors(p, (uintptr_t)x | (uintptr_t)out, es);
  const int st = (in.mom ? ST_MOMENTS : 0) | (in.ext ? ST_EXTREMES : 0);
  cudaStream_t s = (cudaStream_t)stream;
  switch (dtype) {
    case GNO_F32: return ma_fwd<float>(p, vb, st, true, s);
    case GNO_F16: return ma_fwd<__half>(p, vb, st, true, s);
    default: return ma_fwd<__nv_bfloat16>(p, vb, st, true, s);
  }
}

static int ma_backward_args(const MaInfo& in, const int32_t* arg_min, const int32_t* arg_max, const float* mean,
                            const float* var, const int* aggs, int n_aggs, const char* fn) {
  bool has_min = false, has_max = false;
  for (int a = 0; a < n_aggs; ++a) {
    has_min |= aggs[a] == GNO_AGG_MIN;
    has_max |= aggs[a] == GNO_AGG_MAX;
  }
  GNO_CHECK_ARG((!has_min || arg_min) && (!has_max || arg_max), "%s: winners of min / max are NULL", fn);
  GNO_CHECK_ARG(!in.second || (mean && var), "%s: var / std need the saved mean and var", fn);
  return GNO_OK;
}

int gno_multi_aggregate_backward(const gno_csr* g, const void* x, int64_t x_rows, int64_t T, int64_t F,
                                 const int* aggs, int n_aggs, const int* scalers, int n_scalers, double avg_lin,
                                 double avg_log, const void* grad_out, const int32_t* arg_min,
                                 const int32_t* arg_max, const float* mean, const float* var, void* grad_x,
                                 int dtype, gno_stream_t stream) {
  const char* fn = "gno_multi_aggregate_backward";
  MaInfo in;
  if (int rc = ma_check(g, T, F, aggs, n_aggs, scalers, n_scalers, dtype, fn, &in)) return rc;
  GNO_CHECK_ARG(x_rows >= 0, "%s: bad sizes x_rows=%lld", fn, (long long)x_rows);
  if (g->E == 0 || F == 0) return GNO_OK;
  GNO_CHECK_ARG(g->rowptr && g->erow && x && grad_out && grad_x, "%s: NULL buffer", fn);
  if (int rc = ma_backward_args(in, arg_min, arg_max, mean, var, aggs, n_aggs, fn)) return rc;
  const int es = ma_es(dtype);
  GNO_CHECK_ARG((((uintptr_t)x | (uintptr_t)grad_out | (uintptr_t)grad_x) % es) == 0,
                "%s: buffers not aligned to the element size", fn);
  MaParams p;
  ma_fill(p, g, T, F, aggs, n_aggs, scalers, n_scalers, avg_lin, avg_log, es);
  p.x = static_cast<const char*>(x);
  p.g = static_cast<const char*>(grad_out);
  p.out = grad_x;
  p.amin = const_cast<int32_t*>(arg_min);
  p.amax = const_cast<int32_t*>(arg_max);
  p.mean = in.second ? const_cast<float*>(mean) : nullptr;
  p.var = in.second ? const_cast<float*>(var) : nullptr;
  const int vb = ma_vectors(p, (uintptr_t)x | (uintptr_t)grad_out | (uintptr_t)grad_x, es);
  cudaStream_t s = (cudaStream_t)stream;
  switch (dtype) {
    case GNO_F32: return ma_bwd<float>(p, vb, s);
    case GNO_F16: return ma_bwd<__half>(p, vb, s);
    default: return ma_bwd<__nv_bfloat16>(p, vb, s);
  }
}

int gno_multi_aggregate_coeffs(const gno_csr* g, int64_t T, int64_t F, const int* aggs, int n_aggs,
                               const int* scalers, int n_scalers, double avg_lin, double avg_log,
                               const void* grad_out, const int32_t* arg_min, const int32_t* arg_max,
                               const float* mean, const float* var, float* pq, float* c_min, float* c_max,
                               int dtype, gno_stream_t stream) {
  const char* fn = "gno_multi_aggregate_coeffs";
  MaInfo in;
  if (int rc = ma_check(g, T, F, aggs, n_aggs, scalers, n_scalers, dtype, fn, &in)) return rc;
  if (g->N == 0 || F == 0) return GNO_OK;
  GNO_CHECK_ARG(g->rowptr && grad_out && pq, "%s: NULL buffer", fn);
  if (int rc = ma_backward_args(in, arg_min, arg_max, mean, var, aggs, n_aggs, fn)) return rc;
  GNO_CHECK_ARG(((uintptr_t)grad_out % ma_es(dtype)) == 0, "%s: buffers not aligned to the element size", fn);
  MaParams p;
  ma_fill(p, g, T, F, aggs, n_aggs, scalers, n_scalers, avg_lin, avg_log, ma_es(dtype));
  p.g = static_cast<const char*>(grad_out);
  p.amin = const_cast<int32_t*>(arg_min);
  p.amax = const_cast<int32_t*>(arg_max);
  p.mean = in.second ? const_cast<float*>(mean) : nullptr;
  p.var = in.second ? const_cast<float*>(var) : nullptr;
  p.pq = pq;
  p.cmn = c_min;
  p.cmx = c_max;
  cudaStream_t s = (cudaStream_t)stream;
  switch (dtype) {
    case GNO_F32: return ma_coeffs_launch<float>(p, s);
    case GNO_F16: return ma_coeffs_launch<__half>(p, s);
    default: return ma_coeffs_launch<__nv_bfloat16>(p, s);
  }
}

}  // extern "C"
