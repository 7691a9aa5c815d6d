// Segment reduce over a dst-sorted edge list: the hot kernel of the path.
//
//   out[i, :] = reduce_{k : erow[k] = i}  w[k] * x[gidx[k], :]
//
// EDGE-BALANCED segmented reduction.  The sorted edge list is cut into chunks
// of chunk_len edges; a worker (a group of G lanes, G*VB bytes >= one feature
// row, or a full warp per 32-vector column tile for wide rows) owns one chunk,
// so every worker moves the same number of bytes no matter how skewed the
// degrees are (power-law graphs need no special case).  The edge records of a
// CTA's workers (gather index, destination row, edge id, weight) are one
// contiguous slab per array, staged in shared memory by 1-D TMA bulk copies
// (segreduce_staged_kernel; workers narrower than 16 lanes stage them in
// registers and broadcast by shuffle, segreduce_kernel).  A worker keeps U
// independent VB-byte (16/8/4/2 by alignment) feature-row loads in flight and
// accumulates in fp32 (MIN/MAX over 16-bit data stay packed in the storage
// type: comparisons are exact there).  When the destination row changes it
// writes the finished row; the rows cut by a chunk boundary go to a partial
// buffer (two slots per chunk) and are combined IN CHUNK ORDER by
// segfinish_kernel, which also zero-fills empty rows.  No atomics anywhere:
// results are bit-reproducible, and MIN/MAX ties resolve to the lowest
// original edge position exactly like the sequential upstream CPU loop.
//
// Roofline: HBM.  Algorithmic bytes per edge = F*s (feature row) + 4 (index)
// [+4 erow, +4 eid for arg, +s weight]; per row = F*s_out [+8F arg].
#include <climits>
#include <cstdlib>
#include <type_traits>

#include "segreduce.cuh"

namespace gno {

constexpr int kSegThreads = 128;
constexpr int kSegWarps = kSegThreads / 32;
#ifndef GNO_SEG_MINB
#define GNO_SEG_MINB 8  // 64 registers (32 resident warps/SM); arg-tracking and 16-bit variants get 72 (28 warps)
#endif
#ifndef GNO_SEG_INFLIGHT
#define GNO_SEG_INFLIGHT 64  // bytes of gathered rows in flight per lane (sets the unroll U)
#endif
constexpr int kSegMinBlocks = GNO_SEG_MINB;
// per-head weights are one more gathered value per edge and lane: 80 registers (24 warps/SM) keep
// the unrolled batch of gathers and weights out of local memory; the shuffle-staged kernel with
// 16-bit data in 16-byte vectors needs 96 (20 warps/SM)
constexpr int kSegMinBlocksHeads = 6;
constexpr int kSegMinBlocksHeadsWide = 5;
constexpr int kNoArg = INT_MAX;


// Address of row `idx` of the gather source: two bases, one compare and a select (xcol2 is
// pre-offset by -x2_first rows, so both forms add idx * ldx).
__device__ __forceinline__ const char* gather_addr(const char* xcol, const char* xcol2, unsigned x2_first,
                                                   unsigned idx, unsigned ldx) {
  return (idx >= x2_first ? xcol2 : xcol) + (uint64_t)idx * ldx;
}


template <typename T, int RED>
__device__ __forceinline__ float red_init() {
  if constexpr (RED == GNO_SUM) return 0.f;
  if constexpr (RED == GNO_MUL) return 1.f;
  if constexpr (RED == GNO_MAX) return DType<T>::lowest();
  return DType<T>::highest();
}

// Strict "better than" of the upstream CPU loop: NaNs never win.
template <int RED>
__device__ __forceinline__ bool better(float v, float cur) {
  if constexpr (RED == GNO_MAX) return v > cur;
  return v < cur;
}

// IEEE division kept out of line: flush_row is inlined at every row-boundary site of the
// unrolled loops, and an inline quotient (reciprocal, Newton step, slow-path call) per element
// and per site grew the kernel by two thirds.
__device__ __noinline__ float div_rn_call(float a, float b) { return __fdiv_rn(a, b); }

// Final element transform shared by the direct and the combine path.
// mean: divide the sum by cnt, the row length clamped to 1.  cnt must be a normal number >= 1
// even when mean is off: the compiler evaluates the quotient speculatively, and a zero divisor
// sends every element through the division's slow-path subroutine (ncu source view of the RMAT
// shard: 24 % of all executed instructions before this was fixed).
template <typename T, int RED>
__device__ __forceinline__ float finalize(float a, int e, float prev, bool mean, float cnt,
                                          int accumulate, int64_t arg_fill, int64_t* arg_out) {
  if constexpr (RED == GNO_SUM) {
    if (mean) a = div_rn_call(a, cnt);
    if (accumulate) a += prev;
  } else if constexpr (RED == GNO_MUL) {
    if (accumulate) a *= prev;
  } else {
    if (a == red_init<T, RED>()) a = 0.f;  // no element ever won (torch_scatter masked_fill_)
    if (arg_out) *arg_out = (e == kNoArg) ? arg_fill : (int64_t)e;
  }
  return a;
}

// Per-lane accumulator of one VB-byte vector of a row.  fp32 everywhere, except MIN/MAX over
// 16-bit data: comparisons are exact in the storage type, so the running extremes stay packed
// two to a register and are compared with one HSET2 per pair (the fp32 form cost five
// instructions per element — unpack, compare, two selects — and made the bf16 max+arg kernel
// issue-bound at 0.83 of the HBM roofline).
template <typename T, int VB, int RED, bool HAS_W = false>
struct Accum {
  static constexpr int EPV = VB / (int)sizeof(T);
  // (weighted extremes compare products, which are formed in fp32: no packed form)
  static constexpr bool kPacked = sizeof(T) == 2 && EPV >= 2 && (RED == GNO_MIN || RED == GNO_MAX) && !HAS_W;
  float f[kPacked ? 1 : EPV];
  uint32_t h[kPacked ? EPV / 2 : 1];

  __device__ __forceinline__ void reset() {
    if constexpr (kPacked) {
      const uint32_t b = f_to_bits<T>(red_init<T, RED>()) & 0xffffu;
#pragma unroll
      for (int j = 0; j < EPV / 2; ++j) h[j] = b | (b << 16);
    } else {
#pragma unroll
      for (int i = 0; i < EPV; ++i) f[i] = red_init<T, RED>();
    }
  }
  __device__ __forceinline__ void unpack(float (&out)[EPV]) const {
#pragma unroll
    for (int i = 0; i < EPV; ++i) {
      if constexpr (kPacked) out[i] = bits_to_f<T>((h[i >> 1] >> ((i & 1) * 16)) & 0xffffu);
      else out[i] = f[i];
    }
  }
};

// One packed update: for each 16-bit half of val that is strictly better than the same half of
// acc (ordered compare: NaNs never win, +0.0 and -0.0 tie), take it and record the edge id.
// setp.{gt,lt}.{bf16x2,f16x2} yields one predicate per half; two predicated byte-permutes move
// the winning halves, two predicated moves record the position: five instructions per pair.
#define GNO_PACKED_UPDATE(CMP, TY)                                                         \
  asm("{\n\t.reg .pred p, q;\n\t"                                                         \
      "setp." CMP "." TY " p|q, %3, %0;\n\t"                                               \
      "@p prmt.b32 %0, %0, %3, 0x3254;\n\t"                                                \
      "@q prmt.b32 %0, %0, %3, 0x7610;\n\t"                                                \
      "@p mov.b32 %1, %4;\n\t"                                                             \
      "@q mov.b32 %2, %4;\n\t}"                                                            \
      : "+r"(acc), "+r"(e_lo), "+r"(e_hi)                                                  \
      : "r"(val), "r"(e))
template <typename T, int RED>
__device__ __forceinline__ void packed_update(uint32_t& acc, int& e_lo, int& e_hi, uint32_t val, int e) {
  if constexpr (std::is_same<T, __half>::value) {
    if constexpr (RED == GNO_MAX) GNO_PACKED_UPDATE("gt", "f16x2");
    else GNO_PACKED_UPDATE("lt", "f16x2");
  } else {
    if constexpr (RED == GNO_MAX) GNO_PACKED_UPDATE("gt", "bf16x2");
    else GNO_PACKED_UPDATE("lt", "bf16x2");
  }
}
#undef GNO_PACKED_UPDATE

// Write one finished (or partial) row segment held by a worker.
template <typename T, int VB, int RED, bool ARG>
__device__ __forceinline__ void flush_row(const SegParams& p, int row, int chunk, bool head,
                                          bool tail, int seg_len, int v,
                                          const float (&acc)[VB / (int)sizeof(T)],
                                          const int (&ae)[ARG ? VB / (int)sizeof(T) : 1]) {
  constexpr int EPV = VB / (int)sizeof(T);
  if (head || tail) {
    // a chunk that lies entirely inside one row is both: it uses the head slot
    const int64_t slot = 2 * (int64_t)chunk + (head ? 0 : 1);
    float* pv = p.part_val + slot * p.Fp + (int64_t)v * EPV;
#pragma unroll
    for (int i = 0; i < EPV; ++i) pv[i] = acc[i];
    if constexpr (ARG) {
      int32_t* pa = p.part_arg + slot * p.Fp + (int64_t)v * EPV;
#pragma unroll
      for (int i = 0; i < EPV; ++i) pa[i] = ae[i];
    }
    return;
  }
  const float cnt = (float)(seg_len > 1 ? seg_len : 1);
  const bool mean = p.mean != 0;
  if (p.vec_out) {
    char* optr = static_cast<char*>(p.out) + (int64_t)row * p.ldo_bytes + (int64_t)v * VB;
    Words<VB> prev;
    if (p.accumulate) prev = ld_vec<VB>(optr);
    Words<VB> o;
#pragma unroll
    for (int i = 0; i < EPV; ++i) {
      int64_t* ap = nullptr;
      int e = kNoArg;
      if constexpr (ARG) {
        if (p.arg) ap = p.arg + (int64_t)row * p.F + (int64_t)v * EPV + i;
        e = ae[i];
      }
      const float pf = p.accumulate ? elem<T, VB>(prev, i) : 0.f;
      set_elem<T, VB>(o, i, finalize<T, RED>(acc[i], e, pf, mean, cnt, p.accumulate, p.arg_fill, ap));
    }
    st_vec<VB>(optr, o);
  } else {
    // rows gathered with vectors wider than the output alignment (padded x): element stores,
    // dropping the padding columns.  Rare relative to the gathers.
    T* orow = reinterpret_cast<T*>(static_cast<char*>(p.out) + (int64_t)row * p.ldo_bytes);
#pragma unroll
    for (int i = 0; i < EPV; ++i) {
      const int64_t col = (int64_t)v * EPV + i;
      if (col < p.F) {
        int64_t* ap = nullptr;
        int e = kNoArg;
        if constexpr (ARG) {
          if (p.arg) ap = p.arg + (int64_t)row * p.F + col;
          e = ae[i];
        }
        const float pf = p.accumulate ? DType<T>::to_f(orow[col]) : 0.f;
        orow[col] = DType<T>::from_f(finalize<T, RED>(acc[i], e, pf, mean, cnt, p.accumulate, p.arg_fill, ap));
      }
    }
  }
}

// acc (+= | *= | min | max)= one gathered vector
template <typename T, int VB, int RED, bool ARG, bool HAS_W>
__device__ __forceinline__ void accumulate(Accum<T, VB, RED, HAS_W>& acc,
                                           int (&ae)[ARG ? VB / (int)sizeof(T) : 1],
                                           const Words<VB>& val, int e, float w) {
  constexpr int EPV = VB / (int)sizeof(T);
  if constexpr (Accum<T, VB, RED, HAS_W>::kPacked) {
#pragma unroll
    for (int j = 0; j < EPV / 2; ++j) {
      if constexpr (ARG) {
        packed_update<T, RED>(acc.h[j], ae[2 * j], ae[2 * j + 1], val.w[j], e);
      } else {
        int lo = 0, hi = 0;
        packed_update<T, RED>(acc.h[j], lo, hi, val.w[j], e);
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < EPV; ++i) {
      const float f = elem<T, VB>(val, i);
      if constexpr (RED == GNO_SUM) {
        if constexpr (HAS_W) acc.f[i] = fmaf(w, f, acc.f[i]);
        else acc.f[i] += f;
      } else if constexpr (RED == GNO_MUL) {
        acc.f[i] *= f;
      } else {
        // torch_sparse spmm_min/max with edge values compares value * mat, rounded to the
        // storage type like upstream's scalar_t product
        const float c = HAS_W ? bits_to_f<T>(f_to_bits<T>(w * f) & (sizeof(T) == 2 ? 0xffffu : 0xffffffffu)) : f;
        if (better<RED>(c, acc.f[i])) {
          acc.f[i] = c;
          if constexpr (ARG) ae[i] = e;
        }
      }
    }
  }
}

// flush_row on an Accum (unpacks the packed 16-bit extremes; row boundaries are rare next to edges)
template <typename T, int VB, int RED, bool ARG, typename ACC>
__device__ __forceinline__ void flush_acc(const SegParams& p, int row, int chunk, bool head, bool tail,
                                          int seg_len, int v, const ACC& acc,
                                          const int (&ae)[ARG ? VB / (int)sizeof(T) : 1]) {
  if constexpr (ACC::kPacked) {
    float f[VB / (int)sizeof(T)];
    acc.unpack(f);
    flush_row<T, VB, RED, ARG>(p, row, chunk, head, tail, seg_len, v, f, ae);
  } else {
    flush_row<T, VB, RED, ARG>(p, row, chunk, head, tail, seg_len, v, acc.f, ae);
  }
}

// HEADS (with HAS_W): the weight of a lane's vector is w[eid[k] * H + h] for the head h its columns
// belong to, gathered per lane through the original edge id instead of staged per sorted edge.
template <typename T, int VB, int RED, bool ARG, bool HAS_W, int U, bool HEADS = false>
__global__ void __launch_bounds__(kSegThreads,
                                  HEADS ? (sizeof(T) == 2 && VB == 16 ? kSegMinBlocksHeadsWide : kSegMinBlocksHeads)
                                        : (ARG || sizeof(T) == 2) ? kSegMinBlocks - 1 : kSegMinBlocks)
    segreduce_kernel(const SegParams p) {
  // programmatic dependent launch: the finish kernel may become resident while the last wave runs
  // (it fills the empty rows, then waits for this grid before touching the chunk partials)
  asm volatile("griddepcontrol.launch_dependents;");
  constexpr int EPV = VB / (int)sizeof(T);
  const int lane = threadIdx.x & 31;
  const int G = p.G;
  const int li = lane & (G - 1);  // lane within the worker
  const int gbase = lane - li;
  const int64_t warp = (int64_t)blockIdx.x * kSegWarps + (threadIdx.x >> 5);
  const int64_t wk = warp * (32 / G) + lane / G;
  const int64_t chunk64 = wk / p.ncoltiles;
  const int ct = (int)(wk - chunk64 * p.ncoltiles);
  const int chunk = (int)imin64(chunk64, (int64_t)INT_MAX);
  const int C = p.chunk_len;
  const bool active = chunk64 < p.n_chunks;
  const int64_t k0 = chunk64 * C;
  const int nv = active ? (int)imin64(C, p.E - k0) : 0;  // edges in this chunk
  const int v = ct * 32 + li;
  const bool vact = active && (v < p.nvec);
  const char* xcol = static_cast<const char*>(p.x) + (int64_t)v * VB;
  const unsigned ldx = (unsigned)p.ldx_bytes;
  const unsigned x2f = p.x2_first;
  const char* xcol2 = p.x2 ? static_cast<const char*>(p.x2) - (int64_t)x2f * ldx + (int64_t)v * VB : xcol;
  const bool stream_idx = (p.ncoltiles == 1);
  const uint64_t pol_stream = l2_policy_evict_first();
  const int32_t* erow = p.erow + k0;
  const int32_t* gidx = p.gidx ? p.gidx + k0 : nullptr;
  const int32_t* eid = p.eid ? p.eid + k0 : nullptr;
  const T* wgt = (HAS_W && !HEADS) ? static_cast<const T*>(p.w) + k0 : nullptr;
  const T* whead = HEADS ? static_cast<const T*>(p.w) + (v * EPV) / p.head_c : nullptr;

  Accum<T, VB, RED, HAS_W> acc;
  int ae[ARG ? EPV : 1];
  acc.reset();
  if constexpr (ARG) {
#pragma unroll
    for (int i = 0; i < EPV; ++i) ae[i] = kNoArg;
  }
  int cur_row = active ? __ldg(erow) : 0;
  bool head = active && k0 > 0 && __ldg(erow - 1) == cur_row;
  int seg_start = 0;  // chunk-relative position where cur_row's segment began

  // One staged tile = G edge records, one per lane of the worker.
  auto stage = [&](int t, int& s_idx, int& s_row, int& s_e, float& s_w) {
    const int k = t + li;
    s_idx = 0; s_row = 0; s_e = 0; s_w = 0.f;
    if (k < nv) {
      s_row = stream_idx ? ld_stream_i32(erow + k, pol_stream) : __ldg(erow + k);
      if (gidx) s_idx = stream_idx ? ld_stream_i32(gidx + k, pol_stream) : __ldg(gidx + k);
      else s_idx = (int)(k0 + k);
      if constexpr (ARG || HEADS) {
        if (p.eid == p.gidx) s_e = s_idx;
        else if (eid) s_e = stream_idx ? ld_stream_i32(eid + k, pol_stream) : __ldg(eid + k);
        else s_e = (int)(k0 + k);
      }
      if constexpr (HAS_W && !HEADS) s_w = DType<T>::to_f(wgt[k]);
    }
  };

  int my_idx, my_row, my_e;
  float my_w;
  stage(0, my_idx, my_row, my_e, my_w);
  const int ntiles = C / G;
  // Tiles that are full in EVERY worker of the warp take the fast loop (all of them, except in
  // the warp that holds the last chunk); the rest go through the small generic loop below.
  int nfull = (G >= U) ? __reduce_min_sync(0xffffffffu, nv / G) : 0;
  int ti = 0;
  for (; ti < nfull; ++ti) {
    const int t = ti * G;
    // prefetch the next tile's records while this tile's rows are gathered
    int nx_idx = 0, nx_row = 0, nx_e = 0;
    float nx_w = 0.f;
    if (ti + 1 < ntiles) stage(t + G, nx_idx, nx_row, nx_e, nx_w);
    for (int j = 0; j < G; j += U) {
      Words<VB> val[U];
      int e_u[(ARG || HEADS) ? U : 1];
      float w_u[HAS_W ? U : 1];
      const int lane0 = gbase + j;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int idx = __shfl_sync(0xffffffffu, my_idx, lane0 + u);
        if constexpr (ARG || HEADS) e_u[u] = __shfl_sync(0xffffffffu, my_e, lane0 + u);
        if constexpr (HEADS) w_u[u] = vact ? DType<T>::to_f(whead[(int64_t)e_u[u] * p.H]) : 0.f;
        else if constexpr (HAS_W) w_u[u] = __shfl_sync(0xffffffffu, my_w, lane0 + u);
        if (vact) val[u] = ld_vec<VB>(gather_addr(xcol, xcol2, x2f, (unsigned)idx, ldx));
      }
      // rows ascend: the batch's last row equal to cur_row means no boundary inside it
      const int row_last = __shfl_sync(0xffffffffu, my_row, lane0 + U - 1);
      if (__all_sync(0xffffffffu, row_last == cur_row)) {
        if (vact) {
#pragma unroll
          for (int u = 0; u < U; ++u)
            accumulate<T, VB, RED, ARG, HAS_W>(acc, ae, val[u], ARG ? e_u[ARG ? u : 0] : 0,
                                               HAS_W ? w_u[HAS_W ? u : 0] : 0.f);
        }
      } else {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int row_u = __shfl_sync(0xffffffffu, my_row, lane0 + u);
          if (row_u != cur_row) {  // the previous row ended inside this chunk
            const int kk = t + j + u;
            if (vact)
              flush_acc<T, VB, RED, ARG>(p, cur_row, chunk, head, false, kk - seg_start, v, acc, ae);
            head = false;
            cur_row = row_u;
            seg_start = kk;
            acc.reset();
            if constexpr (ARG) {
#pragma unroll
              for (int i = 0; i < EPV; ++i) ae[i] = kNoArg;
            }
          }
          if (vact)
            accumulate<T, VB, RED, ARG, HAS_W>(acc, ae, val[u], ARG ? e_u[ARG ? u : 0] : 0,
                                               HAS_W ? w_u[HAS_W ? u : 0] : 0.f);
        }
      }
    }
    my_idx = nx_idx; my_row = nx_row; my_e = nx_e; my_w = nx_w;
  }
  // Generic loop (chunk tails, workers narrower than a batch, idle workers of the last warp):
  // one edge at a time — rare, so it is kept small rather than fast.
#pragma unroll 1
  for (; ti < ntiles; ++ti) {
    const int t = ti * G;
    const int rem = nv - t;  // valid edges from this tile on (may be <= 0)
    if (__all_sync(0xffffffffu, rem <= 0)) break;
#pragma unroll 1
    for (int slot = 0; slot < G; ++slot) {
      const int src_lane = gbase + slot;
      const int idx = __shfl_sync(0xffffffffu, my_idx, src_lane);
      const int row_u = __shfl_sync(0xffffffffu, my_row, src_lane);
      int e1 = 0;
      float w1 = 0.f;
      if constexpr (ARG || HEADS) e1 = __shfl_sync(0xffffffffu, my_e, src_lane);
      if constexpr (HAS_W && !HEADS) w1 = __shfl_sync(0xffffffffu, my_w, src_lane);
      if (slot < rem) {
        if constexpr (HEADS) {
          if (vact) w1 = DType<T>::to_f(whead[(int64_t)e1 * p.H]);
        }
        Words<VB> val1;
        if (vact) val1 = ld_vec<VB>(gather_addr(xcol, xcol2, x2f, (unsigned)idx, ldx));
        if (row_u != cur_row) {
          const int kk = t + slot;
          if (vact)
            flush_acc<T, VB, RED, ARG>(p, cur_row, chunk, head, false, kk - seg_start, v, acc, ae);
          head = false;
          cur_row = row_u;
          seg_start = kk;
          acc.reset();
          if constexpr (ARG) {
#pragma unroll
            for (int i = 0; i < EPV; ++i) ae[i] = kNoArg;
          }
        }
        if (vact) accumulate<T, VB, RED, ARG, HAS_W>(acc, ae, val1, e1, w1);
      }
    }
    if (ti + 1 < ntiles) stage(t + G, my_idx, my_row, my_e, my_w);
  }
  if (vact && nv > 0) {
    const bool tail = (k0 + nv < p.E) && (__ldg(erow + nv) == cur_row);
    flush_acc<T, VB, RED, ARG>(p, cur_row, chunk, head, tail, nv - seg_start, v, acc, ae);
  }
}

// ---- TMA-staged variant ------------------------------------------------------------------
// The CTA's workers own consecutive chunks, so their edge records (destination row, gather
// index, edge id, weight) are one contiguous slab per array.  One thread issues a 1-D bulk
// copy (cp.async.bulk → the TMA engine, completion on an mbarrier) per array into shared
// memory; the warps then read records with broadcast LDS instead of per-tile global loads and
// shuffles.  No warp-synchronous operation is left in the loop, so every worker follows its own
// row boundaries without dragging the other workers of its warp through the slow path.
template <typename T, int VB, int RED, bool ARG, bool HAS_W, int U, bool HEADS = false>
__global__ void __launch_bounds__(kSegThreads, HEADS ? kSegMinBlocksHeads
                                              : (ARG || sizeof(T) == 2) ? kSegMinBlocks - 1 : kSegMinBlocks)
    segreduce_staged_kernel(const SegParams p) {
  asm volatile("griddepcontrol.launch_dependents;");  // see segreduce_kernel
  constexpr int EPV = VB / (int)sizeof(T);
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31;
  const int G = p.G;
  const int li = lane & (G - 1);
  const int C = p.chunk_len;
  const int wpc = kSegWarps * (32 / G);  // workers per CTA
  const int64_t w0 = (int64_t)blockIdx.x * wpc;
  const int64_t c_first = w0 / p.ncoltiles;
  if (c_first >= p.n_chunks) return;
  const int64_t c_last = imin64((w0 + wpc - 1) / p.ncoltiles, p.n_chunks - 1);
  const int64_t e0 = c_first * C;
  const int n = (int)(imin64((c_last + 1) * C, p.E) - e0);  // records staged by this CTA
  const int cap = wpc * C;

  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
  int* s_row = reinterpret_cast<int*>(smem_raw + 128);
  int* s_idx = s_row + cap;                       // used when p.gidx
  int* s_e = s_idx + (p.gidx ? cap : 0);          // used when ARG (or HEADS) and a separate eid array
  const bool sep_e = (ARG || HEADS) && p.eid && p.eid != p.gidx;
  constexpr bool W_SLAB = HAS_W && !HEADS;        // per-head weights are gathered, not staged
  T* s_w = reinterpret_cast<T*>(s_e + (sep_e ? cap : 0));

  const bool tma = p.tma_ok && (n % 8 == 0);
  if (tma) {
    if (threadIdx.x == 0) mbar_init(bar, 1);
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t bytes = (uint32_t)n * 4u * (1u + (p.gidx ? 1u : 0u) + (sep_e ? 1u : 0u));
      if (W_SLAB) bytes += (uint32_t)n * (uint32_t)sizeof(T);
      mbar_expect_tx(bar, bytes);
      bulk_g2s(s_row, p.erow + e0, (uint32_t)n * 4u, bar);
      if (p.gidx) bulk_g2s(s_idx, p.gidx + e0, (uint32_t)n * 4u, bar);
      if (sep_e) bulk_g2s(s_e, p.eid + e0, (uint32_t)n * 4u, bar);
      if (W_SLAB) bulk_g2s(s_w, static_cast<const T*>(p.w) + e0, (uint32_t)n * (uint32_t)sizeof(T), bar);
    }
    mbar_wait(bar, 0);
  } else {  // unaligned tail slab (or unaligned caller arrays): plain cooperative copy
    for (int i = threadIdx.x; i < n; i += kSegThreads) {
      s_row[i] = __ldg(p.erow + e0 + i);
      if (p.gidx) s_idx[i] = __ldg(p.gidx + e0 + i);
      if (sep_e) s_e[i] = __ldg(p.eid + e0 + i);
      if (W_SLAB) s_w[i] = static_cast<const T*>(p.w)[e0 + i];
    }
    __syncthreads();
  }

  const int64_t wk = w0 + (threadIdx.x >> 5) * (32 / G) + lane / G;
  const int64_t chunk64 = wk / p.ncoltiles;
  if (chunk64 >= p.n_chunks) return;
  const int ct = (int)(wk - chunk64 * p.ncoltiles);
  const int chunk = (int)chunk64;
  const int64_t k0 = chunk64 * C;
  const int nv = (int)imin64(C, p.E - k0);
  const int soff = (int)(k0 - e0);
  const int v = ct * 32 + li;
  const bool vact = v < p.nvec;
  if (!vact) return;  // no warp-synchronous code below: idle lanes simply leave
  const char* xcol = static_cast<const char*>(p.x) + (int64_t)v * VB;
  const unsigned ldx = (unsigned)p.ldx_bytes;
  const unsigned x2f = p.x2_first;
  const char* xcol2 = p.x2 ? static_cast<const char*>(p.x2) - (int64_t)x2f * ldx + (int64_t)v * VB : xcol;
  const int* rowp = s_row + soff;
  const int* idxp = s_idx + soff;
  const int* ep = (sep_e ? s_e : s_idx) + soff;
  const T* wp = s_w + soff;
  const bool has_idx = p.gidx != nullptr;
  const bool e_is_k = (ARG || HEADS) && !sep_e && !(p.eid && p.eid == p.gidx);  // eid == NULL: edge id = k
  const T* whead = HEADS ? static_cast<const T*>(p.w) + (v * EPV) / p.head_c : nullptr;

  Accum<T, VB, RED, HAS_W> acc;
  int ae[ARG ? EPV : 1];
  acc.reset();
  if constexpr (ARG) {
#pragma unroll
    for (int i = 0; i < EPV; ++i) ae[i] = kNoArg;
  }
  int cur_row = rowp[0];
  bool head = (k0 > 0) && (soff > 0 ? rowp[-1] : __ldg(p.erow + k0 - 1)) == cur_row;
  int seg_start = 0;

  auto close_row = [&](int new_row, int kk) {
    flush_acc<T, VB, RED, ARG>(p, cur_row, chunk, head, false, kk - seg_start, v, acc, ae);
    head = false;
    cur_row = new_row;
    seg_start = kk;
    acc.reset();
    if constexpr (ARG) {
#pragma unroll
      for (int i = 0; i < EPV; ++i) ae[i] = kNoArg;
    }
  };

  int t = 0;
  for (; t + U <= nv; t += U) {
    Words<VB> val[U];
    float wh[HEADS ? U : 1];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int idx = has_idx ? idxp[t + u] : (int)(k0 + t + u);
      val[u] = ld_vec<VB>(gather_addr(xcol, xcol2, x2f, (unsigned)idx, ldx));
      if constexpr (HEADS) wh[u] = DType<T>::to_f(whead[(int64_t)(e_is_k ? (int)(k0 + t + u) : ep[t + u]) * p.H]);
    }
    // rows ascend: the batch's last row equal to cur_row means no boundary inside it
    const bool simple = rowp[t + U - 1] == cur_row;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (!simple) {
        const int row_u = rowp[t + u];
        if (row_u != cur_row) close_row(row_u, t + u);
      }
      int e1 = 0;
      float w1 = 0.f;
      if constexpr (ARG) e1 = e_is_k ? (int)(k0 + t + u) : ep[t + u];
      if constexpr (HEADS) w1 = wh[HEADS ? u : 0];
      else if constexpr (HAS_W) w1 = DType<T>::to_f(wp[t + u]);
      accumulate<T, VB, RED, ARG, HAS_W>(acc, ae, val[u], e1, w1);
    }
  }
#pragma unroll 1
  for (; t < nv; ++t) {  // chunk tail
    const int idx = has_idx ? idxp[t] : (int)(k0 + t);
    const Words<VB> val1 = ld_vec<VB>(gather_addr(xcol, xcol2, x2f, (unsigned)idx, ldx));
    const int row_u = rowp[t];
    if (row_u != cur_row) close_row(row_u, t);
    int e1 = 0;
    float w1 = 0.f;
    if constexpr (ARG) e1 = e_is_k ? (int)(k0 + t) : ep[t];
    if constexpr (HEADS) w1 = DType<T>::to_f(whead[(int64_t)(e_is_k ? (int)(k0 + t) : ep[t]) * p.H]);
    else if constexpr (HAS_W) w1 = DType<T>::to_f(wp[t]);
    accumulate<T, VB, RED, ARG, HAS_W>(acc, ae, val1, e1, w1);
  }
  if (nv > 0) {
    const bool tail = (k0 + nv < p.E) &&
                      ((soff + nv < n) ? rowp[nv] : __ldg(p.erow + k0 + nv)) == cur_row;
    flush_acc<T, VB, RED, ARG>(p, cur_row, chunk, head, tail, nv - seg_start, v, acc, ae);
  }
}

// Empty rows can be filled with 16-byte stores: out rows 16-byte aligned and a multiple of 16
// bytes long (which makes the int64 arg rows multiples of 16 bytes too).
__host__ __device__ static inline bool seg_fill16(const SegParams& p, int es, bool arg) {
  return ((uintptr_t)p.out % 16 == 0) && (p.ldo_bytes % 16 == 0) && ((p.F * es) % 16 == 0) &&
         (!arg || !p.arg || (uintptr_t)p.arg % 16 == 0);
}

// Finish pass: (a) rows cut by a chunk boundary — combine their partials in
// chunk order: the tail slot of the first chunk, then the head slot of every
// later chunk; (b) empty rows — write zeros (and arg_fill).  One thread per
// (row, 4 consecutive features).
template <typename T, int RED, bool ARG>
__global__ void __launch_bounds__(256) segfinish_kernel(const SegParams p) {
  const int64_t Q = (p.F + 3) / 4;  // feature quads per row
  const int64_t n_a = p.n_span * Q;
  // Empty rows are a pure fill: 16-byte stores when the rows allow it (RMAT-26 leaves tens of
  // millions of rows without an edge — at 8 bytes per thread this pass was 14 % of the step).
  constexpr int EPV16 = 16 / (int)sizeof(T);
  const bool fill16 = seg_fill16(p, (int)sizeof(T), ARG);
  const int64_t per_empty = fill16 ? p.F / EPV16 : Q;
  const int64_t total = n_a + (p.accumulate ? 0 : p.n_empty * per_empty);
  const bool vec_val = ((uintptr_t)p.out % (4 * sizeof(T)) == 0) && (p.ldo_bytes % (4 * sizeof(T)) == 0);
  const bool vec_arg = ARG && p.arg && ((uintptr_t)p.arg % 16 == 0) && (p.F % 2 == 0);
  // Phase 1 (items >= n_a): empty rows, which no chunk of the main kernel writes.  Phase 2 (items
  // < n_a): rows cut by a chunk boundary, after griddepcontrol.wait — the main grid has completed
  // and its partials are visible.  Launched with programmatic stream serialization, phase 1 and
  // this kernel's launch latency overlap the tail of the main kernel.
  const int64_t tid0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t tstride = (int64_t)gridDim.x * blockDim.x;
  if (fill16 && !p.accumulate) {
    // Empty-row fill, warp-centric: one coalesced load brings 32 row ids, then the warp issues
    // per_empty independent 512-byte stores (the ids travel by shuffle).  The earlier forms — one
    // id load per 16-byte store, then four — waited on a DRAM-latency load for every 64 bytes
    // stored: 2.9 TB/s on RMAT-26's 40 M empty rows, 29 % of the stall samples on that load
    // (profiles/r3b_finish_rmat26_ncu.txt).
    const float fv = finalize<T, RED>(red_init<T, RED>(), kNoArg, 0.f, false, 1.f, 0, p.arg_fill, nullptr);
    Words<16> o;
#pragma unroll
    for (int q = 0; q < EPV16; ++q) set_elem<T, 16>(o, q, fv);
    const int lane = threadIdx.x & 31;
    const int pe = (int)per_empty;
    const int q32 = 32 / pe, r32 = 32 % pe;
    const int64_t wstride = tstride;           // 32 rows per warp per round
    for (int64_t base = tid0 - lane; base < p.n_empty; base += wstride) {
      const int64_t mine = base + lane < p.n_empty ? (int64_t)__ldg(p.zrow + base + lane) : -1;
      int r = lane / pe, c = lane - r * pe;
      for (int k = 0; k < pe; ++k) {   // item t = lane + 32 k of the 32 * pe pieces: the same trip count in every lane
        const int64_t row = __shfl_sync(0xffffffffu, mine, r);
        if (row >= 0) {
          st_vec<16>(static_cast<char*>(p.out) + row * p.ldo_bytes + (int64_t)c * 16, o);
          if constexpr (ARG) {
            if (p.arg) {
              longlong2* ap = reinterpret_cast<longlong2*>(p.arg + row * p.F + (int64_t)c * EPV16);
#pragma unroll
              for (int q = 0; q < EPV16 / 2; ++q) ap[q] = make_longlong2(p.arg_fill, p.arg_fill);
            }
          }
        }
        c += r32;
        r += q32;
        if (c >= pe) { c -= pe; ++r; }
      }
    }
  }
  for (int phase = (fill16 ? 1 : 0); phase < 2; ++phase) {
  if (phase == 1) asm volatile("griddepcontrol.wait;" ::: "memory");
  const int64_t i_begin = phase == 0 ? n_a + tid0 : tid0;
  const int64_t i_end = phase == 0 ? total : n_a;
  for (int64_t i = i_begin; i < i_end; i += tstride) {
    float a[4];
    int e[4];
    int64_t row, f0;
    if (i < n_a) {
      const int64_t s = i / Q;
      f0 = (i - s * Q) * 4;
      row = p.srow[s];
      const int64_t kb = p.rowptr[row], ke = p.rowptr[row + 1];
      const int64_t ca = kb / p.chunk_len, cb = (ke - 1) / p.chunk_len;
      const float4 t = *reinterpret_cast<const float4*>(p.part_val + (2 * ca + 1) * p.Fp + f0);
      a[0] = t.x; a[1] = t.y; a[2] = t.z; a[3] = t.w;
      if constexpr (ARG) {
        const int4 u = *reinterpret_cast<const int4*>(p.part_arg + (2 * ca + 1) * p.Fp + f0);
        e[0] = u.x; e[1] = u.y; e[2] = u.z; e[3] = u.w;
      } else {
        e[0] = e[1] = e[2] = e[3] = kNoArg;
      }
      // Chunk partials of a hub row can number in the thousands and be nearly equal (one source
      // feeding a hub): summing them in fp32 drifts by ~n*eps/2, so the combine runs in fp64
      // (a few adds per output element; the chunks themselves stay fp32).
      double ad[4] = {(double)a[0], (double)a[1], (double)a[2], (double)a[3]};
      for (int64_t c = ca + 1; c <= cb; ++c) {
        const float4 t2 = *reinterpret_cast<const float4*>(p.part_val + (2 * c) * p.Fp + f0);
        const float pv[4] = {t2.x, t2.y, t2.z, t2.w};
        int pe[4] = {0, 0, 0, 0};
        if constexpr (ARG) {
          const int4 u2 = *reinterpret_cast<const int4*>(p.part_arg + (2 * c) * p.Fp + f0);
          pe[0] = u2.x; pe[1] = u2.y; pe[2] = u2.z; pe[3] = u2.w;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if constexpr (RED == GNO_SUM) {
            ad[j] += (double)pv[j];
          } else if constexpr (RED == GNO_MUL) {
            a[j] *= pv[j];
          } else {
            // chunks ascend in edge position, so a strict compare keeps the lowest
            if (better<RED>(pv[j], a[j])) {
              a[j] = pv[j];
              e[j] = pe[j];
            }
          }
        }
      }
      if constexpr (RED == GNO_SUM) {
        if (p.mean) {
          const double dc = (double)imax64(ke - kb, 1);
#pragma unroll
          for (int j = 0; j < 4; ++j) ad[j] /= dc;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) a[j] = (float)ad[j];
      }
      // (mean already applied above in fp64: finalize is called with mean = false)
    } else {
      const int64_t j = i - n_a;
      const int64_t z = j / Q;
      f0 = (j - z * Q) * 4;
      row = p.zrow[z];
      // no edge: the reduction's identity, which finalize turns into torch_scatter's
      // empty-row value (0 for sum/mean/min/max with arg_fill, 1 for mul)
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        a[q] = red_init<T, RED>();
        e[q] = kNoArg;
      }
    }
    T* orow = reinterpret_cast<T*>(static_cast<char*>(p.out) + row * p.ldo_bytes);
    int64_t* arow = (ARG && p.arg) ? p.arg + row * p.F : nullptr;
    const bool full = (f0 + 4 <= p.F);
    float r[4];
    int64_t ra[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const bool in = (f0 + q < p.F);
      const float prev = (p.accumulate && in) ? DType<T>::to_f(orow[f0 + q]) : 0.f;
      int64_t av = 0;
      r[q] = finalize<T, RED>(a[q], e[q], prev, false, 1.f, p.accumulate, p.arg_fill, arow ? &av : nullptr);
      ra[q] = av;
    }
    if (full && vec_val) {
      Words<4 * sizeof(T)> o;
#pragma unroll
      for (int q = 0; q < 4; ++q) set_elem<T, 4 * sizeof(T)>(o, q, r[q]);
      st_vec<4 * sizeof(T)>(reinterpret_cast<char*>(orow + f0), o);
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (f0 + q < p.F) orow[f0 + q] = DType<T>::from_f(r[q]);
    }
    if constexpr (ARG) {
      if (arow) {
        if (full && vec_arg) {
          *reinterpret_cast<longlong2*>(arow + f0) = make_longlong2(ra[0], ra[1]);
          *reinterpret_cast<longlong2*>(arow + f0 + 2) = make_longlong2(ra[2], ra[3]);
        } else {
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (f0 + q < p.F) arow[f0 + q] = ra[q];
        }
      }
    }
  }
  }  // phase
}

// ------------------------------------------------------------- dispatch --
// Shared memory the staged kernel needs for one CTA's record slab.
static int64_t seg_staged_bytes(const SegParams& p, int es, bool arg, bool has_w) {
  const int64_t cap = (int64_t)kSegWarps * (32 / p.G) * p.chunk_len;
  const bool sep_e = arg && p.eid && p.eid != p.gidx;
  return cap * 4 * (1 + (p.gidx ? 1 : 0) + (sep_e ? 1 : 0)) + (has_w ? cap * es : 0);
}

// The finish pass behind a chunk kernel (after_kernel: it was launched just before, so this one
// may start early under programmatic stream serialization).
template <typename T, int RED, bool ARG>
static int launch_segfinish(const SegParams& p, bool after_kernel, cudaStream_t s) {
  const int64_t quads = (p.F + 3) / 4;
  const int64_t per_empty = seg_fill16(p, (int)sizeof(T), ARG) ? p.F / (16 / (int64_t)sizeof(T)) : quads;
  const int64_t total = p.n_span * quads + (p.accumulate ? 0 : p.n_empty * per_empty);
  if (total > 0) {
    const int grid = (int)imin64(ceil_div(total, 256), (int64_t)kNumSMs * 16);
    static const int pdl_env = getenv("GNO_SEG_PDL") ? atoi(getenv("GNO_SEG_PDL")) : 1;
    if (after_kernel && pdl_env) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3((unsigned)grid);
      cfg.blockDim = dim3(256);
      cfg.dynamicSmemBytes = 0;
      cfg.stream = s;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      at[0].val.programmaticStreamSerializationAllowed = 1;
      cfg.attrs = at;
      cfg.numAttrs = 1;
      GNO_CUDA(cudaLaunchKernelEx(&cfg, segfinish_kernel<T, RED, ARG>, p));
    } else {
      segfinish_kernel<T, RED, ARG><<<grid, 256, 0, s>>>(p);
    }
    GNO_LAUNCHED("segfinish_kernel");
  }
  return GNO_OK;
}

template <typename T, int VB, int RED, bool ARG, bool HAS_W, bool HEADS = false>
static int launch_seg(const SegParams& p, cudaStream_t s) {
  constexpr int U0 = (GNO_SEG_INFLIGHT / VB) > 16 ? 16 : (GNO_SEG_INFLIGHT / VB);
  // per-head weights add a gathered value per unrolled edge: half the batch keeps them in registers
  constexpr int U = (HEADS && U0 > 1) ? U0 / 2 : U0;
  const int64_t workers = p.n_chunks * p.ncoltiles;
  const int64_t warps = ceil_div(workers, 32 / p.G);
  const int64_t blocks = ceil_div(warps, kSegWarps);
  static const int carve = getenv("GNO_SEG_CARVEOUT") ? atoi(getenv("GNO_SEG_CARVEOUT")) : -1;
  if (carve >= 0) {
    GNO_CUDA(cudaFuncSetAttribute(segreduce_staged_kernel<T, VB, RED, ARG, HAS_W, U, HEADS>,
                                  cudaFuncAttributePreferredSharedMemoryCarveout, carve));
  }
  if (blocks > 0 && p.staged) {
    const size_t smem = 128 + (size_t)seg_staged_bytes(p, (int)sizeof(T), ARG || HEADS, HAS_W && !HEADS);
    segreduce_staged_kernel<T, VB, RED, ARG, HAS_W, U, HEADS><<<(unsigned)blocks, kSegThreads, smem, s>>>(p);
    GNO_LAUNCHED("segreduce_staged_kernel");
  } else if (blocks > 0) {
    segreduce_kernel<T, VB, RED, ARG, HAS_W, U, HEADS><<<(unsigned)blocks, kSegThreads, 0, s>>>(p);
    GNO_LAUNCHED("segreduce_kernel");
  }
  return launch_segfinish<T, RED, ARG>(p, blocks > 0, s);
}

template <typename T, int VB>
static int dispatch_red(const SegParams& p, int reduce, bool /*with_arg*/, bool has_w,
                        cudaStream_t s) {
  switch (reduce) {
    case GNO_SUM:
    case GNO_MEAN:
      if (p.H > 0) return launch_seg<T, VB, GNO_SUM, false, true, true>(p, s);
      return has_w ? launch_seg<T, VB, GNO_SUM, false, true>(p, s)
                   : launch_seg<T, VB, GNO_SUM, false, false>(p, s);
    case GNO_MUL:
      return launch_seg<T, VB, GNO_MUL, false, false>(p, s);
    // MIN/MAX always track the winner's position (even with arg == NULL) so
    // that ties between +0.0 and -0.0 resolve to the first occurrence, which
    // keeps the VALUES bit-identical to the sequential upstream loop.
    case GNO_MIN:
      return has_w ? launch_seg<T, VB, GNO_MIN, true, true>(p, s) : launch_seg<T, VB, GNO_MIN, true, false>(p, s);
    case GNO_MAX:
      return has_w ? launch_seg<T, VB, GNO_MAX, true, true>(p, s) : launch_seg<T, VB, GNO_MAX, true, false>(p, s);
  }
  return fail(GNO_ERR_INVALID, "gno_segment_reduce: unknown reduce %d", reduce);
}

template <typename T>
static int dispatch_vb(const SegParams& p, int vb, int reduce, bool with_arg, bool has_w,
                       cudaStream_t s) {
  switch (vb) {
    case 16: return dispatch_red<T, 16>(p, reduce, with_arg, has_w, s);
    case 8: return dispatch_red<T, 8>(p, reduce, with_arg, has_w, s);
    case 4: return dispatch_red<T, 4>(p, reduce, with_arg, has_w, s);
    case 2:
      if constexpr (sizeof(T) == 2) return dispatch_red<T, 2>(p, reduce, with_arg, has_w, s);
  }
  return fail(GNO_ERR_INVALID, "gno_segment_reduce: bad vector width %d", vb);
}

static int dtype_size(int dtype) { return dtype == GNO_F32 ? 4 : 2; }

int seg_finish_sum(const SegParams& p, int dtype, bool after_kernel, cudaStream_t s) {
  switch (dtype) {
    case GNO_F32: return launch_segfinish<float, GNO_SUM, false>(p, after_kernel, s);
    case GNO_F16: return launch_segfinish<__half, GNO_SUM, false>(p, after_kernel, s);
    default: return launch_segfinish<__nv_bfloat16, GNO_SUM, false>(p, after_kernel, s);
  }
}

// ---- per-edge, per-head dot product (gradient of the per-head weights) ----------------------
//   ga[eid[k] * H + h] = sum_c go[erow[k], h*C + c] * x[gidx[k], h*C + c]
// One thread per (sorted edge, head); the H threads of an edge read the two rows whole.  Edges
// arrive dst-sorted, so consecutive edges share their go row: it is read from DRAM once per row
// and from L1 for the rest of the row's edges.  fp32 accumulation, one rounding.
template <typename T, int VB>
__global__ void __launch_bounds__(256) edge_head_dot_kernel(const int32_t* __restrict__ erow,
                                                            const int32_t* __restrict__ gidx,
                                                            const int32_t* __restrict__ eid,
                                                            const char* __restrict__ x,
                                                            const char* __restrict__ go, T* __restrict__ ga,
                                                            int64_t total, int H, int64_t row_bytes,
                                                            int nvh, bool narrow) {
  constexpr int EPV = VB / (int)sizeof(T);
  const int64_t t = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (t >= total) return;
  const int64_t k = narrow ? (int64_t)((uint32_t)t / (uint32_t)H) : t / H;
  const int h = (int)(t - k * H);
  const int64_t row = __ldg(erow + k);
  const int64_t s = gidx ? (int64_t)__ldg(gidx + k) : k;
  const int64_t e = eid ? (int64_t)__ldg(eid + k) : k;
  const char* xp = x + s * row_bytes + (int64_t)h * nvh * VB;
  const char* gp = go + row * row_bytes + (int64_t)h * nvh * VB;
  float acc = 0.f;
  for (int j = 0; j < nvh; ++j) {
    const Words<VB> a = ld_vec<VB>(xp + j * VB);
    const Words<VB> b = ld_vec<VB>(gp + j * VB);
#pragma unroll
    for (int i = 0; i < EPV; ++i) acc = fmaf(elem<T, VB>(b, i), elem<T, VB>(a, i), acc);
  }
  ga[e * H + h] = DType<T>::from_f(acc);
}

template <typename T>
static int launch_edge_head_dot(const gno_csr* g, const void* x, const void* go, void* ga, int64_t H,
                                int64_t F, cudaStream_t s) {
  const int es = (int)sizeof(T);
  const int64_t total = g->E * H;
  if (total == 0 || F == 0) return GNO_OK;
  const int vb = head_vector_bytes(F / H * es, (uintptr_t)x | (uintptr_t)go, es);
  const int nvh = (int)(F / H * es / vb);
  const unsigned blocks = (unsigned)ceil_div(total, 256);
  const bool narrow = total < (int64_t(1) << 32);
  const char* xc = static_cast<const char*>(x);
  const char* gc = static_cast<const char*>(go);
  T* out = static_cast<T*>(ga);
  switch (vb) {
    case 16: edge_head_dot_kernel<T, 16><<<blocks, 256, 0, s>>>(g->erow, g->gidx, g->eid, xc, gc, out, total, (int)H, F * es, nvh, narrow); break;
    case 8: edge_head_dot_kernel<T, 8><<<blocks, 256, 0, s>>>(g->erow, g->gidx, g->eid, xc, gc, out, total, (int)H, F * es, nvh, narrow); break;
    case 4: edge_head_dot_kernel<T, 4><<<blocks, 256, 0, s>>>(g->erow, g->gidx, g->eid, xc, gc, out, total, (int)H, F * es, nvh, narrow); break;
    default:
      if constexpr (sizeof(T) == 2) {
        edge_head_dot_kernel<T, 2><<<blocks, 256, 0, s>>>(g->erow, g->gidx, g->eid, xc, gc, out, total, (int)H, F * es, nvh, narrow);
        break;
      }
      return fail(GNO_ERR_INVALID, "gno_edge_head_dot: bad vector width %d", vb);
  }
  GNO_LAUNCHED("edge_head_dot_kernel");
  return GNO_OK;
}

}  // namespace gno

using namespace gno;

extern "C" {

int gno_segment_reduce_workspace(const gno_csr* g, int64_t F, int dtype, int reduce, int with_arg,
                                 size_t* bytes) {
  GNO_CHECK_ARG(g && bytes, "gno_segment_reduce_workspace: NULL argument");
  GNO_CHECK_ARG(g->chunk_len >= 32 && g->chunk_len % 32 == 0, "gno_segment_reduce: bad chunk_len");
  (void)dtype;
  (void)with_arg;
  WorkspaceSizer sz;
  const int64_t n_chunks = ceil_div(g->E, g->chunk_len);
  if (n_chunks > 0) {
    const int64_t Fp = (F + 7) / 8 * 8;
    sz.take<float>((size_t)(2 * n_chunks * Fp));
    if (reduce == GNO_MIN || reduce == GNO_MAX) sz.take<int32_t>((size_t)(2 * n_chunks * Fp));
  }
  *bytes = sz.total();
  return GNO_OK;
}

int gno_segment_reduce(const gno_csr* g, const void* x, int64_t x_rows, int64_t ldx, const void* w,
                       void* out, int64_t ldo, int64_t* arg, int64_t arg_fill, int64_t F, int dtype,
                       int reduce, int accumulate, void* wsp, size_t ws_bytes,
                       gno_stream_t stream) {
  return gno_segment_reduce_two(g, x, x_rows, ldx, nullptr, 0, w, out, ldo, arg, arg_fill, F, dtype, reduce,
                                accumulate, wsp, ws_bytes, stream);
}

}  // extern "C"

// heads > 0: per-head weights (gno_segment_reduce_heads), w is [*, heads] read through g->eid.
static int segment_reduce_impl(const gno_csr* g, const void* x, int64_t x_rows, int64_t ldx, const void* x2,
                               int64_t x2_rows, const void* w, void* out, int64_t ldo, int64_t* arg,
                               int64_t arg_fill, int64_t F, int dtype, int reduce, int accumulate, void* wsp,
                               size_t ws_bytes, gno_stream_t stream, int64_t heads) {
  cudaStream_t s = (cudaStream_t)stream;
  GNO_CHECK_ARG(x2 == nullptr || (x2_rows >= 0 && x_rows + x2_rows < (int64_t(1) << 31)),
                "gno_segment_reduce_two: x_rows + x2_rows must stay below 2^31");
  GNO_CHECK_ARG(g != nullptr, "gno_segment_reduce: graph is NULL");
  GNO_CHECK_ARG(dtype == GNO_F32 || dtype == GNO_F16 || dtype == GNO_BF16,
                "gno_segment_reduce: unknown dtype %d", dtype);
  GNO_CHECK_ARG(reduce >= GNO_SUM && reduce <= GNO_MAX, "gno_segment_reduce: unknown reduce %d", reduce);
  GNO_CHECK_ARG(g->N >= 0 && g->E >= 0 && g->E < (int64_t(1) << 31) && F >= 0 && ldx >= F && ldo >= F,
                "gno_segment_reduce: bad sizes N=%lld E=%lld F=%lld ldx=%lld ldo=%lld",
                (long long)g->N, (long long)g->E, (long long)F, (long long)ldx, (long long)ldo);
  GNO_CHECK_ARG(g->chunk_len >= 32 && g->chunk_len % 32 == 0 && g->chunk_len <= (1 << 20),
                "gno_segment_reduce: chunk_len must be a multiple of 32");
  if (g->N == 0 || F == 0) return GNO_OK;
  GNO_CHECK_ARG(g->rowptr && out && (g->E == 0 || (x && g->erow)), "gno_segment_reduce: NULL buffer");
  GNO_CHECK_ARG(x_rows >= 0, "gno_segment_reduce: x_rows < 0");
  GNO_CHECK_ARG((g->n_span == 0 || g->srow) && (g->n_empty == 0 || g->zrow),
                "gno_segment_reduce: row lists missing");
  const bool with_arg = (arg != nullptr);
  GNO_CHECK_ARG(!with_arg || reduce == GNO_MIN || reduce == GNO_MAX,
                "gno_segment_reduce: arg output only for MIN/MAX");
  GNO_CHECK_ARG(!accumulate || reduce == GNO_SUM || reduce == GNO_MUL,
                "gno_segment_reduce: accumulate only for SUM/MUL");
  if (w != nullptr && reduce == GNO_MUL)
    return fail(GNO_ERR_UNSUPPORTED, "gno_segment_reduce: edge weights with MUL are not defined upstream");

  const int es = dtype_size(dtype);
  GNO_CHECK_ARG((((uintptr_t)x | (uintptr_t)x2 | (uintptr_t)out) % es) == 0,
                "gno_segment_reduce: buffers not aligned to the element size");
  // Widest gather vector the row starts of x allow.  A row whose length is not a multiple of it
  // is still read with full vectors when the row stride leaves room for the over-read (x padded
  // by the caller, e.g. F=602: 1204-byte bf16 rows stored with a 1216-byte stride); the extra
  // columns are dropped on output.
  const uintptr_t ax = (uintptr_t)x | (uintptr_t)x2 | (uintptr_t)(ldx * es);
  int vb = 16;
  while (vb > es && (ax % vb) != 0) vb >>= 1;
  while (vb > es && (F * es) % vb != 0 && ceil_div(F * es, vb) * vb > ldx * es) vb >>= 1;
  if (heads > 0) vb = head_vector_bytes(F / heads * es, (uintptr_t)vb, es);  // a vector stays inside one head
  const uintptr_t ao = (uintptr_t)out | (uintptr_t)(ldo * es) | (uintptr_t)(F * es);

  SegParams p;
  p.gidx = g->gidx;
  p.eid = g->eid;
  p.erow = g->erow;
  p.x = x;
  p.x2 = x2;
  p.x2_first = x2 ? (unsigned)x_rows : 0xffffffffu;
  p.w = w;
  p.out = out;
  p.arg = arg;
  p.rowptr = g->rowptr;
  p.srow = g->srow;
  p.zrow = g->zrow;
  p.N = g->N;
  p.E = g->E;
  p.chunk_len = (int)g->chunk_len;
  p.n_chunks = ceil_div(g->E, g->chunk_len);
  p.n_span = g->n_span;
  p.n_empty = g->n_empty;
  p.F = F;
  p.Fp = (F + 7) / 8 * 8;
  p.vec_out = (ao % vb) == 0;
  p.ldx_bytes = ldx * es;
  p.ldo_bytes = ldo * es;
  p.arg_fill = arg_fill;
  p.nvec = (int)ceil_div(F * es, vb);
  p.ncoltiles = (p.nvec + 31) / 32;
  int G = 1;
  while (G < p.nvec && G < 32) G <<= 1;
  p.G = G;
  p.mean = (reduce == GNO_MEAN);
  p.accumulate = accumulate ? 1 : 0;
  p.H = (int)heads;
  p.head_c = heads > 0 ? (int)(F / heads) : 0;
  p.part_val = nullptr;
  p.part_arg = nullptr;
  if (p.n_chunks > 0) {
    if (wsp == nullptr) return fail(GNO_ERR_WORKSPACE, "gno_segment_reduce: workspace is NULL");
    Workspace ws(wsp, ws_bytes);
    p.part_val = ws.take<float>((size_t)(2 * p.n_chunks * p.Fp));
    if (reduce == GNO_MIN || reduce == GNO_MAX)
      p.part_arg = ws.take<int32_t>((size_t)(2 * p.n_chunks * p.Fp));
    if (!ws.ok())
      return fail(GNO_ERR_WORKSPACE, "gno_segment_reduce: workspace too small (%zu < %zu)", ws_bytes, ws.off);
  }
  const bool has_w = (w != nullptr);
  {
    const bool argv = (reduce == GNO_MIN || reduce == GNO_MAX);
    const bool hd = heads > 0;
    const uintptr_t al = (uintptr_t)g->erow | (uintptr_t)g->gidx | (uintptr_t)(argv || hd ? g->eid : nullptr) |
                         (uintptr_t)(hd ? nullptr : w);
    p.tma_ok = (al % 16) == 0;
    static const int staged_env = getenv("GNO_SEG_STAGED") ? atoi(getenv("GNO_SEG_STAGED")) : 1;
    p.staged = staged_env && seg_staged_bytes(p, es, argv || hd, has_w && !hd) <= 24 * 1024;
  }
  switch (dtype) {
    case GNO_F32: return dispatch_vb<float>(p, vb, reduce, with_arg, has_w, s);
    case GNO_F16: return dispatch_vb<__half>(p, vb, reduce, with_arg, has_w, s);
    case GNO_BF16: return dispatch_vb<__nv_bfloat16>(p, vb, reduce, with_arg, has_w, s);
  }
  return fail(GNO_ERR_INVALID, "gno_segment_reduce: unknown dtype %d", dtype);
}

extern "C" {

int gno_segment_reduce_two(const gno_csr* g, const void* x, int64_t x_rows, int64_t ldx, const void* x2,
                           int64_t x2_rows, const void* w, void* out, int64_t ldo, int64_t* arg,
                           int64_t arg_fill, int64_t F, int dtype, int reduce, int accumulate, void* wsp,
                           size_t ws_bytes, gno_stream_t stream) {
  return segment_reduce_impl(g, x, x_rows, ldx, x2, x2_rows, w, out, ldo, arg, arg_fill, F, dtype, reduce,
                             accumulate, wsp, ws_bytes, stream, 0);
}

int gno_segment_reduce_heads(const gno_csr* g, const void* x, int64_t x_rows, const void* alpha, int64_t H,
                             void* out, int64_t F, int dtype, void* ws, size_t ws_bytes, gno_stream_t stream) {
  GNO_CHECK_ARG(dtype == GNO_F32 || dtype == GNO_F16 || dtype == GNO_BF16,
                "gno_segment_reduce_heads: unknown dtype %d", dtype);
  GNO_CHECK_ARG(H > 0 && H < (int64_t(1) << 20) && F >= 0 && F % H == 0 && x_rows >= 0,
                "gno_segment_reduce_heads: bad sizes H=%lld F=%lld x_rows=%lld", (long long)H, (long long)F,
                (long long)x_rows);
  GNO_CHECK_ARG(g == nullptr || g->E == 0 || F == 0 || alpha != nullptr, "gno_segment_reduce_heads: alpha is NULL");
  return segment_reduce_impl(g, x, x_rows, F, nullptr, 0, alpha, out, F, nullptr, 0, F, dtype, GNO_SUM, 0, ws,
                             ws_bytes, stream, H);
}

int gno_edge_head_dot(const gno_csr* g, const void* x, int64_t x_rows, const void* grad_out, int64_t H,
                      int64_t F, void* grad_alpha, int dtype, gno_stream_t stream) {
  GNO_CHECK_ARG(g != nullptr, "gno_edge_head_dot: graph is NULL");
  GNO_CHECK_ARG(dtype == GNO_F32 || dtype == GNO_F16 || dtype == GNO_BF16, "gno_edge_head_dot: unknown dtype %d",
                dtype);
  GNO_CHECK_ARG(H > 0 && H < (int64_t(1) << 20) && F >= 0 && F % H == 0 && x_rows >= 0 && g->N >= 0 &&
                    g->E >= 0 && g->E < (int64_t(1) << 31),
                "gno_edge_head_dot: bad sizes H=%lld F=%lld x_rows=%lld E=%lld", (long long)H, (long long)F,
                (long long)x_rows, (long long)g->E);
  if (g->E == 0 || F == 0) return GNO_OK;
  GNO_CHECK_ARG(g->erow && x && grad_out && grad_alpha, "gno_edge_head_dot: NULL buffer");
  const int es = dtype_size(dtype);
  GNO_CHECK_ARG((((uintptr_t)x | (uintptr_t)grad_out | (uintptr_t)grad_alpha) % es) == 0,
                "gno_edge_head_dot: buffers not aligned to the element size");
  cudaStream_t s = (cudaStream_t)stream;
  switch (dtype) {
    case GNO_F32: return launch_edge_head_dot<float>(g, x, grad_out, grad_alpha, H, F, s);
    case GNO_F16: return launch_edge_head_dot<__half>(g, x, grad_out, grad_alpha, H, F, s);
    default: return launch_edge_head_dot<__nv_bfloat16>(g, x, grad_out, grad_alpha, H, F, s);
  }
}

}  // extern "C"
