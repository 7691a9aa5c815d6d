// Segment-reduce parameters, vector load/store helpers and the finish pass, shared by
// segreduce.cu and the kernels that write its chunk-partial layout (gatv2.cu).
#pragma once
#include "common.cuh"

namespace gno {

struct SegParams {
  const int32_t* gidx;
  const int32_t* eid;
  const int32_t* erow;
  const void* x;
  const void* x2;      // second gather base (gno_segment_reduce_two): gather ids >= x2_first read row id - x2_first of x2
  const void* w;
  void* out;
  int64_t* arg;
  float* part_val;    // [2 * n_chunks, F] fp32 partials of rows cut by a chunk boundary
  int32_t* part_arg;  // [2 * n_chunks, F]
  const int64_t* rowptr;
  const int32_t* srow;
  const int32_t* zrow;
  int64_t N, E, n_chunks, n_span, n_empty;
  int64_t F;
  int64_t Fp;  // row stride of the partial buffers: F rounded up to 8 elements
  int64_t ldx_bytes, ldo_bytes;
  int64_t arg_fill;
  int chunk_len;  // edges per worker
  int nvec;       // vectors per row
  int ncoltiles;  // column tiles of 32 vectors
  int G;          // lanes per worker (power of two; 32 when ncoltiles > 1)
  int mean;       // divide by max(row length, 1)
  int accumulate;
  int vec_out;    // out rows are aligned for VB-byte vector stores and F*s is a multiple of VB
  int tma_ok;     // edge-record arrays are 16-byte aligned (bulk copies allowed)
  int staged;     // use the TMA-staged kernel (record slab of a CTA fits the shared-memory budget)
  unsigned x2_first;  // 0xffffffff when there is no second base (no gather id reaches it)
  int H;              // per-head weights (gno_segment_reduce_heads): w is [*, H], read at w[eid * H + h]
  int head_c;         // columns per head; a gathered vector never straddles two heads
};

template <int VB>
struct Words {
  static constexpr int n = VB >= 4 ? VB / 4 : 1;
  uint32_t w[n];
};

template <int VB>
__device__ __forceinline__ Words<VB> ld_vec(const char* p) {
  Words<VB> r;
  if constexpr (VB == 16) {
    const uint4 q = __ldg(reinterpret_cast<const uint4*>(p));
    r.w[0] = q.x; r.w[1] = q.y; r.w[2] = q.z; r.w[3] = q.w;
  } else if constexpr (VB == 8) {
    const uint2 q = __ldg(reinterpret_cast<const uint2*>(p));
    r.w[0] = q.x; r.w[1] = q.y;
  } else if constexpr (VB == 4) {
    r.w[0] = __ldg(reinterpret_cast<const uint32_t*>(p));
  } else {
    r.w[0] = __ldg(reinterpret_cast<const unsigned short*>(p));
  }
  return r;
}
template <int VB>
__device__ __forceinline__ void st_vec(char* p, const Words<VB>& r) {
  if constexpr (VB == 16) {
    *reinterpret_cast<uint4*>(p) = make_uint4(r.w[0], r.w[1], r.w[2], r.w[3]);
  } else if constexpr (VB == 8) {
    *reinterpret_cast<uint2*>(p) = make_uint2(r.w[0], r.w[1]);
  } else if constexpr (VB == 4) {
    *reinterpret_cast<uint32_t*>(p) = r.w[0];
  } else {
    *reinterpret_cast<unsigned short*>(p) = (unsigned short)r.w[0];
  }
}

template <typename T>
__device__ __forceinline__ float bits_to_f(uint32_t b);
template <>
__device__ __forceinline__ float bits_to_f<float>(uint32_t b) { return __uint_as_float(b); }
template <>
__device__ __forceinline__ float bits_to_f<__half>(uint32_t b) {
  return __half2float(__ushort_as_half((unsigned short)b));
}
template <>
__device__ __forceinline__ float bits_to_f<__nv_bfloat16>(uint32_t b) {
  return __uint_as_float(b << 16);
}
template <typename T>
__device__ __forceinline__ uint32_t f_to_bits(float f);
template <>
__device__ __forceinline__ uint32_t f_to_bits<float>(float f) { return __float_as_uint(f); }
template <>
__device__ __forceinline__ uint32_t f_to_bits<__half>(float f) {
  return __half_as_ushort(__float2half_rn(f));
}
template <>
__device__ __forceinline__ uint32_t f_to_bits<__nv_bfloat16>(float f) {
  return __bfloat16_as_ushort(__float2bfloat16_rn(f));
}

template <typename T, int VB>
__device__ __forceinline__ float elem(const Words<VB>& r, int i) {
  if constexpr (sizeof(T) == 4) {
    return bits_to_f<T>(r.w[i]);
  } else {
    return bits_to_f<T>((r.w[i >> 1] >> ((i & 1) * 16)) & 0xffffu);
  }
}
template <typename T, int VB>
__device__ __forceinline__ void set_elem(Words<VB>& r, int i, float f) {
  if constexpr (sizeof(T) == 4) {
    r.w[i] = f_to_bits<T>(f);
  } else {
    const uint32_t b = f_to_bits<T>(f) & 0xffffu;
    if (i & 1)
      r.w[i >> 1] |= b << 16;
    else
      r.w[i >> 1] = b;
  }
}

// Widest vector (16/8/4/2 bytes) that divides one head's bytes and the alignment `a`.
static inline int head_vector_bytes(int64_t head_bytes, uintptr_t a, int es) {
  int vb = 16;
  while (vb > es && ((a % vb) != 0 || head_bytes % vb != 0)) vb >>= 1;
  return vb;
}

// Finish pass of a SUM (segfinish_kernel) over p's partials: rows cut by a chunk boundary get the
// sum of their chunk partials in chunk order, empty rows get 0.  `after_kernel`: launched right
// behind the kernel that wrote the partials, with programmatic stream serialization.
int seg_finish_sum(const SegParams& p, int dtype, bool after_kernel, cudaStream_t s);

}  // namespace gno
