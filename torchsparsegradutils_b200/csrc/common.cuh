// common.cuh -- dtype traits, 128-bit vector access, launch bookkeeping (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "../../include/tsgu_b200.h"

namespace tsgu {

// ---------------------------------------------------------------- launch accounting
extern unsigned long long g_launches;  // defined in api.cu
inline void count_launch(int k = 1) { __atomic_fetch_add(&g_launches, (unsigned long long)k, __ATOMIC_RELAXED); }
inline int launch_status() {
  cudaError_t e = cudaPeekAtLastError();
  return e == cudaSuccess ? 0 : (int)e;
}
inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

// SMs the persistent kernels leave free (tsgu_set_sm_margin; per calling thread).  A persistent grid of
// 148 x resident-CTAs owns every SM, so a kernel that should run CONCURRENTLY (NCCL's reduction kernels while the
// grad_B collective of row sharding overlaps the SDDMM) finds no slot until the grid drains.
extern thread_local int g_sm_margin;  // defined in api.cu
inline int64_t persistent_sms() {
  const int m = g_sm_margin;
  return m > 0 && m < kNumSMs ? kNumSMs - m : kNumSMs;
}

// ---------------------------------------------------------------- value-type traits
template <typename V> struct VT;
template <> struct VT<float> {
  using Acc = float;
  __device__ static __forceinline__ float to_acc(float v) { return v; }
  __device__ static __forceinline__ float from_acc(float a) { return a; }
};
template <> struct VT<double> {
  using Acc = double;
  __device__ static __forceinline__ double to_acc(double v) { return v; }
  __device__ static __forceinline__ double from_acc(double a) { return a; }
};
template <> struct VT<__nv_bfloat16> {
  using Acc = float;  // bf16 storage, fp32 accumulate
  __device__ static __forceinline__ float to_acc(__nv_bfloat16 v) { return __bfloat162float(v); }
  __device__ static __forceinline__ __nv_bfloat16 from_acc(float a) { return __float2bfloat16_rn(a); }
};

// ---------------------------------------------------------------- raw vectors of EPV elements
// Raw<V,EPV> is the register image of one load: 16 B (uint4), 8 B (uint2), or one scalar.
template <int BYTES> struct RawBits;
template <> struct RawBits<16> { using T = uint4; };
template <> struct RawBits<8> { using T = uint2; };
template <> struct RawBits<4> { using T = uint32_t; };
template <> struct RawBits<2> { using T = uint16_t; };

template <typename V, int EPV> struct Raw {
  using Bits = typename RawBits<sizeof(V) * EPV>::T;
  Bits bits;
};

template <typename V, int EPV>
__device__ __forceinline__ Raw<V, EPV> raw_zero() {
  Raw<V, EPV> r;
  if constexpr (sizeof(V) * EPV == 16) r.bits = make_uint4(0, 0, 0, 0);
  else if constexpr (sizeof(V) * EPV == 8) r.bits = make_uint2(0, 0);
  else r.bits = 0;
  return r;
}

// read-only path load (ld.global.nc), L1-allocating: B / G rows are re-used by neighbouring rows
template <typename V, int EPV>
__device__ __forceinline__ Raw<V, EPV> raw_ldg(const V* p) {
  Raw<V, EPV> r;
  r.bits = __ldg(reinterpret_cast<const typename Raw<V, EPV>::Bits*>(p));
  return r;
}

template <typename V, int EPV>
__device__ __forceinline__ void raw_unpack(const Raw<V, EPV>& r, typename VT<V>::Acc (&out)[EPV]) {
  if constexpr (EPV == 1) {
    if constexpr (sizeof(V) == 2) {
      out[0] = __uint_as_float(((uint32_t)r.bits) << 16);
    } else if constexpr (sizeof(V) == 4) {
      out[0] = __uint_as_float(r.bits);
    } else {
      out[0] = __longlong_as_double((long long)(((unsigned long long)r.bits.y << 32) | r.bits.x));
    }
  } else if constexpr (sizeof(V) == 4) {  // 4 x fp32
    out[0] = __uint_as_float(r.bits.x); out[1] = __uint_as_float(r.bits.y);
    out[2] = __uint_as_float(r.bits.z); out[3] = __uint_as_float(r.bits.w);
  } else if constexpr (sizeof(V) == 8) {  // 2 x fp64
    out[0] = __longlong_as_double((long long)(((unsigned long long)r.bits.y << 32) | r.bits.x));
    out[1] = __longlong_as_double((long long)(((unsigned long long)r.bits.w << 32) | r.bits.z));
  } else {  // 8 x bf16: bf16 -> fp32 is a 16-bit shift
    const uint32_t w[4] = {r.bits.x, r.bits.y, r.bits.z, r.bits.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      out[2 * i] = __uint_as_float(w[i] << 16);
      out[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
}

template <typename V, int EPV>
__device__ __forceinline__ void store_vec(V* p, const typename VT<V>::Acc (&a)[EPV]) {
  if constexpr (EPV == 1) {
    p[0] = VT<V>::from_acc(a[0]);
  } else if constexpr (sizeof(V) == 4) {
    *reinterpret_cast<float4*>(p) = make_float4(a[0], a[1], a[2], a[3]);
  } else if constexpr (sizeof(V) == 8) {
    *reinterpret_cast<double2*>(p) = make_double2(a[0], a[1]);
  } else {
    uint4 o;
    uint32_t* w = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 h = __floats2bfloat162_rn(a[2 * i], a[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t*>(&h);
    }
    *reinterpret_cast<uint4*>(p) = o;
  }
}

// scalar value load as accumulator type
template <typename V>
__device__ __forceinline__ typename VT<V>::Acc load_scalar(const V* p) {
  return VT<V>::to_acc(__ldg(p));
}
template <>
__device__ __forceinline__ float load_scalar<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __uint_as_float(((uint32_t)__ldg(reinterpret_cast<const unsigned short*>(p))) << 16);
}

// sub-warp group helpers ---------------------------------------------------------------
template <int LPR>
__device__ __forceinline__ unsigned group_mask(int lane) {
  if constexpr (LPR == 32) return 0xffffffffu;
  else return ((1u << LPR) - 1u) << ((lane / LPR) * LPR);
}

template <typename T>
__device__ __forceinline__ T shfl_idx(unsigned mask, T v, int src, int width) {
  return __shfl_sync(mask, v, src, width);
}
template <typename T>
__device__ __forceinline__ T shfl_x(unsigned mask, T v, int lanemask) {
  return __shfl_xor_sync(mask, v, lanemask);
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// L2 capacity of the current device (126 MB on B200), queried once per process.
inline int64_t l2_bytes() {
  static int64_t cached = 0;
  if (cached == 0) {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&v, cudaDevAttrL2CacheSize, dev) == cudaSuccess && v > 0)
      cached = v;
    else
      cached = 96ll << 20;
  }
  return cached;
}

// Problems with fewer rows than this cannot fill 148 SMs with row tiles and take the non-persistent
// row-split kernels (one CTA per 256/LPR rows).  TSGU_TINY_ROWS overrides it (the parity tests set it to 0
// so that small, oracle-sized inputs exercise every persistent-tile kernel variant).
inline int64_t tiny_rows_threshold() {
  const char* e = getenv("TSGU_TINY_ROWS");
  return e ? atoll(e) : (int64_t)64 * 2 * kNumSMs;
}

// K-slicing for L2 residency.  When one item of the dense operand (rows x K) does not fit L2, every
// gathered row is an HBM access and the kernel runs at HBM-gather speed (config 5: 6.6 TB/s).  Cutting K
// into slices whose rows x Ks footprint fits L2 and running the slices as back-to-back launches turns
// the re-reads of a row (once per nonzero of that column) into L2 hits; the sparse structure is re-read
// once per slice, which is small next to the dense traffic.  Returns Ks (== K: do not slice).
// Measured on config 5 (fp32, K = 512 -> 8 slices of 64): forward SpMM over uniform rows 0.646 -> 0.496 ms,
// but the SDDMM (0.62 -> 0.68 ms) and the SpMM over the ragged transposed rows (0.64 -> 0.87 ms: narrower lane
// groups put 4 rows of different lengths in one warp) lose.  So slicing is on only where the caller says the
// rows are uniform (`allow`: TSGU_ALGO_FLAG_KSLICE, forward SpMM); env TSGU_L2_SLICE_FRAC=<share of L2 per
// slice> forces it everywhere (experiments), <= 0 disables it.
inline int64_t pick_k_slice(int64_t rows, int64_t K, int elem_bytes, bool allow = false) {
  const int64_t l2 = l2_bytes();
  const int64_t epv = 16 / elem_bytes;
  static double env_frac = -2.0;  // -2: not read yet; -1: unset
  if (env_frac == -2.0) {
    const char* e = getenv("TSGU_L2_SLICE_FRAC");
    env_frac = e ? atof(e) : -1.0;
  }
  double frac;
  if (env_frac != -1.0) frac = env_frac;
  else frac = allow ? 0.55 : 0.0;
  if (frac <= 0.0 || rows * K * elem_bytes <= (l2 * 3) / 5) return K;
  for (int64_t parts = 2; parts <= 64; parts *= 2) {
    if (K % parts) break;
    const int64_t ks = K / parts;
    if (ks % (4 * epv)) break;  // keep at least 4 lanes x 16 B per row segment
    if ((double)(rows * ks * elem_bytes) <= frac * (double)l2) return ks;
  }
  return K;
}

}  // namespace tsgu

// Dispatch helpers ---------------------------------------------------------------------
#define TSGU_DISPATCH_VAL(vdt, ...)                                        \
  switch (vdt) {                                                           \
    case TSGU_F32: { using V = float; __VA_ARGS__; break; }                \
    case TSGU_F64: { using V = double; __VA_ARGS__; break; }               \
    case TSGU_BF16: { using V = __nv_bfloat16; __VA_ARGS__; break; }       \
    default: return TSGU_ERR_DTYPE;                                        \
  }
#define TSGU_DISPATCH_IDX(idt, ...)                                        \
  switch (idt) {                                                           \
    case TSGU_I32: { using I = int32_t; __VA_ARGS__; break; }              \
    case TSGU_I64: { using I = int64_t; __VA_ARGS__; break; }              \
    default: return TSGU_ERR_DTYPE;                                        \
  }
