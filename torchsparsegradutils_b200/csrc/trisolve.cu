// trisolve.cu -- level-scheduled sparse triangular solve op(A) X = B for sm_100a (sync-free, one row per warp).
//
//   tsgu_trisolve_levels   level[r] = 1 + max level[j] over the dependencies j of row r, plus per-row dependency
//                          counts and the level count (one-off per pattern and triangle)
//   tsgu_trisolve_plan     rows in level order -> per slot the strictly off-diagonal entries of the triangle
//                          (flat dependency row, value position) and the diagonal's value position
//   tsgu_trisolve          the solve over a plan
//
// Protocol.  A warp takes its row with a global atomicAdd ticket, in plan order, so a row can only wait on rows
// with a lower ticket, and those are held by warps that are already running: no deadlock at any grid size or
// occupancy.  For every dependency j the warp spins on ready[j] with a gpu-scope acquire load, reads x[j, :] with
// L2 loads (__ldcg: L1 may hold lines read before the flag was set), stores its own row, fences, and sets ready[r]
// with a release store.  Each row is summed in a fixed entry order and no atomics touch values, so results are
// bit-identical from run to run.  Every wait is bounded (about a second of __nanosleep back-off): past the bound the
// warp writes NaN to its row, still releases its flag and sets the status word, so the kernel always terminates.
#include <cuda/atomic>
#include <math.h>

#include "common.cuh"

namespace tsgu {
namespace {

constexpr int kTriThreads = 256;  // 8 warps, one row each at a time
constexpr unsigned long long kWaitBoundNs = 1000000000ull;
// workspace: [0] uint64 ticket, [8] uint32 status, [12] pad, [16...] uint32 ready flag per row
constexpr size_t kFlagsOffset = 16;

__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// Spin until *flag != 0 (acquire, gpu scope) and return it; 0 once the wait bound has passed.
__device__ __forceinline__ unsigned wait_flag(unsigned* flag) {
  cuda::atomic_ref<unsigned, cuda::thread_scope_device> ref(*flag);
  unsigned v = ref.load(cuda::memory_order_acquire);
  if (v) return v;
  for (int i = 0; i < 64; ++i) {  // a dependency one level down is usually a few hundred ns away: poll hot first
    v = ref.load(cuda::memory_order_acquire);
    if (v) return v;
  }
  const unsigned long long t0 = global_ns();
  unsigned ns = 32;
  for (;;) {
    __nanosleep(ns);
    if (ns < 1024) ns *= 2;
    v = ref.load(cuda::memory_order_acquire);
    if (v) return v;
    if (global_ns() - t0 > kWaitBoundNs) return 0;
  }
}

__device__ __forceinline__ void release_flag(unsigned* flag, unsigned v) {
  cuda::atomic_ref<unsigned, cuda::thread_scope_device>(*flag).store(v, cuda::memory_order_release);
}

__device__ __forceinline__ int64_t take_ticket(unsigned long long* ticket, int lane) {
  unsigned long long s = 0;
  if (lane == 0) s = atomicAdd(ticket, 1ull);
  return (int64_t)__shfl_sync(0xffffffffu, s, 0);
}

// Does entry column c of row r belong to the strictly off-diagonal part of the solved triangle?
__device__ __forceinline__ bool is_dep(int64_t c, int64_t r, bool lower) { return lower ? c < r : c > r; }

// ------------------------------------------------------------------------------------------ level analysis
// Ticket s -> flat row s (lower: dependencies have smaller rows) or rows-1-s (upper).  The ready flag of a row is its
// level (>= 1), so the level values themselves are the dependency flags.
template <typename I>
__global__ void __launch_bounds__(kTriThreads) trisolve_levels_kernel(
    const I* __restrict__ rowptr, const I* __restrict__ colind, int64_t batch, int64_t n, int64_t rowptr_bstride,
    int64_t nnz_bstride, bool lower, unsigned char* __restrict__ ws, int64_t* __restrict__ level_out,
    int64_t* __restrict__ count_out, unsigned long long* __restrict__ stats) {
  unsigned long long* ticket = reinterpret_cast<unsigned long long*>(ws);
  unsigned* ready = reinterpret_cast<unsigned*>(ws + kFlagsOffset);
  const int lane = threadIdx.x & 31;
  const int64_t rows = batch * n;
  for (;;) {
    const int64_t s = take_ticket(ticket, lane);
    if (s >= rows) return;
    const int64_t g = lower ? s : rows - 1 - s;
    const int64_t t = g / n, r = g - t * n;
    const int64_t lo = (int64_t)__ldg(rowptr + t * rowptr_bstride + r) + t * nnz_bstride;
    const int64_t hi = (int64_t)__ldg(rowptr + t * rowptr_bstride + r + 1) + t * nnz_bstride;
    unsigned lvl = 0, cnt = 0;
    bool ok = true;
    for (int64_t e = lo + lane; e < hi; e += 32) {
      const int64_t c = (int64_t)__ldg(colind + e);
      if (is_dep(c, r, lower)) {
        ++cnt;
        const unsigned v = wait_flag(ready + t * n + c);
        ok = ok && v != 0;
        lvl = max(lvl, v);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lvl = max(lvl, __shfl_xor_sync(0xffffffffu, lvl, o));
      cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    }
    const bool timed_out = __any_sync(0xffffffffu, !ok);
    if (lane == 0) {
      ++lvl;
      level_out[g] = (int64_t)lvl - 1;
      count_out[g] = (int64_t)cnt;
      atomicMax(stats + 0, (unsigned long long)lvl);
      atomicAdd(stats + 1, (unsigned long long)cnt);
      if (timed_out) atomicOr(stats + 2, 1ull);
      release_flag(ready + g, lvl);
    }
  }
}

// ------------------------------------------------------------------------------------------ plan fill
// One thread per slot (one-off per pattern): the dependencies of row order[s] in storage order.
template <typename I>
__global__ void __launch_bounds__(256) trisolve_plan_kernel(
    const I* __restrict__ rowptr, const I* __restrict__ colind, const I* __restrict__ perm, int64_t batch, int64_t n,
    int64_t rowptr_bstride, int64_t nnz_bstride, bool lower, const I* __restrict__ order,
    const I* __restrict__ plan_rowptr, I* __restrict__ plan_col, I* __restrict__ plan_pos, I* __restrict__ plan_diag) {
  const int64_t rows = batch * n;
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < rows; s += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = (int64_t)order[s];
    const int64_t t = g / n, r = g - t * n;
    const int64_t lo = (int64_t)rowptr[t * rowptr_bstride + r] + t * nnz_bstride;
    const int64_t hi = (int64_t)rowptr[t * rowptr_bstride + r + 1] + t * nnz_bstride;
    int64_t out = (int64_t)plan_rowptr[s];
    int64_t diag = -1;
    for (int64_t e = lo; e < hi; ++e) {
      const int64_t c = (int64_t)colind[e];
      const int64_t p = perm ? (int64_t)perm[e] : e;
      if (c == r) {
        if (diag < 0) diag = p;
      } else if (is_dep(c, r, lower)) {
        plan_col[out] = (I)(t * n + c);
        plan_pos[out] = (I)p;
        ++out;
      }
    }
    plan_diag[s] = (I)diag;
  }
}

// ------------------------------------------------------------------------------------------ the solve
template <typename V> __device__ __forceinline__ V nan_value();
template <> __device__ __forceinline__ float nan_value<float>() { return __int_as_float(0x7fffffff); }
template <> __device__ __forceinline__ double nan_value<double>() { return __longlong_as_double(0x7ff8000000000000ll); }

template <typename V, int VEC> struct XVec;
template <typename V> struct XVec<V, 1> {
  __device__ static __forceinline__ void load(const V* p, V (&v)[1]) { v[0] = __ldcg(p); }
  __device__ static __forceinline__ void store(V* p, const V (&v)[1]) { p[0] = v[0]; }
};
template <> struct XVec<float, 4> {
  __device__ static __forceinline__ void load(const float* p, float (&v)[4]) {
    const float4 q = __ldcg(reinterpret_cast<const float4*>(p));
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
  }
  __device__ static __forceinline__ void store(float* p, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};
template <> struct XVec<double, 2> {
  __device__ static __forceinline__ void load(const double* p, double (&v)[2]) {
    const double2 q = __ldcg(reinterpret_cast<const double2*>(p));
    v[0] = q.x; v[1] = q.y;
  }
  __device__ static __forceinline__ void store(double* p, const double (&v)[2]) {
    *reinterpret_cast<double2*>(p) = make_double2(v[0], v[1]);
  }
};

constexpr int kEntryModeMaxK = 4;  // K <= 4: lanes over the row's entries + shuffle reduction

// ENTRY = true: lanes run over the row's entries (each lane waits on its own dependencies), K <= 4 partial sums per
// lane, xor-tree reduction.  ENTRY = false: the lanes first wait on all dependencies together, then run over K in
// VEC-wide vectors while the warp walks the entries in order.
template <typename V, typename I, int VEC, bool ENTRY>
__global__ void __launch_bounds__(kTriThreads) trisolve_kernel(
    const I* __restrict__ plan_rowptr, const I* __restrict__ plan_col, const I* __restrict__ plan_pos,
    const I* __restrict__ plan_diag, const I* __restrict__ order, const V* __restrict__ vals, const V* __restrict__ B,
    V* X, int64_t rows, int64_t n, int64_t K, int64_t b_bs, int64_t b_rs, int64_t b_cs, bool unit,
    unsigned char* __restrict__ ws) {
  unsigned long long* ticket = reinterpret_cast<unsigned long long*>(ws);
  unsigned* status = reinterpret_cast<unsigned*>(ws + 8);
  unsigned* ready = reinterpret_cast<unsigned*>(ws + kFlagsOffset);
  const int lane = threadIdx.x & 31;
  for (;;) {
    const int64_t s = take_ticket(ticket, lane);
    if (s >= rows) return;
    const int64_t g = (int64_t)__ldg(order + s);
    const int64_t t = g / n, r = g - t * n;
    const int64_t lo = (int64_t)__ldg(plan_rowptr + s), hi = (int64_t)__ldg(plan_rowptr + s + 1);
    const V* b = B + t * b_bs + r * b_rs;
    V* x = X + g * K;
    V d = V(1);
    if (!unit) {
      const int64_t p = (int64_t)__ldg(plan_diag + s);
      d = p >= 0 ? __ldg(vals + p) : V(0);  // a missing diagonal divides by zero, as the dense solve does
    }
    bool ok = true;
    if constexpr (ENTRY) {
      V acc[kEntryModeMaxK] = {};
      for (int64_t e = lo + lane; e < hi; e += 32) {
        const int64_t j = (int64_t)__ldg(plan_col + e);
        const V a = __ldg(vals + (int64_t)__ldg(plan_pos + e));
        ok = wait_flag(ready + j) != 0 && ok;
        const V* xj = X + j * K;
#pragma unroll
        for (int k = 0; k < kEntryModeMaxK; ++k)
          if (k < K) acc[k] = fma(a, __ldcg(xj + k), acc[k]);
      }
#pragma unroll
      for (int k = 0; k < kEntryModeMaxK; ++k)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
      const bool timed_out = __any_sync(0xffffffffu, !ok);
#pragma unroll
      for (int k = 0; k < kEntryModeMaxK; ++k)
        if (lane == k && k < K) x[k] = timed_out ? nan_value<V>() : (__ldg(b + k * b_cs) - acc[k]) / d;
      if (timed_out && lane == 0) atomicOr(status, 1u);
    } else {
      for (int64_t e = lo + lane; e < hi; e += 32) ok = wait_flag(ready + (int64_t)__ldg(plan_col + e)) != 0 && ok;
      const bool timed_out = __any_sync(0xffffffffu, !ok);
      __syncwarp();  // orders every lane's acquires before all lanes' reads of the dependency rows
      for (int64_t k0 = (int64_t)lane * VEC; k0 < K; k0 += 32 * VEC) {
        V acc[VEC] = {};
        for (int64_t e = lo; e < hi; ++e) {
          const int64_t j = (int64_t)__ldg(plan_col + e);
          const V a = __ldg(vals + (int64_t)__ldg(plan_pos + e));
          V xv[VEC];
          XVec<V, VEC>::load(X + j * K + k0, xv);
#pragma unroll
          for (int v = 0; v < VEC; ++v) acc[v] = fma(a, xv[v], acc[v]);
        }
        V out[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) out[v] = timed_out ? nan_value<V>() : (__ldg(b + (k0 + v) * b_cs) - acc[v]) / d;
        XVec<V, VEC>::store(x + k0, out);
      }
      if (timed_out && lane == 0) atomicOr(status, 1u);
    }
    __threadfence();  // every lane's stores of row g are visible at gpu scope before its flag
    __syncwarp();
    if (lane == 0) release_flag(ready + g, 1u);
  }
}

inline unsigned tri_grid(int64_t rows) {
  const int64_t warps_per_block = kTriThreads / 32;
  const int64_t want = (rows + warps_per_block - 1) / warps_per_block;
  const int64_t cap = (int64_t)persistent_sms() * (2048 / kTriThreads);  // rows are pulled by tickets, not blockIdx
  return (unsigned)(want < 1 ? 1 : (want < cap ? want : cap));
}

inline size_t tri_ws_bytes(int64_t rows) { return (kFlagsOffset + (size_t)rows * 4 + 255) / 256 * 256; }

template <typename V, typename I>
int trisolve_launch(const void* plan_rowptr, const void* plan_col, const void* plan_pos, const void* plan_diag,
                    const void* order, const void* vals, const void* B, void* X, int64_t rows, int64_t n, int64_t K,
                    int64_t b_bs, int64_t b_rs, int64_t b_cs, bool unit, unsigned char* ws, cudaStream_t s) {
  constexpr int kVec = 16 / (int)sizeof(V);
  const unsigned grid = tri_grid(rows);
  const bool vec = K % kVec == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0;
#define TSGU_TRI_ARGS                                                                                              \
  (const I*)plan_rowptr, (const I*)plan_col, (const I*)plan_pos, (const I*)plan_diag, (const I*)order,          \
      (const V*)vals, (const V*)B, (V*)X, rows, n, K, b_bs, b_rs, b_cs, unit, ws
  if (K <= kEntryModeMaxK) trisolve_kernel<V, I, 1, true><<<grid, kTriThreads, 0, s>>>(TSGU_TRI_ARGS);
  else if (vec) trisolve_kernel<V, I, kVec, false><<<grid, kTriThreads, 0, s>>>(TSGU_TRI_ARGS);
  else trisolve_kernel<V, I, 1, false><<<grid, kTriThreads, 0, s>>>(TSGU_TRI_ARGS);
#undef TSGU_TRI_ARGS
  count_launch();
  return launch_status();
}

}  // namespace
}  // namespace tsgu

using namespace tsgu;

extern "C" size_t tsgu_trisolve_workspace_bytes(int64_t batch, int64_t n) {
  return batch < 1 || n < 0 ? 0 : tri_ws_bytes(batch * n);
}

extern "C" int tsgu_trisolve_levels(const void* rowptr, const void* colind, int64_t batch, int64_t n,
                                    int64_t rowptr_bstride, int64_t nnz_bstride, int idx_dtype, int lower,
                                    void* level_out, void* count_out, void* stats_out, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  if (batch < 1 || n < 0) return TSGU_ERR_SHAPE;
  if (idx_dtype != TSGU_I32 && idx_dtype != TSGU_I64) return TSGU_ERR_DTYPE;
  const int64_t rows = batch * n;
  if (rows >= 0xffffffffLL) return TSGU_ERR_RANGE;  // levels travel as 32-bit flags
  cudaStream_t s = as_stream(stream);
  cudaError_t e = cudaMemsetAsync(stats_out, 0, 3 * sizeof(unsigned long long), s);
  if (e != cudaSuccess) return (int)e;
  if (rows == 0) return 0;
  if (!workspace || workspace_bytes < tri_ws_bytes(rows)) return TSGU_ERR_WORKSPACE;
  e = cudaMemsetAsync(workspace, 0, tri_ws_bytes(rows), s);
  if (e != cudaSuccess) return (int)e;
  TSGU_DISPATCH_IDX(idx_dtype, {
    trisolve_levels_kernel<I><<<tri_grid(rows), kTriThreads, 0, s>>>(
        (const I*)rowptr, (const I*)colind, batch, n, rowptr_bstride, nnz_bstride, lower != 0,
        (unsigned char*)workspace, (int64_t*)level_out, (int64_t*)count_out, (unsigned long long*)stats_out);
    count_launch();
  });
  return launch_status();
}

extern "C" int tsgu_trisolve_plan(const void* rowptr, const void* colind, const void* perm, int64_t batch, int64_t n,
                                  int64_t rowptr_bstride, int64_t nnz_bstride, int idx_dtype, int lower,
                                  const void* order, const void* plan_rowptr, void* plan_col, void* plan_pos,
                                  void* plan_diag, void* stream) {
  if (batch < 1 || n < 0) return TSGU_ERR_SHAPE;
  const int64_t rows = batch * n;
  if (rows == 0) return 0;
  cudaStream_t s = as_stream(stream);
  const int64_t blocks = (rows + 255) / 256;
  TSGU_DISPATCH_IDX(idx_dtype, {
    trisolve_plan_kernel<I><<<(unsigned)(blocks < 65535 * 16 ? blocks : 65535 * 16), 256, 0, s>>>(
        (const I*)rowptr, (const I*)colind, (const I*)perm, batch, n, rowptr_bstride, nnz_bstride, lower != 0,
        (const I*)order, (const I*)plan_rowptr, (I*)plan_col, (I*)plan_pos, (I*)plan_diag);
    count_launch();
  });
  return launch_status();
}

extern "C" int tsgu_trisolve(const void* plan_rowptr, const void* plan_col, const void* plan_pos,
                             const void* plan_diag, const void* order, const void* vals, const void* B, void* X,
                             int64_t batch, int64_t n, int64_t K, int64_t b_bs, int64_t b_rs, int64_t b_cs,
                             int unitriangular, int val_dtype, int idx_dtype, void* workspace, size_t workspace_bytes,
                             void* stream) {
  if (batch < 1 || n < 0 || K < 0) return TSGU_ERR_SHAPE;
  if (val_dtype != TSGU_F32 && val_dtype != TSGU_F64) return TSGU_ERR_DTYPE;
  if (idx_dtype != TSGU_I32 && idx_dtype != TSGU_I64) return TSGU_ERR_DTYPE;
  const int64_t rows = batch * n;
  if (rows == 0 || K == 0) return 0;
  if (!workspace || workspace_bytes < tri_ws_bytes(rows)) return TSGU_ERR_WORKSPACE;
  cudaStream_t s = as_stream(stream);
  cudaError_t e = cudaMemsetAsync(workspace, 0, tri_ws_bytes(rows), s);
  if (e != cudaSuccess) return (int)e;
  const bool unit = unitriangular != 0;
  unsigned char* ws = (unsigned char*)workspace;
  if (val_dtype == TSGU_F32) {
    if (idx_dtype == TSGU_I32)
      return trisolve_launch<float, int32_t>(plan_rowptr, plan_col, plan_pos, plan_diag, order, vals, B, X, rows, n, K, b_bs, b_rs, b_cs, unit, ws, s);
    return trisolve_launch<float, int64_t>(plan_rowptr, plan_col, plan_pos, plan_diag, order, vals, B, X, rows, n, K, b_bs, b_rs, b_cs, unit, ws, s);
  }
  if (idx_dtype == TSGU_I32)
    return trisolve_launch<double, int32_t>(plan_rowptr, plan_col, plan_pos, plan_diag, order, vals, B, X, rows, n, K, b_bs, b_rs, b_cs, unit, ws, s);
  return trisolve_launch<double, int64_t>(plan_rowptr, plan_col, plan_pos, plan_diag, order, vals, B, X, rows, n, K, b_bs, b_rs, b_cs, unit, ws, s);
}
