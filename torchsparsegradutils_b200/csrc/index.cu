// index.cu -- integer index builders for sm_100a (bit-exact work, one-off per sparsity pattern).
//
//   tsgu_coo_sort         stable radix sort of (batch,row,col) keys + permutation
//                         (reference utils/utils.py:148-149: torch.unique(sorted) + argsort)
//   tsgu_coo_to_csr       sorted COO -> flat CSR (rowptr by run-boundary detection, no atomics)
//                         (reference utils/utils.py:228-231 bincount+cumsum, :327-344 batch loop)
//   tsgu_compress_rows    histogram + scan for arbitrary-order rows (utils/utils.py:152-233)
//   tsgu_decompress_crow  crow -> row per entry (utils/utils.py:413-470, sparse_matmul.py:190-192)
//   tsgu_csr_transpose    radix-sort/scan transpose (implicit A.t() of sparse_matmul.py:229)
//
// The device-wide radix sort and prefix scan are CUB's (ships with the CUDA toolkit); everything
// around them (key packing, run-boundary rowptr fill, gathers) is hand-written.  All outputs are
// deterministic: the sort is stable and rowptr is derived from run boundaries, never from float or
// order-dependent atomics.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace tsgu {

static inline int bits_for(uint64_t count) {  // bits needed to represent values in [0, count)
  int b = 1;
  while (b < 64 && (count - 1) >> b) ++b;
  return count <= 1 ? 1 : b;
}
static inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }
static inline unsigned blocks_for(int64_t items, int threads) {
  int64_t b = (items + threads - 1) / threads;
  if (b < 1) b = 1;
  if (b > 0x7fffffffLL) b = 0x7fffffffLL;
  return (unsigned)b;
}

// largest r in [0, len) with a[r] <= x, for non-decreasing a with a[0] <= x  (upper_bound - 1)
template <typename I>
__device__ __forceinline__ int64_t row_of(const I* __restrict__ a, int64_t len, int64_t x) {
  int64_t lo = 0, hi = len;  // invariant: a[lo] <= x, (hi == len or a[hi] > x)
  while (hi - lo > 1) {
    const int64_t mid = lo + ((hi - lo) >> 1);
    if ((int64_t)__ldg(a + mid) <= x) lo = mid; else hi = mid;
  }
  return lo;
}

// ------------------------------------------------------------------------------ COO sort
template <typename KeyT, typename P>
__global__ void coo_pack_keys_kernel(const int64_t* __restrict__ idx, int64_t idx_ld, int key_dims,
                                     int64_t d1, int64_t d2, int64_t nnz, KeyT* __restrict__ keys,
                                     P* __restrict__ iota) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += (int64_t)gridDim.x * blockDim.x) {
    uint64_t k = (uint64_t)idx[e];
    if (key_dims > 1) k = k * (uint64_t)d1 + (uint64_t)idx[idx_ld + e];
    if (key_dims > 2) k = k * (uint64_t)d2 + (uint64_t)idx[2 * idx_ld + e];
    keys[e] = (KeyT)k;
    iota[e] = (P)e;
  }
}

template <typename P>
__global__ void coo_gather_sorted_kernel(const int64_t* __restrict__ idx, int64_t idx_ld, int ndim, int64_t nnz,
                                         const P* __restrict__ perm, int64_t* __restrict__ sorted) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += (int64_t)gridDim.x * blockDim.x) {
    const int64_t src = (int64_t)perm[k];
    for (int d = 0; d < ndim; ++d) sorted[(int64_t)d * nnz + k] = idx[(int64_t)d * idx_ld + src];
  }
}

template <typename KeyT, typename P>
static cudaError_t cub_sort_pairs(void* tmp, size_t& tmp_bytes, const KeyT* kin, KeyT* kout, const P* vin,
                                  P* vout, int64_t n, int end_bit, cudaStream_t s) {
  return cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, kin, kout, vin, vout, n, 0, end_bit, s);
}

template <typename KeyT, typename P>
static size_t sort_ws_bytes(int64_t nnz) {
  size_t cub_bytes = 0;
  cudaError_t e = cub_sort_pairs<KeyT, P>(nullptr, cub_bytes, nullptr, nullptr, nullptr, nullptr, nnz, 8 * (int)sizeof(KeyT), 0);
  if (e != cudaSuccess) {  // no device (CPU-only box): conservative bound, never used for a launch
    (void)cudaGetLastError();
    cub_bytes = (size_t)nnz * (sizeof(KeyT) + sizeof(P)) + (1u << 20);
  }
  return 2 * align_up((size_t)nnz * sizeof(KeyT)) + align_up((size_t)nnz * sizeof(P)) + align_up(cub_bytes);
}

// workspace carving shared by coo_sort and csr_transpose
template <typename KeyT, typename P>
struct SortWs {
  KeyT* kin; KeyT* kout; P* vin; void* cub; size_t cub_bytes;
  SortWs(void* ws, size_t ws_bytes, int64_t nnz) {
    char* p = (char*)ws;
    kin = (KeyT*)p; p += align_up((size_t)nnz * sizeof(KeyT));
    kout = (KeyT*)p; p += align_up((size_t)nnz * sizeof(KeyT));
    vin = (P*)p; p += align_up((size_t)nnz * sizeof(P));
    cub = p;
    cub_bytes = (size_t)((char*)ws + ws_bytes - p);
  }
};

template <typename KeyT, typename P>
static int coo_sort_impl(const int64_t* idx, int ndim, int64_t nnz, int64_t idx_ld, const int64_t* dims,
                         int key_dims, int key_bits, int64_t* sorted_idx, P* perm, void* ws, size_t ws_bytes,
                         cudaStream_t s) {
  if (ws_bytes < sort_ws_bytes<KeyT, P>(nnz)) return TSGU_ERR_WORKSPACE;
  SortWs<KeyT, P> w(ws, ws_bytes, nnz);
  const int threads = 256;
  coo_pack_keys_kernel<KeyT, P><<<blocks_for(nnz, threads), threads, 0, s>>>(
      idx, idx_ld, key_dims, key_dims > 1 ? dims[1] : 1, key_dims > 2 ? dims[2] : 1, nnz, w.kin, w.vin);
  count_launch();
  size_t cb = w.cub_bytes;
  cudaError_t e = cub_sort_pairs<KeyT, P>(w.cub, cb, w.kin, w.kout, w.vin, perm, nnz, key_bits, s);
  count_launch();
  if (e != cudaSuccess) return (int)e;
  if (sorted_idx) {
    coo_gather_sorted_kernel<P><<<blocks_for(nnz, threads), threads, 0, s>>>(idx, idx_ld, ndim, nnz, perm, sorted_idx);
    count_launch();
  }
  return launch_status();
}

// ------------------------------------------------------------------- sorted keys -> rowptr
// rowkey(k) is non-decreasing in k.  Thread k owns the rows in (rowkey(k-1), rowkey(k)] and writes
// rowptr[row] = k for them; the last thread also closes the tail.  O(rows + nnz), no atomics.
template <typename O, typename KeyFn>
__device__ __forceinline__ void fill_rowptr(int64_t k, int64_t nnz, int64_t total_rows, O* __restrict__ rowptr,
                                            KeyFn rowkey) {
  const int64_t cur = rowkey(k);
  const int64_t prev = (k == 0) ? -1 : rowkey(k - 1);
  for (int64_t r = prev + 1; r <= cur; ++r) rowptr[r] = (O)k;
  if (k == nnz - 1)
    for (int64_t r = cur + 1; r <= total_rows; ++r) rowptr[r] = (O)nnz;
}

template <typename O>
__global__ void fill_const_kernel(O* __restrict__ p, int64_t count, O v) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}

template <typename P, typename O>
__global__ void coo_to_csr_kernel(const int64_t* __restrict__ idx, int ndim, int64_t nnz, int64_t idx_ld,
                                  int64_t n, int64_t total_rows, const P* __restrict__ perm,
                                  O* __restrict__ rowptr, O* __restrict__ colind) {
  const int64_t* brow = (ndim == 3) ? idx : nullptr;
  const int64_t* rrow = idx + (int64_t)(ndim - 2) * idx_ld;
  const int64_t* crow = idx + (int64_t)(ndim - 1) * idx_ld;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += (int64_t)gridDim.x * blockDim.x) {
    auto rowkey = [&](int64_t kk) -> int64_t {
      const int64_t src = perm ? (int64_t)perm[kk] : kk;
      return (brow ? brow[src] * n : 0) + rrow[src];
    };
    const int64_t src = perm ? (int64_t)perm[k] : k;
    colind[k] = (O)crow[src];
    fill_rowptr<O>(k, nnz, total_rows, rowptr, rowkey);
  }
}

// ---------------------------------------------------------------- compress / decompress rows
template <typename I>
__global__ void row_hist_kernel(const I* __restrict__ rows, int64_t nnz, I* __restrict__ crow) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += (int64_t)gridDim.x * blockDim.x) {
    if constexpr (sizeof(I) == 4) atomicAdd(reinterpret_cast<int*>(crow) + 1 + rows[e], 1);
    else atomicAdd(reinterpret_cast<unsigned long long*>(crow) + 1 + rows[e], 1ull);
  }
}

template <typename I>
__global__ void decompress_kernel(const I* __restrict__ crow, int64_t n, int64_t nnz, I* __restrict__ rows) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += (int64_t)gridDim.x * blockDim.x)
    rows[e] = (I)row_of<I>(crow, n + 1, e);
}

// ------------------------------------------------------------------------- CSR transpose
template <typename I, typename KeyT, typename O>
__global__ void transpose_keys_kernel(const I* __restrict__ rowptr, const I* __restrict__ colind, int64_t batch,
                                      int64_t n, int64_t m, int64_t rowptr_bstride, int64_t nnz_bstride,
                                      int64_t nnz_total, KeyT* __restrict__ keys, O* __restrict__ iota,
                                      O* __restrict__ rowid) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz_total; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t item, row;
    if (nnz_bstride > 0) {  // torch batched CSR: equal nnz per item, per-item rowptr starting at 0
      item = e / nnz_bstride;
      row = row_of<I>(rowptr + item * rowptr_bstride, n + 1, e - item * nnz_bstride);
    } else {  // flat CSR over batch*n rows
      const int64_t gr = row_of<I>(rowptr, batch * n + 1, e);
      item = gr / n;
      row = gr - item * n;
    }
    keys[e] = (KeyT)((uint64_t)item * (uint64_t)m + (uint64_t)colind[e]);
    iota[e] = (O)e;
    rowid[e] = (O)row;
  }
}

template <typename KeyT, typename O>
__global__ void transpose_finish_kernel(const KeyT* __restrict__ keys_sorted, const O* __restrict__ permT,
                                        const O* __restrict__ rowid, int64_t nnz, int64_t total_rows,
                                        O* __restrict__ rowptrT, O* __restrict__ colindT) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += (int64_t)gridDim.x * blockDim.x) {
    colindT[k] = rowid[(int64_t)permT[k]];
    auto rowkey = [&](int64_t kk) -> int64_t { return (int64_t)keys_sorted[kk]; };
    fill_rowptr<O>(k, nnz, total_rows, rowptrT, rowkey);
  }
}

template <typename KeyT, typename O>
static size_t transpose_ws_bytes(int64_t nnz) {
  return sort_ws_bytes<KeyT, O>(nnz) + align_up((size_t)nnz * sizeof(O));
}

template <typename I, typename KeyT, typename O>
static int transpose_impl(const I* rowptr, const I* colind, int64_t batch, int64_t n, int64_t m,
                          int64_t rowptr_bstride, int64_t nnz_bstride, int64_t nnz, int key_bits, O* rowptrT,
                          O* colindT, O* permT, void* ws, size_t ws_bytes, cudaStream_t s) {
  if (ws_bytes < transpose_ws_bytes<KeyT, O>(nnz)) return TSGU_ERR_WORKSPACE;
  O* rowid = (O*)ws;
  char* rest = (char*)ws + align_up((size_t)nnz * sizeof(O));
  SortWs<KeyT, O> w(rest, ws_bytes - align_up((size_t)nnz * sizeof(O)), nnz);
  const int threads = 256;
  transpose_keys_kernel<I, KeyT, O><<<blocks_for(nnz, threads), threads, 0, s>>>(
      rowptr, colind, batch, n, m, rowptr_bstride, nnz_bstride, nnz, w.kin, w.vin, rowid);
  count_launch();
  size_t cb = w.cub_bytes;
  cudaError_t e = cub_sort_pairs<KeyT, O>(w.cub, cb, w.kin, w.kout, w.vin, permT, nnz, key_bits, s);
  count_launch();
  if (e != cudaSuccess) return (int)e;
  transpose_finish_kernel<KeyT, O><<<blocks_for(nnz, threads), threads, 0, s>>>(w.kout, permT, rowid, nnz, batch * m,
                                                                              rowptrT, colindT);
  count_launch();
  return launch_status();
}

// ----------------------------------------------------------------------- value shuffles
// out[k] = perm[k] >= 0 ? in[perm[k]] : 0.  Four entries per thread: the four gathers are independent,
// so each thread keeps four L2 requests in flight (the one-entry version was latency bound at 55 us for
// config 2's 9.2 M entries).
template <typename V, typename I>
__global__ void __launch_bounds__(256) gather_values_kernel(const V* __restrict__ in, const I* __restrict__ perm,
                                                            V* __restrict__ out, int64_t count) {
  const int64_t quads = count / 4;
  // the four permutation entries of a quad are one vector load and the four results one vector store when the arrays
  // are suitably aligned (they are: torch allocations): half the LSU instructions of the scalar version, which was
  // throttled by the LSU queues (ncu: mio_throttle 17.8, lg_throttle 6.6 stall cycles per issue)
  const bool vec_p = (reinterpret_cast<uintptr_t>(perm) % (4 * sizeof(I))) == 0;
  const bool vec_o = (reinterpret_cast<uintptr_t>(out) % (4 * sizeof(V))) == 0;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < quads; q += (int64_t)gridDim.x * blockDim.x) {
    int64_t src[4];
    if (vec_p) {
      if constexpr (sizeof(I) == 4) {
        const int4 p4 = __ldg(reinterpret_cast<const int4*>(perm) + q);
        src[0] = p4.x; src[1] = p4.y; src[2] = p4.z; src[3] = p4.w;
      } else {
        const longlong2 a = __ldg(reinterpret_cast<const longlong2*>(perm) + 2 * q);
        const longlong2 b = __ldg(reinterpret_cast<const longlong2*>(perm) + 2 * q + 1);
        src[0] = a.x; src[1] = a.y; src[2] = b.x; src[3] = b.y;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) src[i] = (int64_t)__ldg(perm + 4 * q + i);
    }
    V v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = src[i] >= 0 ? __ldg(in + src[i]) : VT<V>::from_acc(0);
    if (vec_o) {
      struct alignas(4 * sizeof(V)) Quad { V x[4]; };
      Quad o;
#pragma unroll
      for (int i = 0; i < 4; ++i) o.x[i] = v[i];
      reinterpret_cast<Quad*>(out)[q] = o;
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) out[4 * q + i] = v[i];
    }
  }
  if (blockIdx.x == 0 && threadIdx.x < (count & 3)) {  // tail
    const int64_t k = quads * 4 + threadIdx.x;
    const int64_t s1 = (int64_t)perm[k];
    out[k] = s1 >= 0 ? in[s1] : VT<V>::from_acc(0);
  }
}

// out[perm[k]] = in[k]: the adjoint of gather_values for an injective `perm` (out is zero-filled by the launcher).
template <typename V, typename I>
__global__ void __launch_bounds__(256) scatter_values_kernel(const V* __restrict__ in, const I* __restrict__ perm,
                                                             V* __restrict__ out, int64_t count) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += (int64_t)gridDim.x * blockDim.x) {
    const int64_t dst = (int64_t)__ldg(perm + k);
    if (dst >= 0) out[dst] = in[k];
  }
}

// Position-weighted checksum of an index array, accumulated into *out (integer atomics: order independent, so the
// value is deterministic).  The pattern cache uses it to notice index memory that was rewritten in place.
template <typename I>
__global__ void __launch_bounds__(256) fingerprint_kernel(const I* __restrict__ x, int64_t count,
                                                          unsigned long long* __restrict__ out) {
  unsigned long long acc = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x)
    acc += (unsigned long long)(long long)__ldg(x + i) * (unsigned long long)(i % 65521 + 1);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0 && acc != 0) atomicAdd(out, acc);
}

// Batched CSR (b, n+1) / (b, nnz) -> the block-diagonal CSR over b*n rows and b*m columns that the reference assembles
// item by item (utils/utils.py:604-645): crow_out[t*n + r] = crow[t, r] + t*nnz, col_out[t*nnz + e] = col[t, e] + t*m.
template <typename I>
__global__ void __launch_bounds__(256) block_diag_csr_kernel(const I* __restrict__ crow, const I* __restrict__ col,
                                                             int64_t batch, int64_t n, int64_t m, int64_t nnz,
                                                             I* __restrict__ crow_out, I* __restrict__ col_out) {
  const int64_t total = batch * n + 1 + batch * nnz;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    if (i <= batch * n) {
      if (i == batch * n) {
        crow_out[i] = (I)(batch * nnz);
      } else {
        const int64_t t = i / n, r = i - t * n;
        crow_out[i] = (I)((int64_t)crow[t * (n + 1) + r] + t * nnz);
      }
    } else {
      const int64_t e = i - (batch * n + 1);
      const int64_t t = e / nnz;
      col_out[e] = (I)((int64_t)col[e] + t * m);
    }
  }
}

template <typename V, typename I>
__global__ void segment_sum_kernel(const V* __restrict__ in, const I* __restrict__ perm, const I* __restrict__ seg,
                                   V* __restrict__ out, int64_t nseg) {
  using Acc = typename VT<V>::Acc;
  for (int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; u < nseg; u += (int64_t)gridDim.x * blockDim.x) {
    Acc a = Acc(0);
    for (int64_t k = (int64_t)seg[u]; k < (int64_t)seg[u + 1]; ++k)
      a += VT<V>::to_acc(in[perm ? (int64_t)perm[k] : k]);
    out[u] = VT<V>::from_acc(a);
  }
}

// strided -> strided dense copy (layout change).  A block owns PACK_R consecutive rows and walks the
// columns in chunks of 32 through a padded shared tile; the read phase runs threadIdx along whichever
// source dimension is contiguous, the write phase along whichever destination dimension is, so
// row-major <-> column-major (transposed-view) conversions are coalesced on both sides with
// PACK_R/8 independent loads per thread in flight.
constexpr int PACK_R = 128;
// Optional epilogue operands (tsgu_pack_dense_add): dst = src + add + rowvec[row], where `add` has the destination's
// element strides and `rowvec` is one value per (item, row).
template <typename V>
struct PackAdd {
  const V* add;     // nullable, addressed with the destination strides
  const V* rowvec;  // nullable
  int64_t v_bs, v_rs;
};

template <typename V, bool ADD = false>
__global__ void __launch_bounds__(256) pack_dense_kernel(const V* __restrict__ src, V* __restrict__ dst, int64_t rows,
                                                         int64_t cols, int64_t s_bs, int64_t s_rs, int64_t s_cs,
                                                         int64_t d_bs, int64_t d_rs, int64_t d_cs,
                                                         int64_t blocks_per_item, PackAdd<V> ep = PackAdd<V>{}) {
  using Acc = typename VT<V>::Acc;
  __shared__ V tile[PACK_R][33];
  const int64_t item = blockIdx.x / blocks_per_item;
  const int64_t r0 = (blockIdx.x - item * blocks_per_item) * PACK_R;
  const V* sp = src + item * s_bs;
  V* dp = dst + item * d_bs;
  auto put = [&](int r, int c, int64_t c0) {
    const int64_t off = (r0 + r) * d_rs + (c0 + c) * d_cs;
    if constexpr (ADD) {
      Acc x = VT<V>::to_acc(tile[r][c]);
      if (ep.add) x += VT<V>::to_acc(ep.add[item * d_bs + off]);
      if (ep.rowvec) x += VT<V>::to_acc(ep.rowvec[item * ep.v_bs + (r0 + r) * ep.v_rs]);
      dp[off] = VT<V>::from_acc(x);
    } else {
      dp[off] = tile[r][c];
    }
  };
  const bool src_row_fast = s_rs < s_cs;  // contiguous along rows (column-major view)
  const bool dst_row_fast = d_rs < d_cs;
  constexpr int NIT = PACK_R * 32 / 256;  // elements per thread and chunk (16)
  for (int64_t c0 = 0; c0 < cols; c0 += 32) {
    // all of a thread's loads are issued before the first shared-memory store (16 independent loads in flight)
    V tmp[NIT];
    if (src_row_fast) {
      const int r = threadIdx.x % PACK_R, cb = threadIdx.x / PACK_R;
#pragma unroll
      for (int i = 0; i < NIT; ++i) {
        const int c = cb + i * (256 / PACK_R);
        tmp[i] = (r0 + r < rows && c0 + c < cols) ? __ldg(sp + (r0 + r) * s_rs + (c0 + c) * s_cs) : VT<V>::from_acc(0);
      }
#pragma unroll
      for (int i = 0; i < NIT; ++i) tile[r][cb + i * (256 / PACK_R)] = tmp[i];
    } else {
      const int c = threadIdx.x % 32, rb = threadIdx.x / 32;
#pragma unroll
      for (int i = 0; i < NIT; ++i) {
        const int r = rb + i * 8;
        tmp[i] = (r0 + r < rows && c0 + c < cols) ? __ldg(sp + (r0 + r) * s_rs + (c0 + c) * s_cs) : VT<V>::from_acc(0);
      }
#pragma unroll
      for (int i = 0; i < NIT; ++i) tile[rb + i * 8][c] = tmp[i];
    }
    __syncthreads();
    if (dst_row_fast) {
      const int r = threadIdx.x % PACK_R;
      for (int c = threadIdx.x / PACK_R; c < 32; c += 256 / PACK_R)
        if (r0 + r < rows && c0 + c < cols) put(r, c, c0);
    } else {
      const int c = threadIdx.x % 32;
      for (int r = threadIdx.x / 32; r < PACK_R; r += 8)
        if (r0 + r < rows && c0 + c < cols) put(r, c, c0);
    }
    __syncthreads();
  }
}

}  // namespace tsgu

using namespace tsgu;

extern "C" size_t tsgu_coo_sort_workspace_bytes(int ndim, int64_t nnz, int perm_dtype) {
  (void)ndim;
  if (nnz <= 0) return 0;
  // sized for the widest key (64-bit); narrower keys need less
  return perm_dtype == TSGU_I32 ? sort_ws_bytes<uint64_t, int32_t>(nnz) : sort_ws_bytes<uint64_t, int64_t>(nnz);
}

extern "C" int tsgu_coo_sort(const int64_t* idx, int ndim, int64_t nnz, int64_t idx_ld, const int64_t* dims,
                             int key_dims, int64_t* sorted_idx, void* perm, int perm_dtype, void* workspace,
                             size_t workspace_bytes, void* stream) {
  if (ndim < 2 || ndim > 3 || key_dims < 1 || key_dims > ndim || nnz < 0) return TSGU_ERR_SHAPE;
  if (perm_dtype != TSGU_I32 && perm_dtype != TSGU_I64) return TSGU_ERR_DTYPE;
  if (nnz == 0) return 0;
  if (perm_dtype == TSGU_I32 && nnz > 0x7fffffffLL) return TSGU_ERR_RANGE;
  if (!workspace) return TSGU_ERR_WORKSPACE;
  unsigned __int128 span = 1;
  for (int d = 0; d < key_dims; ++d) {
    if (dims[d] <= 0) return TSGU_ERR_SHAPE;
    span *= (unsigned __int128)dims[d];
    if (span >> 63) return TSGU_ERR_RANGE;
  }
  const int key_bits = bits_for((uint64_t)span);
  cudaStream_t s = as_stream(stream);
  if (key_bits <= 32) {
    if (perm_dtype == TSGU_I32)
      return coo_sort_impl<uint32_t, int32_t>(idx, ndim, nnz, idx_ld, dims, key_dims, key_bits, sorted_idx, (int32_t*)perm, workspace, workspace_bytes, s);
    return coo_sort_impl<uint32_t, int64_t>(idx, ndim, nnz, idx_ld, dims, key_dims, key_bits, sorted_idx, (int64_t*)perm, workspace, workspace_bytes, s);
  }
  if (perm_dtype == TSGU_I32)
    return coo_sort_impl<uint64_t, int32_t>(idx, ndim, nnz, idx_ld, dims, key_dims, key_bits, sorted_idx, (int32_t*)perm, workspace, workspace_bytes, s);
  return coo_sort_impl<uint64_t, int64_t>(idx, ndim, nnz, idx_ld, dims, key_dims, key_bits, sorted_idx, (int64_t*)perm, workspace, workspace_bytes, s);
}

extern "C" int tsgu_coo_to_csr(const int64_t* idx, int ndim, int64_t nnz, int64_t idx_ld, int64_t batch, int64_t n,
                               const void* perm, void* rowptr_out, void* colind_out, int out_idx_dtype,
                               void* stream) {
  if (ndim < 2 || ndim > 3 || nnz < 0 || batch < 1 || n < 0) return TSGU_ERR_SHAPE;
  if (out_idx_dtype != TSGU_I32 && out_idx_dtype != TSGU_I64) return TSGU_ERR_DTYPE;
  if (out_idx_dtype == TSGU_I32 && (nnz > 0x7fffffffLL || batch * n >= 0x7fffffffLL)) return TSGU_ERR_RANGE;
  cudaStream_t s = as_stream(stream);
  const int64_t total_rows = batch * n;
  const int threads = 256;
  if (out_idx_dtype == TSGU_I32) {
    using O = int32_t;
    if (nnz == 0) fill_const_kernel<O><<<blocks_for(total_rows + 1, threads), threads, 0, s>>>((O*)rowptr_out, total_rows + 1, 0);
    else coo_to_csr_kernel<O, O><<<blocks_for(nnz, threads), threads, 0, s>>>(idx, ndim, nnz, idx_ld, n, total_rows, (const O*)perm, (O*)rowptr_out, (O*)colind_out);
  } else {
    using O = int64_t;
    if (nnz == 0) fill_const_kernel<O><<<blocks_for(total_rows + 1, threads), threads, 0, s>>>((O*)rowptr_out, total_rows + 1, 0);
    else coo_to_csr_kernel<O, O><<<blocks_for(nnz, threads), threads, 0, s>>>(idx, ndim, nnz, idx_ld, n, total_rows, (const O*)perm, (O*)rowptr_out, (O*)colind_out);
  }
  count_launch();
  return launch_status();
}

extern "C" size_t tsgu_compress_rows_workspace_bytes(int64_t n, int idx_dtype) {
  size_t b = 0;
  cudaError_t e;
  if (idx_dtype == TSGU_I32) e = cub::DeviceScan::InclusiveSum(nullptr, b, (int32_t*)nullptr, (int32_t*)nullptr, n + 1);
  else e = cub::DeviceScan::InclusiveSum(nullptr, b, (int64_t*)nullptr, (int64_t*)nullptr, n + 1);
  if (e != cudaSuccess) { (void)cudaGetLastError(); b = (size_t)(n + 1) * 8 + (1u << 16); }
  return align_up(b);
}

extern "C" int tsgu_compress_rows(const void* rows, int64_t nnz, int64_t n, void* crow_out, int idx_dtype,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  if (nnz < 0 || n < 0) return TSGU_ERR_SHAPE;
  cudaStream_t s = as_stream(stream);
  const int threads = 256;
  TSGU_DISPATCH_IDX(idx_dtype, {
    fill_const_kernel<I><<<blocks_for(n + 1, threads), threads, 0, s>>>((I*)crow_out, n + 1, (I)0);
    count_launch();
    if (nnz > 0) {
      row_hist_kernel<I><<<blocks_for(nnz, threads), threads, 0, s>>>((const I*)rows, nnz, (I*)crow_out);
      count_launch();
    }
    size_t b = workspace_bytes;
    if (!workspace) return TSGU_ERR_WORKSPACE;
    cudaError_t e = cub::DeviceScan::InclusiveSum(workspace, b, (I*)crow_out, (I*)crow_out, n + 1, s);
    count_launch();
    if (e != cudaSuccess) return (int)e;
  });
  return launch_status();
}

extern "C" int tsgu_decompress_crow(const void* crow, int64_t n, int64_t nnz, void* rows_out, int idx_dtype,
                                    void* stream) {
  if (nnz < 0 || n < 0) return TSGU_ERR_SHAPE;
  if (nnz == 0) return 0;
  cudaStream_t s = as_stream(stream);
  TSGU_DISPATCH_IDX(idx_dtype, {
    decompress_kernel<I><<<blocks_for(nnz, 256), 256, 0, s>>>((const I*)crow, n, nnz, (I*)rows_out);
    count_launch();
  });
  return launch_status();
}

extern "C" size_t tsgu_csr_transpose_workspace_bytes(int64_t batch, int64_t m, int64_t nnz_total, int out_idx_dtype) {
  (void)batch; (void)m;
  if (nnz_total <= 0) return 0;
  return out_idx_dtype == TSGU_I32 ? transpose_ws_bytes<uint64_t, int32_t>(nnz_total)
                                   : transpose_ws_bytes<uint64_t, int64_t>(nnz_total);
}

extern "C" int tsgu_csr_transpose(const void* rowptr, const void* colind, int64_t batch, int64_t n, int64_t m,
                                  int64_t rowptr_bstride, int64_t nnz_bstride, int64_t nnz_total, int idx_dtype,
                                  void* rowptrT, void* colindT, void* permT, int out_idx_dtype, void* workspace,
                                  size_t workspace_bytes, void* stream) {
  if (batch < 1 || n < 0 || m < 0 || nnz_total < 0) return TSGU_ERR_SHAPE;
  if (out_idx_dtype != TSGU_I32 && out_idx_dtype != TSGU_I64) return TSGU_ERR_DTYPE;
  if (out_idx_dtype == TSGU_I32 && (nnz_total > 0x7fffffffLL || batch * m >= 0x7fffffffLL || n > 0x7fffffffLL)) return TSGU_ERR_RANGE;
  cudaStream_t s = as_stream(stream);
  const int64_t total_rows = batch * m;
  if (nnz_total == 0) {
    if (out_idx_dtype == TSGU_I32) fill_const_kernel<int32_t><<<blocks_for(total_rows + 1, 256), 256, 0, s>>>((int32_t*)rowptrT, total_rows + 1, 0);
    else fill_const_kernel<int64_t><<<blocks_for(total_rows + 1, 256), 256, 0, s>>>((int64_t*)rowptrT, total_rows + 1, 0);
    count_launch();
    return launch_status();
  }
  if (!workspace) return TSGU_ERR_WORKSPACE;
  const int key_bits = bits_for((uint64_t)total_rows);
  TSGU_DISPATCH_IDX(idx_dtype, {
    if (out_idx_dtype == TSGU_I32) {
      using O = int32_t;
      if (key_bits <= 32) return transpose_impl<I, uint32_t, O>((const I*)rowptr, (const I*)colind, batch, n, m, rowptr_bstride, nnz_bstride, nnz_total, key_bits, (O*)rowptrT, (O*)colindT, (O*)permT, workspace, workspace_bytes, s);
      return transpose_impl<I, uint64_t, O>((const I*)rowptr, (const I*)colind, batch, n, m, rowptr_bstride, nnz_bstride, nnz_total, key_bits, (O*)rowptrT, (O*)colindT, (O*)permT, workspace, workspace_bytes, s);
    } else {
      using O = int64_t;
      if (key_bits <= 32) return transpose_impl<I, uint32_t, O>((const I*)rowptr, (const I*)colind, batch, n, m, rowptr_bstride, nnz_bstride, nnz_total, key_bits, (O*)rowptrT, (O*)colindT, (O*)permT, workspace, workspace_bytes, s);
      return transpose_impl<I, uint64_t, O>((const I*)rowptr, (const I*)colind, batch, n, m, rowptr_bstride, nnz_bstride, nnz_total, key_bits, (O*)rowptrT, (O*)colindT, (O*)permT, workspace, workspace_bytes, s);
    }
  });
  return 0;
}

extern "C" int tsgu_gather_values(const void* in, const void* perm, void* out, int64_t count, int val_dtype,
                                  int idx_dtype, void* stream) {
  if (count < 0) return TSGU_ERR_SHAPE;
  if (count == 0) return 0;
  cudaStream_t s = as_stream(stream);
  TSGU_DISPATCH_VAL(val_dtype, TSGU_DISPATCH_IDX(idx_dtype, {
    gather_values_kernel<V, I><<<blocks_for((count + 3) / 4, 256), 256, 0, s>>>((const V*)in, (const I*)perm, (V*)out, count);
    count_launch();
  }));
  return launch_status();
}

extern "C" int tsgu_scatter_values(const void* in, const void* perm, void* out, int64_t count, int64_t out_count,
                                   int val_dtype, int idx_dtype, void* stream) {
  if (count < 0 || out_count < 0) return TSGU_ERR_SHAPE;
  cudaStream_t s = as_stream(stream);
  TSGU_DISPATCH_VAL(val_dtype, TSGU_DISPATCH_IDX(idx_dtype, {
    if (out_count > 0) {
      cudaError_t e = cudaMemsetAsync(out, 0, (size_t)out_count * sizeof(V), s);
      if (e != cudaSuccess) return (int)e;
    }
    if (count > 0) {
      scatter_values_kernel<V, I><<<blocks_for(count, 256), 256, 0, s>>>((const V*)in, (const I*)perm, (V*)out, count);
      count_launch();
    }
  }));
  return launch_status();
}

extern "C" int tsgu_block_diag_csr(const void* crow, const void* col, int64_t batch, int64_t n, int64_t m, int64_t nnz,
                                   void* crow_out, void* col_out, int idx_dtype, void* stream) {
  if (batch < 1 || n < 0 || m < 0 || nnz < 0) return TSGU_ERR_SHAPE;
  if (idx_dtype == TSGU_I32 && (batch * nnz > 0x7fffffffLL || batch * m > 0x7fffffffLL)) return TSGU_ERR_RANGE;
  cudaStream_t s = as_stream(stream);
  TSGU_DISPATCH_IDX(idx_dtype, {
    block_diag_csr_kernel<I><<<blocks_for(batch * n + 1 + batch * nnz, 256), 256, 0, s>>>(
        (const I*)crow, (const I*)col, batch, n, m, nnz, (I*)crow_out, (I*)col_out);
    count_launch();
  });
  return launch_status();
}

extern "C" int tsgu_fingerprint(const void* data, int64_t count, int idx_dtype, void* out, void* stream) {
  if (count < 0 || !out) return TSGU_ERR_SHAPE;
  if (count == 0) return 0;
  cudaStream_t s = as_stream(stream);
  const unsigned blocks = min(blocks_for(count, 256 * 8), 148u * 8u);
  TSGU_DISPATCH_IDX(idx_dtype, {
    fingerprint_kernel<I><<<blocks, 256, 0, s>>>((const I*)data, count, (unsigned long long*)out);
    count_launch();
  });
  return launch_status();
}

extern "C" int tsgu_segment_sum_values(const void* in, const void* perm, const void* seg, void* out, int64_t nseg,
                                       int val_dtype, int idx_dtype, void* stream) {
  if (nseg < 0) return TSGU_ERR_SHAPE;
  if (nseg == 0) return 0;
  cudaStream_t s = as_stream(stream);
  TSGU_DISPATCH_VAL(val_dtype, TSGU_DISPATCH_IDX(idx_dtype, {
    segment_sum_kernel<V, I><<<blocks_for(nseg, 256), 256, 0, s>>>((const V*)in, (const I*)perm, (const I*)seg, (V*)out, nseg);
    count_launch();
  }));
  return launch_status();
}

extern "C" int tsgu_pack_dense(const void* src, void* dst, int64_t batch, int64_t rows, int64_t cols, int64_t s_bs,
                               int64_t s_rs, int64_t s_cs, int64_t d_bs, int64_t d_rs, int64_t d_cs, int val_dtype,
                               void* stream) {
  if (batch < 0 || rows < 0 || cols < 0) return TSGU_ERR_SHAPE;
  if (batch == 0 || rows == 0 || cols == 0) return 0;
  cudaStream_t s = as_stream(stream);
  const int64_t bpi = (rows + PACK_R - 1) / PACK_R;
  const int64_t blocks = batch * bpi;
  if (blocks > 0x7fffffffLL) return TSGU_ERR_RANGE;
  TSGU_DISPATCH_VAL(val_dtype, {
    pack_dense_kernel<V><<<(unsigned)blocks, 256, 0, s>>>((const V*)src, (V*)dst, rows, cols, s_bs, s_rs, s_cs, d_bs, d_rs, d_cs, bpi);
    count_launch();
  });
  return launch_status();
}

extern "C" int tsgu_pack_dense_add(const void* src, const void* add, const void* rowvec, void* dst, int64_t batch,
                                   int64_t rows, int64_t cols, int64_t s_bs, int64_t s_rs, int64_t s_cs, int64_t d_bs,
                                   int64_t d_rs, int64_t d_cs, int64_t v_bs, int64_t v_rs, int val_dtype, void* stream) {
  if (batch < 0 || rows < 0 || cols < 0) return TSGU_ERR_SHAPE;
  if (batch == 0 || rows == 0 || cols == 0) return 0;
  cudaStream_t s = as_stream(stream);
  const int64_t bpi = (rows + PACK_R - 1) / PACK_R;
  const int64_t blocks = batch * bpi;
  if (blocks > 0x7fffffffLL) return TSGU_ERR_RANGE;
  TSGU_DISPATCH_VAL(val_dtype, {
    PackAdd<V> ep{(const V*)add, (const V*)rowvec, v_bs, v_rs};
    pack_dense_kernel<V, true><<<(unsigned)blocks, 256, 0, s>>>((const V*)src, (V*)dst, rows, cols, s_bs, s_rs, s_cs, d_bs,
                                                                 d_rs, d_cs, bpi, ep);
    count_launch();
  });
  return launch_status();
}
