// merge.cu -- nnz-balanced (merge-path) SpMM and SDDMM for sm_100a, for matrices whose row lengths
// are badly skewed (power-law graphs: BASELINE config 4) or that have long runs of empty rows.
//
// The (row-end, nonzero) merge path of the CSR matrix (Merrill & Garland's decomposition) is cut
// into tiles of MERGE_P path items, so every CTA gets the same amount of "rows finished + nonzeros
// consumed" work no matter how the nonzeros are distributed.  A tile's slices of rowptr / colind /
// vals are contiguous, so they are streamed into shared memory with the bulk-copy engine one tile
// ahead (same pipeline as tile.cuh); inside the CTA the tile's path is split again, evenly, over
// the lane groups.  Rows cut by a group or tile boundary are completed in a fixed order (group
// partials in shared memory, tile partials in a workspace + a small fix-up kernel): no float
// atomics, bit-reproducible results.
#include <climits>

#include "common.cuh"
#include "tile.cuh"

#ifndef TSGU_MERGE_P
#define TSGU_MERGE_P 3072  // path items per tile (swept on config 4 with 2 CTAs/SM: 1024 2.59, 2048 2.20, 3072 2.10, 4096 2.96 ms per SpMM)
#endif
#ifndef TSGU_MERGE_MINB
#define TSGU_MERGE_MINB 2   // resident CTAs per SM the register allocation aims for (swept on config 4: 2 CTAs x 16 loads beat 3 x 8)
#endif
#ifndef TSGU_MERGE_SDDMM_MINB
#define TSGU_MERGE_SDDMM_MINB 3
#endif
#ifndef TSGU_MERGE_LOADS
#define TSGU_MERGE_LOADS 16  // 128-bit dense-row loads in flight per lane (SpMM)
#endif
#ifndef TSGU_MERGE_SDDMM_LOADS
#define TSGU_MERGE_SDDMM_LOADS 8  // ... and in the SDDMM, which wants more warps instead (row changes stall on a G-row fetch)
#endif

namespace tsgu {

constexpr int MERGE_P = TSGU_MERGE_P;

// ------------------------------------------------------------------------------------ partition
// Merge-path split at diagonal d: i = row-ends consumed, j = d - i nonzeros consumed.
template <typename I>
__device__ __forceinline__ void merge_search(const I* __restrict__ rowptr, int64_t rows, int64_t nnz, int64_t d,
                                             int64_t& i, int64_t& j) {
  int64_t lo = d > nnz ? d - nnz : 0;
  int64_t hi = d < rows ? d : rows;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if ((int64_t)__ldg(rowptr + mid + 1) <= d - mid - 1) lo = mid + 1; else hi = mid;
  }
  i = lo;
  j = d - lo;
}

template <typename I>
__global__ void merge_partition_kernel(const I* __restrict__ rowptr, int64_t rows, int64_t nnz, int64_t num_tiles,
                                       int64_t* __restrict__ part) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t > num_tiles) return;
  int64_t d = t * MERGE_P;
  if (d > rows + nnz) d = rows + nnz;
  int64_t i, j;
  merge_search<I>(rowptr, rows, nnz, d, i, j);
  part[2 * t] = i;
  part[2 * t + 1] = j;
}

// same search on the tile's rowptr slice in shared memory (second-level split over lane groups);
// rp[k] = rowptr[i0 + k]; returns absolute (i, j)
template <typename I>
__device__ __forceinline__ void merge_search_smem(const I* rp, int64_t i0, int64_t j0, int rows_t, int nnz_t, int d,
                                                  int64_t& i, int64_t& j) {
  int lo = d > nnz_t ? d - nnz_t : 0;
  int hi = d < rows_t ? d : rows_t;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if ((int64_t)rp[mid + 1] - j0 <= (int64_t)(d - mid - 1)) lo = mid + 1; else hi = mid;
  }
  i = i0 + lo;
  j = j0 + (d - lo);
}

// ------------------------------------------------------------------------------------ shared memory
template <typename V, typename I, int VALS>
struct MergeStage {
  static constexpr int AI = 16 / (int)sizeof(I), AV = 16 / (int)sizeof(V);
  alignas(16) I rp[MERGE_P + 2 + 2 * AI];
  alignas(16) I col[MERGE_P + 2 * AI];
  alignas(16) V val[VALS == 1 ? MERGE_P + 2 * AV : AV];
  alignas(16) I prm[VALS == 2 ? MERGE_P + 2 * AI : AI];
};

template <typename V, typename I, int VALS>
struct MergeProducer {
  using Stage = MergeStage<V, I, VALS>;
  const I* rowptr; const I* colind; const V* vals; const I* perm;
  int64_t rowptr_len, nnz_len;
  __device__ __forceinline__ void issue(Stage& st, uint64_t* bar, int64_t i0, int64_t j0, int64_t i1, int64_t j1) const {
    using TP = TileProducer<V, I, 0>;
    uint32_t tx = TP::template span<I>(st.rp, rowptr, i0, i1 + 2 < rowptr_len ? i1 + 2 : rowptr_len, rowptr_len, bar);
    if (j1 > j0) {
      tx += TP::template span<I>(st.col, colind, j0, j1, nnz_len, bar);
      if constexpr (VALS == 1) tx += TP::template span<V>(st.val, vals, j0, j1, nnz_len, bar);
      if constexpr (VALS == 2) tx += TP::template span<I>(st.prm, perm, j0, j1, nnz_len, bar);
    }
    mbar_expect_tx(bar, tx);
  }
};

template <typename V, typename I, int VALS, int LPR, int VPL>
struct MergeSpmmSmem {
  using Acc = typename VT<V>::Acc;
  static constexpr int GROUPS = 256 / LPR;
  static constexpr int KSLOT = LPR * VPL * (16 / (int)sizeof(V));  // accumulators per partial vector (>= K)
  MergeStage<V, I, VALS> st[2];
  alignas(16) Acc head[GROUPS][KSLOT];
  alignas(16) Acc tail[GROUPS][KSLOT];
  int64_t head_row[GROUPS];
  int64_t tail_row[GROUPS];
  alignas(8) uint64_t full[2];
};

template <typename V, typename I>
struct MergeSpmmParams {
  const I* rowptr; const I* colind; const V* vals; const I* perm; const V* B; V* C;
  int64_t rows, K, nnz, b_rs, ldc;
  const int64_t* part;      // (num_tiles + 1) x (i, j)
  typename VT<V>::Acc* carry;  // num_tiles x 2 x Kpad : [tile][0] = head partial, [tile][1] = tail partial
  int64_t* carry_row;       // num_tiles x 2 : row of the head / tail partial, -1 if none
  int64_t kpad;             // K rounded up to the lane tiling
};

// =========================================================================================== SpMM
template <typename V, typename I, int LPR, int VPL, int U, bool EXACT, bool PERM>
__global__ void __launch_bounds__(256, TSGU_MERGE_MINB) spmm_merge_kernel(const MergeSpmmParams<V, I> p, const int64_t num_tiles) {
  using Acc = typename VT<V>::Acc;
  using Stage = MergeStage<V, I, PERM ? 2 : 1>;
  constexpr int EPV = 16 / sizeof(V);
  constexpr int AI = Stage::AI, AV = Stage::AV;
  using Smem = MergeSpmmSmem<V, I, PERM ? 2 : 1, LPR, VPL>;
  constexpr int GROUPS = Smem::GROUPS;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);

  const int tid = threadIdx.x, lane = tid & 31, gl = lane % LPR, group = tid / LPR;
  const unsigned gmask = group_mask<LPR>(lane);
  const int kv = (int)(p.K / EPV);
  const uint32_t row_bytes = (uint32_t)(p.b_rs * sizeof(V));
  bool on[VPL];
#pragma unroll
  for (int w = 0; w < VPL; ++w) on[w] = EXACT || (w * LPR + gl < kv);

  if (tid == 0) {
    mbar_init(&sm.full[0], 1);
    mbar_init(&sm.full[1], 1);
    mbar_fence_init();
  }
  __syncthreads();

  MergeProducer<V, I, PERM ? 2 : 1> prod{p.rowptr, p.colind, p.vals, p.perm, p.rows + 1, p.nnz};
  const int64_t t0 = blockIdx.x;
  int64_t n_i0 = 0, n_j0 = 0, n_i1 = 0, n_j1 = 0;  // thread 0: coordinates of the tile to issue next
  if (tid == 0 && t0 < num_tiles) {
    prod.issue(sm.st[0], &sm.full[0], p.part[2 * t0], p.part[2 * t0 + 1], p.part[2 * t0 + 2], p.part[2 * t0 + 3]);
    const int64_t tn = t0 + gridDim.x;
    if (tn < num_tiles) { n_i0 = p.part[2 * tn]; n_j0 = p.part[2 * tn + 1]; n_i1 = p.part[2 * tn + 2]; n_j1 = p.part[2 * tn + 3]; }
  }

  const char* Bb = reinterpret_cast<const char*>(p.B) + (size_t)gl * 16;
  int it = 0;
  for (int64_t t = t0; t < num_tiles; t += gridDim.x, ++it) {
    const int stage = it & 1;
    if (tid == 0) {
      const int64_t tn = t + gridDim.x;
      if (tn < num_tiles) {
        prod.issue(sm.st[stage ^ 1], &sm.full[stage ^ 1], n_i0, n_j0, n_i1, n_j1);
        const int64_t tnn = tn + gridDim.x;
        if (tnn < num_tiles) { n_i0 = p.part[2 * tnn]; n_j0 = p.part[2 * tnn + 1]; n_i1 = p.part[2 * tnn + 2]; n_j1 = p.part[2 * tnn + 3]; }
      }
    }
    // tile coordinates (L2-resident, read by everyone; tiny)
    const int64_t ti0 = __ldg(p.part + 2 * t), tj0 = __ldg(p.part + 2 * t + 1);
    const int64_t ti1 = __ldg(p.part + 2 * t + 2), tj1 = __ldg(p.part + 2 * t + 3);
    mbar_wait(&sm.full[stage], (uint32_t)((it >> 1) & 1));

    const Stage& st = sm.st[stage];
    const I* rp = st.rp + (int)(ti0 & (AI - 1));    // rp[k] = rowptr[ti0 + k]
    const I* scol = st.col + (int)(tj0 & (AI - 1));  // scol[k] = colind[tj0 + k]
    const V* sval = st.val + (int)(tj0 & (AV - 1));
    const I* sprm = st.prm + (int)(tj0 & (AI - 1));
    const int rows_t = (int)(ti1 - ti0), nnz_t = (int)(tj1 - tj0);
    const int path_t = rows_t + nnz_t;

    // second-level split: this group's piece of the tile's path
    const int per = (path_t + GROUPS - 1) / GROUPS;
    int d0 = group * per, d1 = d0 + per;
    if (d0 > path_t) d0 = path_t;
    if (d1 > path_t) d1 = path_t;
    int64_t gi0, gj0, gi1, gj1;
    merge_search_smem<I>(rp, ti0, tj0, rows_t, nnz_t, d0, gi0, gj0);
    merge_search_smem<I>(rp, ti0, tj0, rows_t, nnz_t, d1, gi1, gj1);

    Acc acc[VPL][EPV];
#pragma unroll
    for (int w = 0; w < VPL; ++w)
#pragma unroll
      for (int i = 0; i < EPV; ++i) acc[w][i] = Acc(0);

    // Tile-local 32-bit coordinates from here on (a tile holds at most MERGE_P entries and row ends):
    // entries [gj0l, gj1l) and row ends [rowl, gi1l) belong to this group.  `row_end` is the local end of
    // the current row, INT_MAX once the row does not finish inside this group's range.
    const int gj0l = (int)(gj0 - tj0), gj1l = (int)(gj1 - tj0);
    const int gi0l = (int)(gi0 - ti0), gi1l = (int)(gi1 - ti0);
    int rowl = gi0l;
    int row_end = rowl < gi1l ? (int)((int64_t)rp[rowl + 1] - tj0) : INT_MAX;
    bool head = gi0 < p.rows && (int64_t)rp[gi0l] < gj0;  // the first row began before this group's range
    if (gl == 0) sm.head_row[group] = -1;
    if (tid == 0) p.carry_row[t * 2 + 0] = -1;  // overwritten after the barrier if this tile has a head partial

    // finish the current row: interior rows go straight to C, a head row that began before this group's
    // range is parked in shared memory for the ordered combine below
    auto flush = [&]() {
      if (head) {
#pragma unroll
        for (int w = 0; w < VPL; ++w)
#pragma unroll
          for (int i = 0; i < EPV; ++i) sm.head[group][(w * LPR + gl) * EPV + i] = acc[w][i];
        if (gl == 0) sm.head_row[group] = gi0;
        head = false;
      } else {
        V* Crow = p.C + (ti0 + rowl) * p.ldc;
#pragma unroll
        for (int w = 0; w < VPL; ++w)
          if (EXACT || on[w]) store_vec<V, EPV>(Crow + (int64_t)(w * LPR + gl) * EPV, acc[w]);
      }
#pragma unroll
      for (int w = 0; w < VPL; ++w)
#pragma unroll
        for (int i = 0; i < EPV; ++i) acc[w][i] = Acc(0);
      ++rowl;
      row_end = rowl < gi1l ? (int)((int64_t)rp[rowl + 1] - tj0) : INT_MAX;
    };
    auto accumulate = [&](const uint4 (&bu)[VPL], const Acc vj) {
#pragma unroll
      for (int w = 0; w < VPL; ++w) {
        Acc x[EPV];
        Raw<V, EPV> raw;
        raw.bits = bu[w];
        raw_unpack<V, EPV>(raw, x);
#pragma unroll
        for (int i = 0; i < EPV; ++i) acc[w][i] = fma(vj, x[i], acc[w][i]);
      }
    };

    for (int basel = gj0l; basel < gj1l; basel += LPR) {
      const int el = basel + gl;
      uint32_t cu = 0;
      Acc v = Acc(0);
      if (el < gj1l) {
        cu = (uint32_t)scol[el];
        if constexpr (PERM) v = load_scalar<V>(p.vals + (int64_t)sprm[el]);
        else v = VT<V>::to_acc(sval[el]);
      }
      const int cnt = min(LPR, gj1l - basel);
      for (int j = 0; j < cnt; j += U) {
        // all broadcasts of the batch first (one convergence check for the lot), then U dense-row gathers in
        // flight (they do not depend on the row structure), then the segmented accumulation walks the rows
        uint32_t cj[U];
        Acc vj[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          cj[u] = shfl_idx(gmask, cu, j + u, LPR);
          vj[u] = shfl_idx(gmask, v, j + u, LPR);
        }
        uint4 b[U][VPL];
        if (j + U <= cnt) {  // full batch (group-uniform branch): nothing is predicated
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const char* brow = Bb + (uint64_t)cj[u] * row_bytes;
#pragma unroll
            for (int w = 0; w < VPL; ++w) {
              if (EXACT || on[w]) b[u][w] = __ldg(reinterpret_cast<const uint4*>(brow + w * (LPR * 16)));
              else b[u][w] = make_uint4(0, 0, 0, 0);
            }
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int eu = basel + j + u;
            while (eu >= row_end) flush();  // also steps over empty rows
            accumulate(b[u], vj[u]);
          }
        } else {  // ragged end of this group's range
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const char* brow = Bb + (uint64_t)cj[u] * row_bytes;
#pragma unroll
            for (int w = 0; w < VPL; ++w) {
              b[u][w] = make_uint4(0, 0, 0, 0);
              if (j + u < cnt && (EXACT || on[w])) b[u][w] = __ldg(reinterpret_cast<const uint4*>(brow + w * (LPR * 16)));
            }
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {
            if (j + u < cnt) {
              const int eu = basel + j + u;
              while (eu >= row_end) flush();
              accumulate(b[u], vj[u]);
            }
          }
        }
      }
    }
    while (rowl < gi1l) flush();  // rows whose end lies in this group's range but have no entry left
    // what is left belongs to row gi1, which finishes in a later group / tile
#pragma unroll
    for (int w = 0; w < VPL; ++w)
#pragma unroll
      for (int i = 0; i < EPV; ++i) sm.tail[group][(w * LPR + gl) * EPV + i] = acc[w][i];
    if (gl == 0) sm.tail_row[group] = gi1;
    __syncthreads();

    // ---- ordered combine of rows cut by group boundaries --------------------------------
    {
      const int64_t hr = sm.head_row[group];
      if (hr >= 0) {
        int glo = group;
        while (glo > 0 && sm.tail_row[glo - 1] == hr) --glo;
        Acc tot[VPL][EPV];
#pragma unroll
        for (int w = 0; w < VPL; ++w)
#pragma unroll
          for (int i = 0; i < EPV; ++i) tot[w][i] = Acc(0);
        for (int g2 = glo; g2 < group; ++g2)
#pragma unroll
          for (int w = 0; w < VPL; ++w)
#pragma unroll
            for (int i = 0; i < EPV; ++i) tot[w][i] += sm.tail[g2][(w * LPR + gl) * EPV + i];
#pragma unroll
        for (int w = 0; w < VPL; ++w)
#pragma unroll
          for (int i = 0; i < EPV; ++i) tot[w][i] += sm.head[group][(w * LPR + gl) * EPV + i];
        const bool from_earlier_tile = (glo == 0) && ((int64_t)rp[(int)(hr - ti0)] < tj0);
        if (from_earlier_tile) {  // completed by the fix-up kernel together with earlier tiles' tails
          Acc* dst = p.carry + (t * 2 + 0) * p.kpad;
#pragma unroll
          for (int w = 0; w < VPL; ++w)
#pragma unroll
            for (int i = 0; i < EPV; ++i) dst[(w * LPR + gl) * EPV + i] = tot[w][i];
          if (gl == 0) p.carry_row[t * 2 + 0] = hr;
        } else {
          V* Crow = p.C + hr * p.ldc;
#pragma unroll
          for (int w = 0; w < VPL; ++w)
            if (EXACT || on[w]) store_vec<V, EPV>(Crow + (int64_t)(w * LPR + gl) * EPV, tot[w]);
        }
      }
      if (group == GROUPS - 1) {  // the tile's tail: everything accumulated for row ti1
        int glo = GROUPS - 1;
        while (glo > 0 && sm.tail_row[glo - 1] == ti1) --glo;
        Acc tot[VPL][EPV];
#pragma unroll
        for (int w = 0; w < VPL; ++w)
#pragma unroll
          for (int i = 0; i < EPV; ++i) tot[w][i] = Acc(0);
        for (int g2 = glo; g2 < GROUPS; ++g2)
#pragma unroll
          for (int w = 0; w < VPL; ++w)
#pragma unroll
            for (int i = 0; i < EPV; ++i) tot[w][i] += sm.tail[g2][(w * LPR + gl) * EPV + i];
        Acc* dst = p.carry + (t * 2 + 1) * p.kpad;
#pragma unroll
        for (int w = 0; w < VPL; ++w)
#pragma unroll
          for (int i = 0; i < EPV; ++i) dst[(w * LPR + gl) * EPV + i] = tot[w][i];
        if (gl == 0) p.carry_row[t * 2 + 1] = ti1 < p.rows ? ti1 : -1;
      }
    }
    __syncthreads();
  }
}

// One group per tile t that holds a head partial: row = head_row[t]; total = tails of the run of
// preceding tiles that were accumulating the same row (in tile order) + the head.  Writes C[row].
template <typename V, int LPR, int VPL>
__global__ void __launch_bounds__(256) spmm_merge_fixup_kernel(const typename VT<V>::Acc* __restrict__ carry,
                                                               const int64_t* __restrict__ carry_row, int64_t num_tiles,
                                                               int64_t kpad, int64_t K, V* __restrict__ C, int64_t ldc) {
  using Acc = typename VT<V>::Acc;
  constexpr int EPV = 16 / sizeof(V);
  const int lane = threadIdx.x & 31, gl = lane % LPR;
  const int64_t t = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPR;
  if (t >= num_tiles) return;
  const int64_t row = carry_row[2 * t];
  if (row < 0) return;
  int64_t lo = t;
  while (lo > 0 && carry_row[2 * (lo - 1) + 1] == row) --lo;
  Acc tot[VPL][EPV];
#pragma unroll
  for (int w = 0; w < VPL; ++w)
#pragma unroll
    for (int i = 0; i < EPV; ++i) tot[w][i] = Acc(0);
  for (int64_t q = lo; q < t; ++q) {
    const Acc* src = carry + (q * 2 + 1) * kpad;
#pragma unroll
    for (int w = 0; w < VPL; ++w)
#pragma unroll
      for (int i = 0; i < EPV; ++i) tot[w][i] += src[(w * LPR + gl) * EPV + i];
  }
  const Acc* src = carry + (t * 2) * kpad;
#pragma unroll
  for (int w = 0; w < VPL; ++w)
#pragma unroll
    for (int i = 0; i < EPV; ++i) tot[w][i] += src[(w * LPR + gl) * EPV + i];
#pragma unroll
  for (int w = 0; w < VPL; ++w)
    if ((int64_t)(w * LPR + gl) * EPV < K) store_vec<V, EPV>(C + row * ldc + (int64_t)(w * LPR + gl) * EPV, tot[w]);
}

template <typename V, typename I, int LPR, int VPL, bool PERM>
static int launch_spmm_merge(const I* rowptr, const I* colind, const V* vals, const I* perm, const V* B, V* C,
                             int64_t rows, int64_t K, int64_t nnz, int64_t b_rs, int64_t ldc, void* ws, size_t ws_bytes,
                             cudaStream_t s) {
  using Acc = typename VT<V>::Acc;
  constexpr int EPV = 16 / sizeof(V);
  constexpr int U0 = TSGU_MERGE_LOADS / VPL;
  constexpr int U = U0 < LPR ? U0 : LPR;
  const int64_t num_tiles = (rows + nnz + MERGE_P - 1) / MERGE_P;
  const int64_t kpad = (int64_t)LPR * VPL * EPV;
  const size_t part_bytes = ((size_t)(num_tiles + 1) * 2 * sizeof(int64_t) + 255) / 256 * 256;
  const size_t row_bytes = ((size_t)num_tiles * 2 * sizeof(int64_t) + 255) / 256 * 256;
  const size_t carry_bytes = (size_t)num_tiles * 2 * kpad * sizeof(Acc);
  if (!ws || ws_bytes < part_bytes + row_bytes + carry_bytes) return TSGU_ERR_WORKSPACE;
  MergeSpmmParams<V, I> p;
  p.rowptr = rowptr; p.colind = colind; p.vals = vals; p.perm = perm; p.B = B; p.C = C;
  p.rows = rows; p.K = K; p.nnz = nnz; p.b_rs = b_rs; p.ldc = ldc; p.kpad = kpad;
  int64_t* part = (int64_t*)ws;
  p.part = part;
  p.carry_row = (int64_t*)((char*)ws + part_bytes);
  p.carry = (Acc*)((char*)ws + part_bytes + row_bytes);

  merge_partition_kernel<I><<<(unsigned)((num_tiles + 1 + 255) / 256), 256, 0, s>>>(rowptr, rows, nnz, num_tiles, part);
  count_launch();
  const bool exact = (K / EPV) == (int64_t)LPR * VPL;
  auto kern = exact ? spmm_merge_kernel<V, I, LPR, VPL, U, true, PERM> : spmm_merge_kernel<V, I, LPR, VPL, U, false, PERM>;
  const int smem = (int)sizeof(MergeSpmmSmem<V, I, PERM ? 2 : 1, LPR, VPL>);
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return (int)e;
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 256, smem) != cudaSuccess || occ < 1) occ = 1;
  int64_t grid = persistent_sms() * occ;
  if (grid > num_tiles) grid = num_tiles;
  kern<<<(unsigned)grid, 256, smem, s>>>(p, num_tiles);
  count_launch();
  const int64_t fix_threads = num_tiles * LPR;
  spmm_merge_fixup_kernel<V, LPR, VPL><<<(unsigned)((fix_threads + 255) / 256), 256, 0, s>>>(p.carry, p.carry_row, num_tiles,
                                                                                            kpad, K, C, ldc);
  count_launch();
  return launch_status();
}

size_t spmm_merge_workspace_bytes(int64_t rows, int64_t K, int64_t nnz, int val_dtype) {
  const int64_t num_tiles = (rows + nnz + MERGE_P - 1) / MERGE_P;
  const int esz = val_dtype == TSGU_F64 ? 8 : val_dtype == TSGU_BF16 ? 2 : 4;
  const int asz = val_dtype == TSGU_F64 ? 8 : 4;
  const int epv = 16 / esz;
  int64_t kv = (K + epv - 1) / epv;  // vectors per row -> lane tiling used by the dispatcher
  int64_t slots = kv <= 4 ? 4 : kv <= 8 ? 8 : kv <= 16 ? 16 : kv <= 32 ? 32 : kv <= 64 ? 64 : 128;  // = LPR*VPL in both lane tables
  const int64_t kpad = slots * epv;
  const size_t part_bytes = ((size_t)(num_tiles + 1) * 2 * sizeof(int64_t) + 255) / 256 * 256;
  const size_t row_bytes = ((size_t)num_tiles * 2 * sizeof(int64_t) + 255) / 256 * 256;
  return part_bytes + row_bytes + (size_t)num_tiles * 2 * kpad * asz;
}

// true if the merge-path SpMM can take this problem (same addressing requirements as the tile path)
template <typename V, typename I>
int spmm_merge_dispatch(const I* rowptr, const I* colind, const V* vals, const I* perm, const V* B, V* C, int64_t rows,
                        int64_t K, int64_t nnz, int64_t b_rs, int64_t ldc, void* ws, size_t ws_bytes, cudaStream_t s) {
  constexpr int EPVF = 16 / sizeof(V);
  const int64_t kv = K / EPVF;
#define TSGU_MERGE(LPR_, VPL_)                                                                                      \
  return perm ? launch_spmm_merge<V, I, LPR_, VPL_, true>(rowptr, colind, vals, perm, B, C, rows, K, nnz, b_rs, ldc, ws, ws_bytes, s) \
              : launch_spmm_merge<V, I, LPR_, VPL_, false>(rowptr, colind, vals, perm, B, C, rows, K, nnz, b_rs, ldc, ws, ws_bytes, s)
  if (kv <= 4) TSGU_MERGE(4, 1);
  if (kv <= 8) TSGU_MERGE(8, 1);
  // 8-lane groups with 2-4 vectors per lane, as the tile kernels (config 4: 9.7 ms with 16/32-lane groups, 9.2 ms)
  if (kv <= 16) TSGU_MERGE(8, 2);
  if (kv <= 32) TSGU_MERGE(8, 4);
  if (kv <= 64) TSGU_MERGE(16, 4);
  TSGU_MERGE(32, 4);
#undef TSGU_MERGE
}

#define TSGU_INST_MERGE(V, I)                                                                                     \
  template int spmm_merge_dispatch<V, I>(const I*, const I*, const V*, const I*, const V*, V*, int64_t, int64_t,  \
                                         int64_t, int64_t, int64_t, void*, size_t, cudaStream_t);
TSGU_INST_MERGE(float, int32_t)
TSGU_INST_MERGE(float, int64_t)
TSGU_INST_MERGE(double, int32_t)
TSGU_INST_MERGE(double, int64_t)
TSGU_INST_MERGE(__nv_bfloat16, int32_t)
TSGU_INST_MERGE(__nv_bfloat16, int64_t)


// Reduce NB per-lane partials across the LPR lanes of a group (see sddmm.cu): lane gl ends up with the
// total of entry gl / (LPR/NB) in p[0].
template <typename Acc, int LPR, int NB>
__device__ __forceinline__ void butterfly_reduce_m(Acc (&p)[NB], unsigned gmask, int gl) {
  int width = NB;
#pragma unroll
  for (int s = LPR / 2; s >= 1; s >>= 1) {
    if (width > 1) {
      const int half = width / 2;
      const bool upper = (gl & s) != 0;
#pragma unroll
      for (int i = 0; i < NB / 2; ++i) {
        if (i < half) {
          const Acc send = upper ? p[i] : p[i + half];
          const Acc keep = upper ? p[i + half] : p[i];
          p[i] = keep + shfl_x(gmask, send, s);
        }
      }
      width = half;
    } else {
      p[0] += shfl_x(gmask, p[0], s);
    }
  }
}

// ========================================================================================== SDDMM
// Same decomposition; entries are independent, so there are no carries -- only the row of the
// upstream gradient held in registers has to follow the row structure.
template <typename V, typename I>
struct MergeSddmmParams {
  const I* rowptr; const I* colind; const I* out_index; const V* G; const V* B; V* out;
  int64_t rows, K, nnz, g_rs, b_rs;
  const int64_t* part;
};

template <typename V, typename I>
struct MergeSddmmSmem {
  MergeStage<V, I, 0> st[2];
  alignas(8) uint64_t full[2];
};

template <typename V, typename I, int LPR, int VPL, int NB, int U, bool EXACT>
__global__ void __launch_bounds__(256, TSGU_MERGE_SDDMM_MINB) sddmm_merge_kernel(const MergeSddmmParams<V, I> p, const int64_t num_tiles) {
  using Acc = typename VT<V>::Acc;
  using Stage = MergeStage<V, I, 0>;
  using Smem = MergeSddmmSmem<V, I>;
  constexpr int EPV = 16 / sizeof(V);
  constexpr int AI = Stage::AI;
  constexpr int GROUPS = 256 / LPR;
  constexpr int LPE = LPR / NB;
  static_assert(NB % U == 0, "batch is processed in chunks of U entries");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);

  const int tid = threadIdx.x, lane = tid & 31, gl = lane % LPR, group = tid / LPR;
  const unsigned gmask = group_mask<LPR>(lane);
  const int kv = (int)(p.K / EPV);
  const uint32_t row_bytes = (uint32_t)(p.b_rs * sizeof(V));
  bool on[VPL];
#pragma unroll
  for (int w = 0; w < VPL; ++w) on[w] = EXACT || (w * LPR + gl < kv);

  if (tid == 0) {
    mbar_init(&sm.full[0], 1);
    mbar_init(&sm.full[1], 1);
    mbar_fence_init();
  }
  __syncthreads();

  MergeProducer<V, I, 0> prod{p.rowptr, p.colind, nullptr, nullptr, p.rows + 1, p.nnz};
  const int64_t t0 = blockIdx.x;
  int64_t n_i0 = 0, n_j0 = 0, n_i1 = 0, n_j1 = 0;
  if (tid == 0 && t0 < num_tiles) {
    prod.issue(sm.st[0], &sm.full[0], p.part[2 * t0], p.part[2 * t0 + 1], p.part[2 * t0 + 2], p.part[2 * t0 + 3]);
    const int64_t tn = t0 + gridDim.x;
    if (tn < num_tiles) { n_i0 = p.part[2 * tn]; n_j0 = p.part[2 * tn + 1]; n_i1 = p.part[2 * tn + 2]; n_j1 = p.part[2 * tn + 3]; }
  }

  const char* Bb = reinterpret_cast<const char*>(p.B) + (size_t)gl * 16;
  int it = 0;
  for (int64_t t = t0; t < num_tiles; t += gridDim.x, ++it) {
    const int stage = it & 1;
    if (tid == 0) {
      const int64_t tn = t + gridDim.x;
      if (tn < num_tiles) {
        prod.issue(sm.st[stage ^ 1], &sm.full[stage ^ 1], n_i0, n_j0, n_i1, n_j1);
        const int64_t tnn = tn + gridDim.x;
        if (tnn < num_tiles) { n_i0 = p.part[2 * tnn]; n_j0 = p.part[2 * tnn + 1]; n_i1 = p.part[2 * tnn + 2]; n_j1 = p.part[2 * tnn + 3]; }
      }
    }
    const int64_t ti0 = __ldg(p.part + 2 * t), tj0 = __ldg(p.part + 2 * t + 1);
    const int64_t ti1 = __ldg(p.part + 2 * t + 2), tj1 = __ldg(p.part + 2 * t + 3);
    mbar_wait(&sm.full[stage], (uint32_t)((it >> 1) & 1));

    const Stage& st = sm.st[stage];
    const I* rp = st.rp + (int)(ti0 & (AI - 1));
    const I* scol = st.col + (int)(tj0 & (AI - 1));
    const int nnz_t = (int)(tj1 - tj0);

    // entries are split evenly over the groups (multiples of NB so every batch is full but the last);
    // tile-local 32-bit coordinates: this group's entries are [gj0l, gj1l)
    int per = (nnz_t + GROUPS - 1) / GROUPS;
    per = (per + NB - 1) / NB * NB;
    int gj0l = group * per, gj1l = gj0l + per;
    if (gj0l > nnz_t) gj0l = nnz_t;
    if (gj1l > nnz_t) gj1l = nnz_t;

    if (gj0l < gj1l) {
      // row of the first entry: last row r in the slice with rowptr[r] <= gj0
      const int64_t gj0 = tj0 + gj0l;
      int lo = 0, hi = (int)(ti1 - ti0) + 1;  // rp[lo] <= gj0 < rp[hi] (rp[rows_t + 1] > tj1 - 1 >= gj0)
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if ((int64_t)rp[mid] <= gj0) lo = mid; else hi = mid;
      }
      int rowl = lo;
      // local end of the current row, clamped: a row that runs past the tile ends "never" for this tile
      auto local_end = [&](int r) {
        const int64_t d = (int64_t)rp[r + 1] - tj0;
        return d > (int64_t)nnz_t ? INT_MAX : (int)d;
      };
      int row_end = local_end(rowl);
      Acc g[VPL][EPV];
      auto load_g = [&]() {
        const V* Grow = p.G + (ti0 + rowl) * p.g_rs;
#pragma unroll
        for (int w = 0; w < VPL; ++w) {
          Raw<V, EPV> raw = (EXACT || on[w]) ? raw_ldg<V, EPV>(Grow + (int64_t)(w * LPR + gl) * EPV) : raw_zero<V, EPV>();
          raw_unpack<V, EPV>(raw, g[w]);
        }
      };
      load_g();
      auto next_row = [&](int eu) {  // skip empties, fetch that row of G
        do {
          ++rowl;
          row_end = local_end(rowl);
        } while (eu >= row_end);
        load_g();
      };
      auto dot = [&](const uint4 (&bu)[VPL], Acc& out) {
#pragma unroll
        for (int w = 0; w < VPL; ++w) {
          Acc x[EPV];
          Raw<V, EPV> raw;
          raw.bits = bu[w];
          raw_unpack<V, EPV>(raw, x);
#pragma unroll
          for (int i = 0; i < EPV; ++i) out = fma(g[w][i], x[i], out);
        }
      };

      for (int basel = gj0l; basel < gj1l; basel += NB) {
        const int el = basel + gl;
        uint32_t cu = 0;
        if (gl < NB && el < gj1l) cu = (uint32_t)scol[el];
        const int cnt = min(NB, gj1l - basel);
        Acc part[NB];
#pragma unroll
        for (int j = 0; j < NB; ++j) part[j] = Acc(0);
        if (cnt == NB) {  // full batch (group-uniform branch): nothing is predicated
#pragma unroll
          for (int j0 = 0; j0 < NB; j0 += U) {
            uint4 b[U][VPL];
#pragma unroll
            for (int u = 0; u < U; ++u) {
              const uint32_t cj = shfl_idx(gmask, cu, j0 + u, LPR);
              const char* brow = Bb + (uint64_t)cj * row_bytes;
#pragma unroll
              for (int w = 0; w < VPL; ++w) {
                if (EXACT || on[w]) b[u][w] = __ldg(reinterpret_cast<const uint4*>(brow + w * (LPR * 16)));
                else b[u][w] = make_uint4(0, 0, 0, 0);
              }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
              const int eu = basel + j0 + u;
              if (eu >= row_end) next_row(eu);
              dot(b[u], part[j0 + u]);
            }
          }
        } else {  // ragged end of this group's range
#pragma unroll
          for (int j0 = 0; j0 < NB; j0 += U) {
            if (j0 < cnt) {
              uint4 b[U][VPL];
#pragma unroll
              for (int u = 0; u < U; ++u) {
                const uint32_t cj = shfl_idx(gmask, cu, j0 + u, LPR);
                const char* brow = Bb + (uint64_t)cj * row_bytes;
#pragma unroll
                for (int w = 0; w < VPL; ++w) {
                  b[u][w] = make_uint4(0, 0, 0, 0);
                  if (j0 + u < cnt && (EXACT || on[w])) b[u][w] = __ldg(reinterpret_cast<const uint4*>(brow + w * (LPR * 16)));
                }
              }
#pragma unroll
              for (int u = 0; u < U; ++u) {
                if (j0 + u < cnt) {
                  const int eu = basel + j0 + u;
                  if (eu >= row_end) next_row(eu);
                  dot(b[u], part[j0 + u]);
                }
              }
            }
          }
        }
        butterfly_reduce_m<Acc, LPR, NB>(part, gmask, gl);
        const int slot = gl / LPE;
        if ((gl % LPE) == 0 && slot < cnt) {
          const int64_t eo = tj0 + basel + slot;
          int64_t dst = eo;
          if (p.out_index) dst = (int64_t)__ldg(p.out_index + eo);
          if (dst >= 0) p.out[dst] = VT<V>::from_acc(part[0]);
        }
      }
    }
    __syncthreads();
  }
}

template <typename V, typename I, int LPR, int VPL>
static int launch_sddmm_merge(const MergeSddmmParams<V, I>& p0, void* ws, size_t ws_bytes, cudaStream_t s) {
  constexpr int EPV = 16 / sizeof(V);
  constexpr int NB = LPR < 16 ? LPR : 16;
  constexpr int U0 = TSGU_MERGE_SDDMM_LOADS / VPL;
  constexpr int U = U0 < NB ? U0 : NB;
  MergeSddmmParams<V, I> p = p0;
  const int64_t num_tiles = (p.rows + p.nnz + MERGE_P - 1) / MERGE_P;
  const size_t part_bytes = (size_t)(num_tiles + 1) * 2 * sizeof(int64_t);
  if (!ws || ws_bytes < part_bytes) return TSGU_ERR_WORKSPACE;
  int64_t* part = (int64_t*)ws;
  p.part = part;
  merge_partition_kernel<I><<<(unsigned)((num_tiles + 1 + 255) / 256), 256, 0, s>>>(p.rowptr, p.rows, p.nnz, num_tiles, part);
  count_launch();
  const bool exact = (p.K / EPV) == (int64_t)LPR * VPL;
  auto kern = exact ? sddmm_merge_kernel<V, I, LPR, VPL, NB, U, true> : sddmm_merge_kernel<V, I, LPR, VPL, NB, U, false>;
  const int smem = (int)sizeof(MergeSddmmSmem<V, I>);
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return (int)e;
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 256, smem) != cudaSuccess || occ < 1) occ = 1;
  int64_t grid = persistent_sms() * occ;
  if (grid > num_tiles) grid = num_tiles;
  kern<<<(unsigned)grid, 256, smem, s>>>(p, num_tiles);
  count_launch();
  return launch_status();
}

size_t sddmm_merge_workspace_bytes(int64_t rows, int64_t nnz) {
  const int64_t num_tiles = (rows + nnz + MERGE_P - 1) / MERGE_P;
  return (size_t)(num_tiles + 1) * 2 * sizeof(int64_t);
}

template <typename V, typename I>
int sddmm_merge_dispatch(const I* rowptr, const I* colind, const I* out_index, const V* G, const V* B, V* out,
                         int64_t rows, int64_t K, int64_t nnz, int64_t g_rs, int64_t b_rs, void* ws, size_t ws_bytes,
                         cudaStream_t s) {
  constexpr int EPVF = 16 / sizeof(V);
  MergeSddmmParams<V, I> p{rowptr, colind, out_index, G, B, out, rows, K, nnz, g_rs, b_rs, nullptr};
  const int64_t kv = K / EPVF;
  if (kv <= 4) return launch_sddmm_merge<V, I, 4, 1>(p, ws, ws_bytes, s);
  if (kv <= 8) return launch_sddmm_merge<V, I, 8, 1>(p, ws, ws_bytes, s);
  if (kv <= 16) return launch_sddmm_merge<V, I, 8, 2>(p, ws, ws_bytes, s);
  if (kv <= 32) return launch_sddmm_merge<V, I, 8, 4>(p, ws, ws_bytes, s);
  if (kv <= 64) return launch_sddmm_merge<V, I, 16, 4>(p, ws, ws_bytes, s);
  return launch_sddmm_merge<V, I, 32, 4>(p, ws, ws_bytes, s);
}

#define TSGU_INST_MERGE_SDDMM(V, I)                                                                              \
  template int sddmm_merge_dispatch<V, I>(const I*, const I*, const I*, const V*, const V*, V*, int64_t, int64_t, \
                                          int64_t, int64_t, int64_t, void*, size_t, cudaStream_t);
TSGU_INST_MERGE_SDDMM(float, int32_t)
TSGU_INST_MERGE_SDDMM(float, int64_t)
TSGU_INST_MERGE_SDDMM(double, int32_t)
TSGU_INST_MERGE_SDDMM(double, int64_t)
TSGU_INST_MERGE_SDDMM(__nv_bfloat16, int32_t)
TSGU_INST_MERGE_SDDMM(__nv_bfloat16, int64_t)

}  // namespace tsgu
