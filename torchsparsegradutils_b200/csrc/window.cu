// window.cu -- "column-window" SpMM / SDDMM for structured sparsity (sm_100a).
//
// Banded / stencil matrices (BASELINE config 3: the 27-point PairwiseEncoder precision matrix) re-read every
// row of the dense operand once per nonzero of that column out of L1/L2, although the rows a tile of
// consecutive rows of A touches form a handful of contiguous runs (for a 3-D stencil: one run per (dz, dy)
// offset pair).  Here that structure is found ONCE per sparsity pattern and then exploited by the kernels:
//
//   tsgu_window_plan   per tile of T rows: bitmap of the columns it touches -> dense rank of every column
//                      (its slot in the tile's window), the maximal runs of consecutive columns, and a
//                      16-bit window slot per stored entry (replaces the 32/64-bit column index: the sparse
//                      operand gets SMALLER).  One CTA per tile, no sort.  A tile that does not fit (too many
//                      distinct columns / runs, too wide a span, too many entries) is flagged; the host uses
//                      the plan only if no tile is.
//   spmm_window_kernel / sddmm_window_kernel
//                      persistent CTAs with a dedicated PRODUCER WARP: lane r issues one cp.async.bulk for
//                      run r of the next tile (contiguous rows of the dense operand -> the stage's window in
//                      shared memory), lane 0 adds the tile's rowptr / slot / value slices; everything
//                      completes on the stage's `full` mbarrier.  The consumer warps gather dense rows from
//                      SHARED memory (LDS.128), never wait on global memory, and hand the stage back through
//                      an `empty` mbarrier -- no CTA-wide barrier anywhere in the loop.
//
// Replaces the same ATen call sites as spmm.cu / sddmm.cu (reference sparse_matmul.py:155, :229, :190-205).
// Arithmetic and accumulation order per row are those of the row-tile kernels (CSR order, fp32 accumulate).
#include <climits>
#include <type_traits>

#include "common.cuh"
#include "tile.cuh"

#ifndef TSGU_WIN_STAGES
#define TSGU_WIN_STAGES 2
#endif
#ifndef TSGU_WIN_ROWS
#define TSGU_WIN_ROWS 320   // dense rows a stage's window holds
#endif
#ifndef TSGU_WIN_ECAP
#define TSGU_WIN_ECAP 1024  // stored entries a tile may hold
#endif
#ifndef TSGU_WIN_TMAX
#define TSGU_WIN_TMAX 64    // rows per tile (capacity of the staged rowptr slice)
#endif
#ifndef TSGU_WIN_CW
#define TSGU_WIN_CW 8       // consumer warps per CTA
#endif
#ifndef TSGU_WIN_LPR8
#define TSGU_WIN_LPR8 8     // lanes per row for 8-vector dense rows (8 x 1 vector or 4 x 2 vectors per lane)
#endif

namespace tsgu {

constexpr int WIN_RMAX = 15;          // runs per tile descriptor
constexpr int WIN_DESC_WORDS = 32;    // int32 words per tile: [0] nruns (-1: does not fit), [1] distinct columns,
                                      // then per run: first column, slot | len << 16
constexpr int WIN_SPAN_WORDS = 8192;  // bitmap words per tile: column span <= 262144 (dynamic smem: 2 bitmaps + ranks = 80 KB)
constexpr int WIN_CLOSE = 8;          // holes between touched columns are bridged when a touched column lies within
                                      // WIN_CLOSE on either side (fewer, longer runs; the bridged rows are loaded unused)

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// =========================================================================================== plan
// exclusive block scan of two counters (256 threads); also returns the block totals
__device__ __forceinline__ void block_scan2(int a, int b, int& ea, int& eb, int& ta, int& tb, int (*wsum)[8]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int ia = a, ib = b;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int xa = __shfl_up_sync(0xffffffffu, ia, o), xb = __shfl_up_sync(0xffffffffu, ib, o);
    if (lane >= o) { ia += xa; ib += xb; }
  }
  if (lane == 31) { wsum[0][warp] = ia; wsum[1][warp] = ib; }
  __syncthreads();
  int oa = 0, ob = 0, sa = 0, sb = 0;
#pragma unroll
  for (int w = 0; w < 8; ++w) {
    if (w < warp) { oa += wsum[0][w]; ob += wsum[1][w]; }
    sa += wsum[0][w]; sb += wsum[1][w];
  }
  ea = oa + ia - a; eb = ob + ib - b; ta = sa; tb = sb;
  __syncthreads();
}

template <typename I>
__global__ void __launch_bounds__(256) window_plan_kernel(const I* __restrict__ rowptr, const I* __restrict__ colind,
                                                          int64_t n, int64_t rowptr_bstride, int64_t nnz_bstride,
                                                          int tile_rows, int64_t tiles_per_item, int64_t num_tiles,
                                                          int wrows_cap, int ecap, uint16_t* __restrict__ lcol,
                                                          int32_t* __restrict__ desc, int32_t* __restrict__ stats) {
  extern __shared__ __align__(16) unsigned char plan_smem[];
  uint32_t* touched = reinterpret_cast<uint32_t*>(plan_smem);       // columns some entry of the tile sits in
  uint32_t* bitmap = touched + WIN_SPAN_WORDS;                      // ... plus the bridged holes: what gets loaded
  uint16_t* prefix = reinterpret_cast<uint16_t*>(bitmap + WIN_SPAN_WORDS);
  __shared__ int wsum[2][8];
  __shared__ long long red_min[8], red_max[8];
  __shared__ int run_slot[WIN_RMAX + 1];
  __shared__ int run_col[WIN_RMAX + 1];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  for (int64_t t = blockIdx.x; t < num_tiles; t += gridDim.x) {
    const TileCoord c = tile_coord(t, tiles_per_item, n, tile_rows);
    const I* rp = rowptr + c.item * rowptr_bstride + c.r0;
    const int64_t s_abs = (int64_t)rp[0] + c.item * nnz_bstride;
    const int64_t e_abs = (int64_t)rp[c.rows] + c.item * nnz_bstride;
    const int64_t cnt = e_abs - s_abs;
    int32_t* d = desc + t * WIN_DESC_WORDS;
    if (cnt <= 0) {
      if (tid == 0) { d[0] = 0; d[1] = 0; }
      continue;
    }
    // column span of the tile
    long long lo = LLONG_MAX, hi = -1;
    for (int64_t e = s_abs + tid; e < e_abs; e += 256) {
      const long long col = (long long)colind[e];
      lo = col < lo ? col : lo;
      hi = col > hi ? col : hi;
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
      const long long a = __shfl_xor_sync(0xffffffffu, lo, o), b = __shfl_xor_sync(0xffffffffu, hi, o);
      lo = a < lo ? a : lo;
      hi = b > hi ? b : hi;
    }
    if (lane == 0) { red_min[warp] = lo; red_max[warp] = hi; }
    __syncthreads();
    lo = red_min[0]; hi = red_max[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) {
      lo = red_min[w] < lo ? red_min[w] : lo;
      hi = red_max[w] > hi ? red_max[w] : hi;
    }
    const long long span = hi - lo + 1;
    bool fail = cnt > ecap || span > (long long)WIN_SPAN_WORDS * 32 || lo < 0 || hi > 0x7fffffffLL;
    int total = 0, nruns = 0;
    if (!fail) {  // block-uniform
      const int nwords = (int)((span + 31) >> 5);
      for (int w = tid; w < nwords; w += 256) touched[w] = 0u;
      __syncthreads();
      for (int64_t e = s_abs + tid; e < e_abs; e += 256) {
        const uint32_t rel = (uint32_t)((long long)colind[e] - lo);
        atomicOr(&touched[rel >> 5], 1u << (rel & 31));
      }
      __syncthreads();
      // closing: a column is loaded if it is touched, or has touched columns within WIN_CLOSE on both sides
      for (int w = tid; w < nwords; w += 256) {
        const uint32_t x = touched[w], xl = w > 0 ? touched[w - 1] : 0u, xr = w + 1 < nwords ? touched[w + 1] : 0u;
        uint32_t from_below = 0u, from_above = 0u;  // a touched column at distance 1..WIN_CLOSE below / above
#pragma unroll
        for (int k = 1; k <= WIN_CLOSE; ++k) {
          from_below |= (x << k) | (xl >> (32 - k));
          from_above |= (x >> k) | (xr << (32 - k));
        }
        bitmap[w] = x | (from_below & from_above);
      }
      __syncthreads();
      const int ch = (nwords + 255) / 256;
      const int w0 = tid * ch, w1 = (w0 + ch < nwords) ? w0 + ch : nwords;
      int cb = 0, cs = 0;
      for (int w = w0; w < w1; ++w) {
        const uint32_t bits = bitmap[w];
        const uint32_t prev = w > 0 ? bitmap[w - 1] >> 31 : 0u;
        cb += __popc(bits);
        cs += __popc(bits & ~((bits << 1) | prev));
      }
      int eb, es;
      block_scan2(cb, cs, eb, es, total, nruns, wsum);
      int running = eb, ridx = es;
      for (int w = w0; w < w1; ++w) {
        const uint32_t bits = bitmap[w];
        const uint32_t prev = w > 0 ? bitmap[w - 1] >> 31 : 0u;
        prefix[w] = (uint16_t)(running > 0xffff ? 0xffff : running);
        uint32_t starts = bits & ~((bits << 1) | prev);
        while (starts) {
          const int b = __ffs(starts) - 1;
          starts &= starts - 1;
          if (ridx < WIN_RMAX) {
            run_col[ridx] = (int)(lo + (long long)w * 32 + b);
            run_slot[ridx] = running + __popc(bits & ((1u << b) - 1u));
          }
          ++ridx;
        }
        running += __popc(bits);
      }
      fail = total > wrows_cap || total > 0xffff || nruns > WIN_RMAX;
      __syncthreads();
      if (!fail) {
        for (int64_t e = s_abs + tid; e < e_abs; e += 256) {
          const uint32_t rel = (uint32_t)((long long)colind[e] - lo);
          const uint32_t bits = bitmap[rel >> 5];
          lcol[e] = (uint16_t)(prefix[rel >> 5] + __popc(bits & ((1u << (rel & 31)) - 1u)));
        }
        if (tid < nruns) {
          const int nxt = (tid + 1 < nruns) ? run_slot[tid + 1] : total;
          d[2 + 2 * tid] = run_col[tid];
          d[3 + 2 * tid] = (int32_t)((uint32_t)run_slot[tid] | ((uint32_t)(nxt - run_slot[tid]) << 16));
        }
      }
    }
    if (tid == 0) {
      d[0] = fail ? -1 : nruns;
      d[1] = total;
      if (fail) atomicAdd(&stats[0], 1);
      atomicMax(&stats[1], total);
      atomicMax(&stats[2], nruns);
      atomicMax(&stats[3], (int)(cnt > 0x7fffffffLL ? 0x7fffffffLL : cnt));
    }
    __syncthreads();
  }
}

// ======================================================================================== kernels
template <typename V, typename I, int ROWB, bool GROWS = false>
struct WinStage {
  static constexpr int AI = 16 / (int)sizeof(I), AV = 16 / (int)sizeof(V);
  alignas(128) unsigned char win[TSGU_WIN_ROWS * ROWB];
  alignas(128) unsigned char grows[GROWS ? TSGU_WIN_TMAX * ROWB : 16];  // SDDMM: the tile's rows of the left operand
  alignas(16) I rp[TSGU_WIN_TMAX + 1 + 2 * AI];
  alignas(16) uint16_t lcol[TSGU_WIN_ECAP + 16];
  alignas(16) V val[TSGU_WIN_ECAP + 2 * AV];
};

#ifndef TSGU_WIN_LOOKAHEAD
#define TSGU_WIN_LOOKAHEAD 8
#endif
template <typename I>
struct WinInfoRing {
  alignas(16) int32_t desc[TSGU_WIN_LOOKAHEAD][WIN_DESC_WORDS];
  alignas(16) I bounds[TSGU_WIN_LOOKAHEAD][2];
};
template <typename V, typename I, int ROWB, bool GROWS = false>
struct WinSmem {
  WinStage<V, I, ROWB, GROWS> st[TSGU_WIN_STAGES];
  WinInfoRing<I> ring;
  // SpMM with a column-major result: double-buffered CTA scratch for the (rows of one pass) x K transpose; rows are
  // padded by one element (conflict-free column reads).  Sized for 64 rows per pass (4-lane groups).
  alignas(16) unsigned char cscr[GROWS ? 16 : 2 * 64 * (ROWB + 4)];
  alignas(8) uint64_t full[TSGU_WIN_STAGES];
  alignas(8) uint64_t empty[TSGU_WIN_STAGES];
};

template <typename V, typename I>
struct WinParams {
  const I* rowptr;
  const uint16_t* lcol;
  const int32_t* desc;
  const V* vals;       // SpMM, in pattern order
  const I* out_index;  // SDDMM, nullable
  const V* G;          // SDDMM: left dense operand (rows of A)
  const V* B;          // windowed dense operand (columns of A)
  V* out;              // SpMM: C; SDDMM: values
  int64_t batch, n;
  int64_t rowptr_bstride, nnz_bstride, rowptr_len, nnz_len;
  int64_t b_bs, b_rs, g_bs, g_rs, c_bs, ldc;
  int64_t c_cs;  // SpMM result: element (r, k) of an item at r * ldc + k * c_cs; c_cs == 1 row-major, ldc == 1 column-major
  int64_t tiles_per_item, num_tiles;
  int tile_rows;
};

// Tiles are walked with a stride of gridDim.x; (item, first row) are kept incrementally in 32 bits (no division).
struct WinTileIter {
  int item, tile;  // batch item, tile index inside the item
  int tiles_per_item, step;
  __device__ __forceinline__ WinTileIter(int64_t first, int64_t tpi, int stride) : tiles_per_item((int)tpi), step(stride) {
    item = (int)(first / tpi);
    tile = (int)(first - (int64_t)item * tpi);
  }
  __device__ __forceinline__ void next() {
    tile += step;
    while (tile >= tiles_per_item) { tile -= tiles_per_item; ++item; }
  }
};

__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}

// What the producer warp needs to know about a tile: its run descriptor and its entry range.  They are
// fetched TSGU_WIN_LOOKAHEAD tiles ahead of their use with per-lane cp.async copies into a small shared-memory
// ring, so that no global-load latency sits between a stage being released and its refill being issued.
struct WinTileInfo {
  int nruns;
  uint32_t col0, sl;     // this lane's run
  int64_t s_abs, e_abs;  // lane 0: entry range of the tile
};

__device__ __forceinline__ void cp_async4(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async8(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <typename V, typename I>
__device__ __forceinline__ void win_fetch_info(const WinParams<V, I>& p, WinInfoRing<I>& ring, int slot, int64_t t, int item,
                                               int r0, int rows, int lane) {
  if (t < p.num_tiles) {
    cp_async4(&ring.desc[slot][lane], p.desc + t * WIN_DESC_WORDS + lane);
    if (lane < 2) {
      const I* src = p.rowptr + (int64_t)item * p.rowptr_bstride + r0 + (lane ? rows : 0);
      if constexpr (sizeof(I) == 4) cp_async4(&ring.bounds[slot][lane], src);
      else cp_async8(&ring.bounds[slot][lane], src);
    }
  }
  cp_async_commit();  // one group per slot, committed even when empty, so the group count stays uniform
}

// producer warp: stream a tile into stage `st`
template <typename V, typename I, int ROWB, bool WITH_VALS>
__device__ __forceinline__ void win_produce(const WinParams<V, I>& p, WinStage<V, I, ROWB, !WITH_VALS>& st, uint64_t* bar,
                                            const WinTileInfo& ti, int item, int r0, int rows, int lane) {
  using TP = TileProducer<V, I, 0>;
  uint32_t tx = 0;
  if (lane < ti.nruns) {
    const uint32_t slot = ti.sl & 0xffffu, len = ti.sl >> 16;
    const char* src = reinterpret_cast<const char*>(p.B + (int64_t)item * p.b_bs) + (size_t)ti.col0 * (size_t)(p.b_rs * sizeof(V));
    if (p.b_rs * (int64_t)sizeof(V) == ROWB) {  // dense rows are contiguous: one copy per run
      tx = len * ROWB;
      bulk_g2s(st.win + slot * ROWB, src, tx, bar);
    } else {  // padded rows: one copy per dense row
      for (uint32_t r = 0; r < len; ++r)
        bulk_g2s(st.win + (slot + r) * ROWB, src + (size_t)r * (size_t)(p.b_rs * sizeof(V)), ROWB, bar);
      tx = len * ROWB;
    }
  }
  if (lane == 0) {
    const int64_t rp_lo = (int64_t)item * p.rowptr_bstride + r0;
    tx += TP::template span<I>(st.rp, p.rowptr, rp_lo, rp_lo + rows + 1, p.rowptr_len, bar);
    if (ti.e_abs > ti.s_abs) {
      tx += TP::template span<uint16_t>(st.lcol, p.lcol, ti.s_abs, ti.e_abs, p.nnz_len, bar);
      if constexpr (WITH_VALS) tx += TP::template span<V>(st.val, p.vals, ti.s_abs, ti.e_abs, p.nnz_len, bar);
    }
  }
  if constexpr (!WITH_VALS) {  // SDDMM: the tile's rows of the upstream gradient (consecutive rows)
    if (lane == 31) {
      const char* gsrc = reinterpret_cast<const char*>(p.G + (int64_t)item * p.g_bs) + (size_t)r0 * (size_t)(p.g_rs * sizeof(V));
      if (p.g_rs * (int64_t)sizeof(V) == ROWB) {
        bulk_g2s(st.grows, gsrc, (uint32_t)rows * ROWB, bar);
      } else {
        for (int r = 0; r < rows; ++r) bulk_g2s(st.grows + r * ROWB, gsrc + (size_t)r * (size_t)(p.g_rs * sizeof(V)), ROWB, bar);
      }
      tx += (uint32_t)rows * ROWB;
    }
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) tx += __shfl_xor_sync(0xffffffffu, tx, o);
  if (lane == 0) mbar_expect_tx(bar, tx);  // the only arrival of this phase; also publishes span()'s tail stores
}

template <typename V, typename I, int ROWB, bool WITH_VALS>
__device__ __forceinline__ void win_producer_loop(const WinParams<V, I>& p, WinSmem<V, I, ROWB, !WITH_VALS>& sm, int lane) {
  constexpr int NST = TSGU_WIN_STAGES;
  constexpr int PD = TSGU_WIN_LOOKAHEAD;
  WinInfoRing<I>& ring = sm.ring;
  WinTileIter cur(blockIdx.x, p.tiles_per_item, (int)gridDim.x);  // tile being produced
  WinTileIter ahead = cur;                                        // tile whose info is being fetched
  auto geom = [&](const WinTileIter& ti, int& r0, int& rows) {
    r0 = ti.tile * p.tile_rows;
    rows = (int)p.n - r0 < p.tile_rows ? (int)p.n - r0 : p.tile_rows;
  };
  int64_t t_ahead = blockIdx.x;
#pragma unroll 1
  for (int k = 0; k < PD; ++k) {
    int r0, rows;
    geom(ahead, r0, rows);
    win_fetch_info<V, I>(p, ring, k, t_ahead, ahead.item, r0, rows, lane);
    t_ahead += gridDim.x;
    if (t_ahead < p.num_tiles) ahead.next();
  }
  int it = 0;
  for (int64_t t = blockIdx.x; t < p.num_tiles; t += gridDim.x, ++it) {
    const int slot = it % PD;
    cp_async_wait<PD - 1>();  // the oldest group = this tile's info has landed (each lane's own copies) ...
    __syncwarp();             // ... and is visible to the other lanes
    WinTileInfo ti;
    ti.nruns = ring.desc[slot][0];
    ti.col0 = (uint32_t)ring.desc[slot][(2 + 2 * lane) & (WIN_DESC_WORDS - 1)];
    ti.sl = (uint32_t)ring.desc[slot][(3 + 2 * lane) & (WIN_DESC_WORDS - 1)];
    ti.s_abs = (int64_t)ring.bounds[slot][0] + (int64_t)cur.item * p.nnz_bstride;
    ti.e_abs = (int64_t)ring.bounds[slot][1] + (int64_t)cur.item * p.nnz_bstride;
    __syncwarp();  // everyone has read the slot before it is refilled
    {
      int r0, rows;
      geom(ahead, r0, rows);
      win_fetch_info<V, I>(p, ring, slot, t_ahead, ahead.item, r0, rows, lane);
      t_ahead += gridDim.x;
      if (t_ahead < p.num_tiles) ahead.next();
    }
    int r0, rows;
    geom(cur, r0, rows);
    const int s = it % NST;
    if (it >= NST) mbar_wait(&sm.empty[s], (uint32_t)((it / NST - 1) & 1));
    win_produce<V, I, ROWB, WITH_VALS>(p, sm.st[s], &sm.full[s], ti, cur.item, r0, rows, lane);
    cur.next();
  }
  cp_async_wait<0>();
}

// ------------------------------------------------------------------------------------------ SpMM
// LPR lanes own a row, VPL 128-bit vectors per lane: LPR * VPL * 16 == ROWB == K * sizeof(V) (exact K only).
template <typename V, typename I, int LPR, int VPL, int U>
__global__ void __launch_bounds__(TSGU_WIN_CW * 32 + 32) spmm_window_kernel(const WinParams<V, I> p) {
  using Acc = typename VT<V>::Acc;
  constexpr int ROWB = LPR * VPL * 16;
  constexpr int EPV = 16 / sizeof(V);
  constexpr int NST = TSGU_WIN_STAGES;
  using Stage = WinStage<V, I, ROWB>;
  using Smem = WinSmem<V, I, ROWB>;
  constexpr int AI = Stage::AI, AV = Stage::AV;
  constexpr int GROUPS = TSGU_WIN_CW * 32 / LPR;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    for (int s = 0; s < NST; ++s) {
      mbar_init(&sm.full[s], 1);
      mbar_init(&sm.empty[s], TSGU_WIN_CW);
    }
    mbar_fence_init();
  }
  __syncthreads();

  if (warp == TSGU_WIN_CW) {  // ------------------------------------------------ producer warp
    win_producer_loop<V, I, ROWB, true>(p, sm, lane);
    return;
  }

  // --------------------------------------------------------------------------- consumer warps
  const int gl = lane % LPR;
  const int group = tid / LPR;
  const int n32 = (int)p.n;
  WinTileIter ti(blockIdx.x, p.tiles_per_item, (int)gridDim.x);
  int it = 0;
  int cm_pass = 0;  // passes stored through the column-major scratch so far (selects its buffer)
  for (int64_t t = blockIdx.x; t < p.num_tiles; t += gridDim.x, ++it, ti.next()) {
    const int s = it % NST;
    const int r0 = ti.tile * p.tile_rows;
    const int rows = n32 - r0 < p.tile_rows ? n32 - r0 : p.tile_rows;
    const Stage& st = sm.st[s];
    const int rp_shift = (int)(((int64_t)ti.item * p.rowptr_bstride + r0) & (AI - 1));
    const uint32_t win0 = smem_u32(st.win) + gl * 16;
    mbar_wait(&sm.full[s], (uint32_t)((it / NST) & 1));
    // entry positions relative to the tile's first entry: rp[] values are item-local, the tile's own offset cancels
    const int s_rel = (int)st.rp[rp_shift];
    const int s_al = (int)(((int64_t)s_rel + (int64_t)ti.item * p.nnz_bstride) & 7);
    const uint16_t* slc = st.lcol + s_al - s_rel;                 // slc[rp value] = slot of that entry
    const V* sval = st.val + (s_al & (AV - 1)) - s_rel;

    for (int lr0 = 0; lr0 < rows; lr0 += GROUPS) {  // warp-uniform trip count; a group past the tile's end idles
      const int lr = lr0 + group;
      const bool active = lr < rows;
      const int e0 = active ? (int)st.rp[rp_shift + lr] : 0;
      const int e1 = active ? (int)st.rp[rp_shift + lr + 1] : 0;
      Acc acc[VPL][EPV];
#pragma unroll
      for (int w = 0; w < VPL; ++w)
#pragma unroll
        for (int i = 0; i < EPV; ++i) acc[w][i] = Acc(0);

      auto fma_row = [&](const uint4 (&b)[VPL], const Acc vj) {
#pragma unroll
        for (int w = 0; w < VPL; ++w) {
          Acc x[EPV];
          Raw<V, EPV> raw;
          raw.bits = b[w];
          raw_unpack<V, EPV>(raw, x);
#pragma unroll
          for (int i = 0; i < EPV; ++i) acc[w][i] = fma(vj, x[i], acc[w][i]);
        }
      };

      // A row is walked in chunks of 8, 4, 2, 1 entries: every chunk is full, nothing is predicated.  (Peeling single
      // entries until the staged arrays are 4-entry aligned and reading slots / values as LDS.64 / LDS.128 vectors
      // was measured: fewer shared-memory wavefronts (95 M -> 77 M on config 3), but the peel length differs between
      // the rows of a warp, and the divergence costs more: 0.362 -> 0.374 ms.)
      auto chunk = [&](auto UC, int e) {
        constexpr int N = decltype(UC)::value;
        uint32_t slot[N];
        Acc v[N];
#pragma unroll
        for (int u = 0; u < N; ++u) {
          slot[u] = slc[e + u];
          v[u] = VT<V>::to_acc(sval[e + u]);
        }
        uint4 b[N][VPL];
#pragma unroll
        for (int u = 0; u < N; ++u)
#pragma unroll
          for (int w = 0; w < VPL; ++w) b[u][w] = lds128(win0 + slot[u] * ROWB + w * (LPR * 16));
#pragma unroll
        for (int u = 0; u < N; ++u) fma_row(b[u], v[u]);
      };
      int e = e0;
      if constexpr (U >= 8) for (; e + 8 <= e1; e += 8) chunk(std::integral_constant<int, 8>{}, e);
      if constexpr (U >= 8) { if (e + 4 <= e1) { chunk(std::integral_constant<int, 4>{}, e); e += 4; } }
      else for (; e + 4 <= e1; e += 4) chunk(std::integral_constant<int, 4>{}, e);
      if (e + 2 <= e1) { chunk(std::integral_constant<int, 2>{}, e); e += 2; }
      if (e < e1) chunk(std::integral_constant<int, 1>{}, e);
      if (p.c_cs == 1) {  // row-major result: one 128-bit store per vector
        if (active) {
          V* Crow = p.out + (int64_t)ti.item * p.c_bs + (int64_t)(r0 + lr) * p.ldc;
#pragma unroll
          for (int w = 0; w < VPL; ++w) store_vec<V, EPV>(Crow + (w * LPR + gl) * EPV, acc[w]);
        }
      } else {
        // column-major result (grad_B handed back in the layout of a column-major B): the GROUPS rows of this pass go
        // through a CTA-wide transpose in shared memory, after which every warp stores whole columns -- 32 consecutive
        // rows = one fully coalesced 128-byte (fp32) store per column.  (A warp-local 4 x K transpose with 16-byte
        // stores was measured first: half-filled sectors made the SpMM 0.13 ms slower than the layout pass it saved.)
        // One named barrier among the consumer warps per pass; the scratch is double-buffered, so a warp that runs ahead
        // cannot overwrite rows another warp is still storing.
        constexpr int KE = ROWB / (int)sizeof(V), PITCH = KE + 1;
        V* scr = reinterpret_cast<V*>(sm.cscr) + (cm_pass & 1) * (64 * PITCH);
        ++cm_pass;
        {
          V* dstrow = scr + group * PITCH;
#pragma unroll
          for (int w = 0; w < VPL; ++w)
#pragma unroll
            for (int i = 0; i < EPV; ++i) dstrow[(w * LPR + gl) * EPV + i] = VT<V>::from_acc(acc[w][i]);
        }
        asm volatile("bar.sync 1, %0;" ::"n"(TSGU_WIN_CW * 32) : "memory");
        const int pass_rows = rows - lr0 < GROUPS ? rows - lr0 : GROUPS;
        V* Cit = p.out + (int64_t)ti.item * p.c_bs + (int64_t)(r0 + lr0) * p.ldc;
        for (int idx = warp; idx < KE * (GROUPS / 32); idx += TSGU_WIN_CW) {
          const int k = idx % KE, r = (idx / KE) * 32 + lane;
          if (r < pass_rows) Cit[(int64_t)k * p.c_cs + (int64_t)r * p.ldc] = scr[r * PITCH + k];
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&sm.empty[s]);  // this warp is done reading the stage
  }
}

// ----------------------------------------------------------------------------------------- SDDMM
// SDDMM mapping: a group of LPR lanes owns a row of A; lane j computes the WHOLE dot product of entry base + j
// (no cross-lane reduction).  Every lane holds the full row of the upstream gradient in registers, in the order
// it consumes it: at step i lane j reads 16-byte chunk (i ^ (lane & 7)) of its entry's dense row, so the 8 lanes of a
// quarter warp always hit 8 different bank groups although they read 8 different rows (conflict-free LDS.128).
template <typename V, typename I, int LPR, int VPL>
__global__ void __launch_bounds__(TSGU_WIN_CW * 32 + 32) sddmm_window_kernel(const WinParams<V, I> p) {
  using Acc = typename VT<V>::Acc;
  constexpr int ROWB = LPR * VPL * 16;
  constexpr int NCH = LPR * VPL;  // 16-byte chunks per dense row
  constexpr int EPV = 16 / sizeof(V);
  constexpr int NST = TSGU_WIN_STAGES;
  using Stage = WinStage<V, I, ROWB, true>;
  using Smem = WinSmem<V, I, ROWB, true>;
  constexpr int AI = Stage::AI;
  constexpr int GROUPS = TSGU_WIN_CW * 32 / LPR;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    for (int s = 0; s < NST; ++s) {
      mbar_init(&sm.full[s], 1);
      mbar_init(&sm.empty[s], TSGU_WIN_CW);
    }
    mbar_fence_init();
  }
  __syncthreads();

  if (warp == TSGU_WIN_CW) {
    win_producer_loop<V, I, ROWB, false>(p, sm, lane);
    return;
  }

  const int gl = lane % LPR;
  const int rot = (NCH >= 8 ? lane & 7 : gl);  // chunk rotation: distinct bank groups inside every quarter warp
  const int group = tid / LPR;
  const int n32 = (int)p.n;
  WinTileIter ti(blockIdx.x, p.tiles_per_item, (int)gridDim.x);
  int it = 0;
  for (int64_t t = blockIdx.x; t < p.num_tiles; t += gridDim.x, ++it, ti.next()) {
    const int s = it % NST;
    const int r0 = ti.tile * p.tile_rows;
    const int rows = n32 - r0 < p.tile_rows ? n32 - r0 : p.tile_rows;
    const Stage& st = sm.st[s];
    const int rp_shift = (int)(((int64_t)ti.item * p.rowptr_bstride + r0) & (AI - 1));
    const uint32_t win0 = smem_u32(st.win);
    mbar_wait(&sm.full[s], (uint32_t)((it / NST) & 1));
    const int s_rel = (int)st.rp[rp_shift];
    const int64_t s_abs = (int64_t)s_rel + (int64_t)ti.item * p.nnz_bstride;
    const uint16_t* slc = st.lcol + (int)(s_abs & 7) - s_rel;

    for (int lr = group; lr < rows; lr += GROUPS) {
      const int e0 = (int)st.rp[rp_shift + lr];
      const int e1 = (int)st.rp[rp_shift + lr + 1];
      // this lane's copy of the row of the upstream gradient (staged with the tile), chunk i ^ rot at position i
      Raw<V, EPV> graw[NCH];
      {
        const uint32_t gaddr = smem_u32(st.grows) + lr * ROWB;
#pragma unroll
        for (int i = 0; i < NCH; ++i) graw[i].bits = lds128(gaddr + ((i ^ rot) << 4));
      }
      for (int base = e0; base < e1; base += LPR) {
        const int el = base + gl;
        const bool ok = el < e1;
        const uint32_t rowaddr = win0 + (ok ? (uint32_t)slc[el] : 0u) * ROWB;
        Acc part[4] = {Acc(0), Acc(0), Acc(0), Acc(0)};
#pragma unroll
        for (int i0 = 0; i0 < NCH; i0 += 4) {
          uint4 b[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) b[u] = lds128(rowaddr + (((i0 + u) ^ rot) << 4));
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            Acc x[EPV], g[EPV];
            Raw<V, EPV> raw;
            raw.bits = b[u];
            raw_unpack<V, EPV>(raw, x);
            raw_unpack<V, EPV>(graw[i0 + u], g);
#pragma unroll
            for (int k = 0; k < EPV; ++k) part[u] = fma(g[k], x[k], part[u]);
          }
        }
        if (ok) {
          const int64_t eo = (int64_t)el + (int64_t)ti.item * p.nnz_bstride;
          int64_t dst = eo;
          if (p.out_index) dst = (int64_t)__ldg(p.out_index + eo);
          if (dst >= 0) p.out[dst] = VT<V>::from_acc((part[0] + part[1]) + (part[2] + part[3]));
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&sm.empty[s]);
  }
}

// ---------------------------------------------------------------------------------------- launch
template <typename Kern, typename Params>
static int win_launch(Kern kern, int smem, int64_t num_tiles, cudaStream_t s, int* occ_cache, const Params& params) {
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return (int)e;
  if (*occ_cache == 0) {
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, TSGU_WIN_CW * 32 + 32, smem) != cudaSuccess || occ < 1) occ = 1;
    *occ_cache = occ;
  }
  int64_t grid = persistent_sms() * *occ_cache;
  if (grid > num_tiles) grid = num_tiles;
  kern<<<(unsigned)grid, TSGU_WIN_CW * 32 + 32, smem, s>>>(params);
  count_launch();
  return launch_status();
}

template <typename V, typename I, int LPR, int VPL>
static int launch_spmm_window(const WinParams<V, I>& p, cudaStream_t s) {
  constexpr int ROWB = LPR * VPL * 16;
  constexpr int U = VPL >= 4 ? 2 : (VPL == 2 ? 4 : 8);
  static int occ = 0;
  return win_launch(spmm_window_kernel<V, I, LPR, VPL, U>, (int)sizeof(WinSmem<V, I, ROWB>), p.num_tiles, s, &occ, p);
}

template <typename V, typename I, int LPR, int VPL>
static int launch_sddmm_window(const WinParams<V, I>& p, cudaStream_t s) {
  constexpr int ROWB = LPR * VPL * 16;
  static int occ = 0;
  return win_launch(sddmm_window_kernel<V, I, LPR, VPL>, (int)sizeof(WinSmem<V, I, ROWB, true>), p.num_tiles, s, &occ, p);
}

template <typename V, typename I>
static int window_dispatch(const WinParams<V, I>& p, int64_t K, bool sddmm, cudaStream_t s) {
  constexpr int EPV = 16 / (int)sizeof(V);
  if (K % EPV) return TSGU_ERR_SHAPE;
  const int64_t kv = K / EPV;  // 128-bit vectors per dense row; the window kernels take exact widths only
#define TSGU_WIN(LPR_, VPL_) return sddmm ? launch_sddmm_window<V, I, LPR_, VPL_>(p, s) : launch_spmm_window<V, I, LPR_, VPL_>(p, s)
  if (kv == 4) TSGU_WIN(4, 1);
  if (kv == 8) TSGU_WIN(TSGU_WIN_LPR8, 8 / TSGU_WIN_LPR8);
  if (kv == 16) TSGU_WIN(8, 2);
#undef TSGU_WIN
  return TSGU_ERR_SHAPE;
}

}  // namespace tsgu

using namespace tsgu;

extern "C" int tsgu_window_limits(int* tile_rows_max, int* entries_max, int* window_rows, int* runs_max) {
  if (tile_rows_max) *tile_rows_max = TSGU_WIN_TMAX;
  if (entries_max) *entries_max = TSGU_WIN_ECAP;
  if (window_rows) *window_rows = TSGU_WIN_ROWS;
  if (runs_max) *runs_max = WIN_RMAX;
  return 0;
}

extern "C" int tsgu_window_plan(const void* rowptr, const void* colind, int64_t batch, int64_t n, int64_t rowptr_bstride,
                                int64_t nnz_bstride, int idx_dtype, int tile_rows, void* lcol_out, void* desc_out,
                                void* stats_out, void* stream) {
  if (batch < 1 || n < 0 || tile_rows < 1 || tile_rows > TSGU_WIN_TMAX) return TSGU_ERR_SHAPE;
  if (!lcol_out || !desc_out || !stats_out) return TSGU_ERR_WORKSPACE;
  cudaStream_t s = as_stream(stream);
  const int64_t tiles_per_item = (n + tile_rows - 1) / tile_rows;
  const int64_t num_tiles = tiles_per_item * batch;
  cudaError_t e = cudaMemsetAsync(stats_out, 0, 4 * sizeof(int32_t), s);
  if (e != cudaSuccess) return (int)e;
  if (num_tiles == 0) return 0;
  int64_t grid = num_tiles < (int64_t)kNumSMs * 8 ? num_tiles : (int64_t)kNumSMs * 8;
  const int plan_smem = WIN_SPAN_WORDS * (4 + 4 + 2);
  TSGU_DISPATCH_IDX(idx_dtype, {
    e = cudaFuncSetAttribute(window_plan_kernel<I>, cudaFuncAttributeMaxDynamicSharedMemorySize, plan_smem);
    if (e != cudaSuccess) return (int)e;
    window_plan_kernel<I><<<(unsigned)grid, 256, plan_smem, s>>>((const I*)rowptr, (const I*)colind, n, rowptr_bstride, nnz_bstride,
                                                         tile_rows, tiles_per_item, num_tiles, TSGU_WIN_ROWS, TSGU_WIN_ECAP,
                                                         (uint16_t*)lcol_out, (int32_t*)desc_out, (int32_t*)stats_out);
    count_launch();
  });
  return launch_status();
}

template <typename V, typename I>
static int window_run(bool sddmm, const void* rowptr, const void* lcol, const void* desc, const void* vals,
                      const void* out_index, const void* G, const void* B, void* out, int64_t batch, int64_t n, int64_t K,
                      int64_t rowptr_bstride, int64_t nnz_bstride, int64_t nnz_len, int tile_rows, int64_t g_bs, int64_t g_rs,
                      int64_t b_bs, int64_t b_rs, int64_t c_bs, int64_t ldc, int64_t c_cs, cudaStream_t s) {
  constexpr int EPV = 16 / (int)sizeof(V);
  WinParams<V, I> p;
  p.rowptr = (const I*)rowptr; p.lcol = (const uint16_t*)lcol; p.desc = (const int32_t*)desc;
  p.vals = (const V*)vals; p.out_index = (const I*)out_index;
  p.G = (const V*)G; p.B = (const V*)B; p.out = (V*)out;
  p.batch = batch; p.n = n; p.rowptr_bstride = rowptr_bstride; p.nnz_bstride = nnz_bstride;
  p.rowptr_len = nnz_bstride > 0 ? batch * rowptr_bstride : batch * n + 1;
  p.nnz_len = nnz_len;
  p.b_bs = b_bs; p.b_rs = b_rs; p.g_bs = g_bs; p.g_rs = g_rs; p.c_bs = c_bs; p.ldc = ldc; p.c_cs = c_cs;
  p.tile_rows = tile_rows;
  p.tiles_per_item = (n + tile_rows - 1) / tile_rows;
  p.num_tiles = p.tiles_per_item * batch;
  const bool ok = (b_rs % EPV) == 0 && (b_bs % EPV) == 0 && aligned16(B) && aligned16(rowptr) && aligned16(lcol) &&
                  aligned16(vals) &&
                  (sddmm ? ((g_rs % EPV) == 0 && (g_bs % EPV) == 0 && aligned16(G))
                         : (c_cs == 1 ? ((ldc % EPV) == 0 && (c_bs % EPV) == 0 && aligned16(out)) : true));
  if (!ok) return TSGU_ERR_SHAPE;
  return window_dispatch<V, I>(p, K, sddmm, s);
}

#define TSGU_WIN_DISPATCH(...)                                                                                         \
  if (idx_dtype != TSGU_I32) return TSGU_ERR_DTYPE; /* window plans exist for 32-bit structures only */               \
  switch (val_dtype) {                                                                                                 \
    case TSGU_F32: { using V = float; using I = int32_t; return __VA_ARGS__; }                                         \
    case TSGU_BF16: { using V = __nv_bfloat16; using I = int32_t; return __VA_ARGS__; }                                \
    default: return TSGU_ERR_DTYPE;                                                                                    \
  }

extern "C" int tsgu_spmm_window(const void* rowptr, const void* lcol, const void* desc, const void* vals,
                                const void* B, void* C, int64_t batch, int64_t n, int64_t K, int64_t rowptr_bstride,
                                int64_t nnz_bstride, int64_t nnz_len, int tile_rows, int64_t b_bs, int64_t b_rs, int64_t c_bs,
                                int64_t ldc, int64_t c_cs, int val_dtype, int idx_dtype, void* stream) {
  if (batch < 0 || n < 0 || K <= 0 || tile_rows < 1 || tile_rows > TSGU_WIN_TMAX) return TSGU_ERR_SHAPE;
  if (batch == 0 || n == 0) return 0;
  TSGU_WIN_DISPATCH(window_run<V, I>(false, rowptr, lcol, desc, vals, nullptr, nullptr, B, C, batch, n, K, rowptr_bstride,
                                     nnz_bstride, nnz_len, tile_rows, 0, 0, b_bs, b_rs, c_bs, ldc, c_cs, as_stream(stream)));
}

extern "C" int tsgu_sddmm_window(const void* rowptr, const void* lcol, const void* desc, const void* out_index, const void* G,
                                 const void* B, void* out, int64_t batch, int64_t n, int64_t K, int64_t rowptr_bstride,
                                 int64_t nnz_bstride, int64_t nnz_len, int tile_rows, int64_t g_bs, int64_t g_rs, int64_t b_bs,
                                 int64_t b_rs, int val_dtype, int idx_dtype, void* stream) {
  if (batch < 0 || n < 0 || K <= 0 || tile_rows < 1 || tile_rows > TSGU_WIN_TMAX) return TSGU_ERR_SHAPE;
  if (batch == 0 || n == 0 || nnz_len == 0) return 0;
  TSGU_WIN_DISPATCH(window_run<V, I>(true, rowptr, lcol, desc, nullptr, out_index, G, B, out, batch, n, K,
                                     rowptr_bstride, nnz_bstride, nnz_len, tile_rows, g_bs, g_rs, b_bs, b_rs, 0, 0, 1,
                                     as_stream(stream)));
}
