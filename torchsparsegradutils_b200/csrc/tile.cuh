// tile.cuh -- persistent row-tile pipeline shared by the SpMM and SDDMM fast paths (sm_100a).
//
// A CTA walks tiles of consecutive rows (tile_rows, chosen per launch by pick_tile_rows).  For every tile the three slices it needs from
// the sparse operand -- rowptr[r0 .. r1], colind[s .. e) and (SpMM) vals[s .. e) -- are contiguous in
// global memory, so one elected thread streams them into shared memory with the bulk async-copy
// engine (cp.async.bulk, SASS UBLKCP) completing on an mbarrier, one tile ahead of the warps that
// consume them.  The only long-latency loads left in the consumers are the dense-row gathers, which is
// what the memory system should be busy with.
#pragma once
#include "common.cuh"

// tunables (overridable at build time for experiments: TSGU_EXTRA_NVCC_FLAGS='-DTSGU_TILE_MINB(VPL)=2 ...')
// (resident CTAs per SM the register allocation aims for, 128-bit dense-row loads in flight per lane
// before the FMA chain) as a function of the vectors per lane; swept on the box: one vector per lane
// (K*s_v <= 128 B, config 3) wants more warps and shorter bursts, four vectors per lane (configs 2, 5)
// the opposite
#ifndef TSGU_TILE_MINB
#define TSGU_TILE_MINB(VPL) ((VPL) == 1 ? 3 : 2)
#endif
#ifndef TSGU_TILE_LOADS
#define TSGU_TILE_LOADS(VPL) ((VPL) == 1 ? 8 : 16)
#endif
#ifndef TSGU_TILE_STAGE_BYTES
#define TSGU_TILE_STAGE_BYTES 36864  // colind + vals bytes staged per tile and stage (36 KB: a 224-row tile of a padded
                                     // transpose fits, so a one-item shard runs ONE wave: 0.1319 -> 0.128 ms per step)
#endif
#ifndef TSGU_TILE_ROWS
#define TSGU_TILE_ROWS 256  // capacity of the staged rowptr slice: most rows a tile may hold
#endif
#ifndef TSGU_TILE_ROWS_DEFAULT
#define TSGU_TILE_ROWS_DEFAULT 128  // rows per tile the launchers ask for unless they pass their own bound (swept:
                                    // 256 helps only the SDDMM with one vector per lane, config 3 0.688 -> 0.650 ms)
#endif

namespace tsgu {

// ------------------------------------------------------------------ mbarrier / bulk copy PTX
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
// global -> shared bulk copy; dst/src 16-B aligned, bytes a multiple of 16
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ------------------------------------------------------------------ tile geometry
// VALS: 0 = pattern only (SDDMM), 1 = values staged (SpMM), 2 = a value permutation staged instead
// (SpMM over a transposed / COO-derived structure: the value of entry e is vals[perm[e]]).
template <typename V, typename I, int VALS>
struct TileCfg {
  static constexpr int TILE_ROWS = TSGU_TILE_ROWS;
  // entries of colind / vals staged per tile: 32 KB per stage (4096 for fp32 + int32)
  static constexpr int CAP = (TSGU_TILE_STAGE_BYTES / (int)(sizeof(I) + (VALS == 1 ? sizeof(V) : VALS == 2 ? sizeof(I) : 0))) & ~15;
  static constexpr int ALN_I = 16 / (int)sizeof(I);
  static constexpr int ALN_V = 16 / (int)sizeof(V);
  static constexpr int STAGES = 2;
  struct Stage {
    alignas(16) I rp[TILE_ROWS + 1 + 2 * ALN_I];
    alignas(16) I col[CAP + 2 * ALN_I];
    alignas(16) V val[VALS == 1 ? CAP + 2 * ALN_V : ALN_V];
    alignas(16) I prm[VALS == 2 ? CAP + 2 * ALN_I : ALN_I];
  };
  struct Smem {
    Stage st[STAGES];
    alignas(8) uint64_t full[STAGES];
  };
};

// rows per tile for a launch: as many as fit the staging capacity with 25 % slack for uneven rows,
// capped by TSGU_TILE_ROWS, and a multiple of the number of lane groups so every group gets whole rows
inline int pick_tile_rows(int64_t total_rows, int64_t nnz_total, int cap_entries, int groups,
                          int max_rows = TSGU_TILE_ROWS_DEFAULT) {
  if (max_rows > TSGU_TILE_ROWS) max_rows = TSGU_TILE_ROWS;
  const double avg = total_rows > 0 ? (double)nnz_total / (double)total_rows : 0.0;
  int64_t r = avg > 0 ? (int64_t)((double)cap_entries / (1.25 * avg)) : max_rows;
  if (r > max_rows) r = max_rows;
  r = r / groups * groups;
  if (r < groups) r = groups < max_rows ? groups : max_rows;
  return (int)r;
}

// Wave quantisation: the persistent kernels hand tiles out round-robin, so every CTA runs floor or ceil(tiles / grid)
// of them, and inside a tile the lane groups take rows in passes of `groups` rows.  A launch with only a few tiles per
// CTA (one rank's share of a strongly scaled batch: 65 536 rows = 512 tiles of 128 rows on 296 CTAs -> 2 waves of 4
// passes where 1.73 waves would do) wastes the difference.  For such launches pick the tile height (a multiple of
// `groups`, within the staging capacity) that minimises waves x passes; e.g. 224 rows -> 293 tiles -> ONE wave of 7
// passes.  Launches with >= 4 waves keep the swept default.  (Simply shrinking tiles until there are many waves was
// measured slower -- 32-row tiles: 0.1455 -> 0.153 ms per step on that shard: the per-tile cost grows.)
inline int balance_tile_rows(int tile_rows, int64_t rows_per_item, int64_t batch, int64_t nnz_total, int cap_entries,
                             int64_t grid, int groups) {
  auto waves = [&](int t) { return (((rows_per_item + t - 1) / t) * batch + grid - 1) / grid; };
  if (grid <= 0 || rows_per_item <= 0 || waves(tile_rows) >= 4) return tile_rows;
  const double avg = (double)nnz_total / (double)(rows_per_item * batch);
  double best_cost = 1e300;
  int best = tile_rows;
  for (int t = groups; t <= TSGU_TILE_ROWS; t += groups) {
    if (t != tile_rows && 1.1 * avg * t > (double)cap_entries) break;  // a tile over the staging capacity falls back to global reads
    const double cost = (double)waves(t) * ((double)((t + groups - 1) / groups) + 0.5);  // + half a pass of fixed cost per tile
    if (cost < best_cost - 1e-9 || (cost < best_cost + 1e-9 && abs(t - tile_rows) < abs(best - tile_rows))) {
      best_cost = cost;
      best = t;
    }
  }
  return best;
}

struct TileCoord {
  int64_t item, r0;
  int rows;  // rows in this tile (<= TILE_ROWS)
};

__device__ __forceinline__ TileCoord tile_coord(int64_t t, int64_t tiles_per_item, int64_t n, int TILE_ROWS) {
  TileCoord c;
  if (tiles_per_item < 0x7fffffffLL && t < 0x7fffffffLL) {  // 32-bit division in the common case
    c.item = (uint32_t)t / (uint32_t)tiles_per_item;
  } else {
    c.item = t / tiles_per_item;
  }
  c.r0 = (t - c.item * tiles_per_item) * TILE_ROWS;
  const int64_t left = n - c.r0;
  c.rows = (int)(left < TILE_ROWS ? left : TILE_ROWS);
  return c;
}

// ------------------------------------------------------------------ producer (one elected thread)
// Streams rowptr[r0..r1], colind[s..e) and (WITH_VALS) vals[s..e) of a tile into a stage so that
// element `lo` of each global array lands at dst[lo % ALN] (bulk copies need 16-B aligned ends).
template <typename V, typename I, int VALS>
struct TileProducer {
  using Cfg = TileCfg<V, I, VALS>;
  const I* rowptr;
  const I* colind;
  const V* vals;
  const I* perm;
  int64_t n, rowptr_bstride, nnz_bstride, tiles_per_item, rowptr_len, nnz_len;
  int tile_rows;

  __device__ __forceinline__ void bounds(int64_t t, int64_t& s_abs, int64_t& e_abs) const {
    const TileCoord c = tile_coord(t, tiles_per_item, n, tile_rows);
    const I* rp = rowptr + c.item * rowptr_bstride + c.r0;
    s_abs = (int64_t)__ldg(rp) + c.item * nnz_bstride;
    e_abs = (int64_t)__ldg(rp + c.rows) + c.item * nnz_bstride;
  }

  template <typename T>
  __device__ __forceinline__ static uint32_t span(T* dst, const T* src, int64_t lo, int64_t hi, int64_t len,
                                                  uint64_t* bar) {
    constexpr int64_t A = 16 / (int64_t)sizeof(T);
    const int64_t lo_al = lo & ~(A - 1);
    int64_t hi_al = (hi + A - 1) & ~(A - 1);
    const int64_t len_dn = len & ~(A - 1);
    if (hi_al > len_dn) {  // the 16-B vector holding the array's ragged end is copied element-wise
      for (int64_t k = (lo > len_dn ? lo : len_dn); k < hi; ++k) dst[k - lo_al] = src[k];
      hi_al = len_dn;
    }
    if (hi_al <= lo_al) return 0u;
    const uint32_t bytes = (uint32_t)((hi_al - lo_al) * (int64_t)sizeof(T));
    bulk_g2s(dst, src + lo_al, bytes, bar);
    return bytes;
  }

  __device__ __forceinline__ void issue(typename Cfg::Stage& st, uint64_t* bar, int64_t t, int64_t s_abs,
                                        int64_t e_abs) const {
    const TileCoord c = tile_coord(t, tiles_per_item, n, tile_rows);
    const int64_t rp_lo = c.item * rowptr_bstride + c.r0;
    uint32_t tx = span<I>(st.rp, rowptr, rp_lo, rp_lo + c.rows + 1, rowptr_len, bar);
    if ((e_abs - s_abs) <= Cfg::CAP && e_abs > s_abs) {
      tx += span<I>(st.col, colind, s_abs, e_abs, nnz_len, bar);
      if constexpr (VALS == 1) tx += span<V>(st.val, vals, s_abs, e_abs, nnz_len, bar);
      if constexpr (VALS == 2) tx += span<I>(st.prm, perm, s_abs, e_abs, nnz_len, bar);
    }
    // arrive.expect_tx after the copies were issued is fine (the phase cannot complete before this
    // arrival) and, having release semantics, it also publishes the element-wise tail stores above
    mbar_expect_tx(bar, tx);
  }
};

// Description of where a tile's slices landed in a stage (every thread recomputes it from the rowptr
// slice in shared memory; nothing but the data itself is communicated).
struct TileView {
  int rp_shift;     // rp[rp_shift + k] = rowptr[r0 + k]
  int64_t s_abs;    // absolute index of the tile's first stored entry
  int64_t e_abs;    // one past its last entry
  int col_shift;    // col[col_shift + (e - s_abs)] = colind[e]
  int val_shift;
  bool staged;      // colind / vals are in shared memory (tile fits CAP); else read them from global
};

}  // namespace tsgu
