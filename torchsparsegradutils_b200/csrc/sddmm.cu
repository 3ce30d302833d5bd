// sddmm.cu -- fused SDDMM for sm_100a:  out[e] = < G[r_e, :], B[c_e, :] >.
//
// Replaces the reference's un-fused grad_A (sparse_matmul.py:190-205): repeat_interleave row
// expansion + 2x index_select + mul + sum, which materialise 3 nnz x K temporaries.  Here the row
// index is implied by the row-split (never materialised), G[r,:] is held in registers for the whole
// row, each B row is read once with 128-bit loads, and the NB per-entry partial dot products that a
// group of LPR lanes holds are reduced with a halving butterfly: (NB-1) + log2(LPR/NB) shuffles per
// NB entries instead of NB*log2(LPR).
#include "common.cuh"
#include "merge.cuh"
#include "tile.cuh"

namespace tsgu {

template <typename V, typename I>
struct SddmmParams {
  const I* rowptr;
  const I* colind;
  const I* out_index;  // nullable
  const V* G;
  const V* B;
  V* out;
  int64_t batch, n, K;
  int64_t rowptr_bstride, nnz_bstride;
  int64_t g_bs, g_rs, g_cs, b_bs, b_rs, b_cs;
  int accumulate;  // tile kernel: out[dst] += dot (K processed in L2-sized slices)
};

template <typename V, typename I, int EPV, int LPR, int VPL, int NB>
__global__ void __launch_bounds__(256) sddmm_rowsplit_kernel(const SddmmParams<V, I> p) {
  using Acc = typename VT<V>::Acc;
  static_assert(EPV == 1 || EPV * sizeof(V) == 16, "vector path is 128-bit");
  constexpr int CHUNK = LPR * VPL * EPV;
  constexpr int LPE = LPR / NB;  // lanes that end up holding the same entry

  const int lane = threadIdx.x & 31;
  const int gl = lane % LPR;
  const unsigned gmask = group_mask<LPR>(lane);
  const int64_t groups_per_block = blockDim.x / LPR;
  const int64_t total_rows = p.batch * p.n;
  const bool single_chunk = p.K <= CHUNK;

  for (int64_t r = (int64_t)blockIdx.x * groups_per_block + threadIdx.x / LPR; r < total_rows;
       r += (int64_t)gridDim.x * groups_per_block) {
    const int64_t item = (p.batch == 1) ? 0 : r / p.n;
    const int64_t lr = r - item * p.n;
    const I* rp = p.rowptr + item * p.rowptr_bstride + lr;
    const int64_t e0 = (int64_t)__ldg(rp) + item * p.nnz_bstride;
    const int64_t e1 = (int64_t)__ldg(rp + 1) + item * p.nnz_bstride;
    if (e0 >= e1) continue;
    const V* Bi = p.B + item * p.b_bs;
    const V* Grow = p.G + item * p.g_bs + lr * p.g_rs;

    Acc g[VPL][EPV];
    auto load_g = [&](int64_t k0) {
#pragma unroll
      for (int w = 0; w < VPL; ++w) {
        const int64_t kk = k0 + (int64_t)(w * LPR + gl) * EPV;
        Raw<V, EPV> raw = (kk < p.K) ? raw_ldg<V, EPV>(Grow + (EPV == 1 ? kk * p.g_cs : kk)) : raw_zero<V, EPV>();
        raw_unpack<V, EPV>(raw, g[w]);
      }
    };
    if (single_chunk) load_g(0);

    for (int64_t base = e0; base < e1; base += NB) {
      const int64_t e = base + gl;
      I c = (gl < NB && e < e1) ? __ldg(p.colind + e) : I(0);
      const int cnt = (int)min((int64_t)NB, e1 - base);
      Acc part[NB];
#pragma unroll
      for (int j = 0; j < NB; ++j) part[j] = Acc(0);

      for (int64_t k0 = 0; k0 < p.K; k0 += CHUNK) {
        if (!single_chunk) load_g(k0);
#pragma unroll
        for (int j = 0; j < NB; ++j) {
          const int64_t cj = (int64_t)shfl_idx(gmask, c, j, LPR);
          const V* brow = Bi + cj * p.b_rs;
          Raw<V, EPV> b[VPL];
#pragma unroll
          for (int w = 0; w < VPL; ++w) {
            const int64_t kk = k0 + (int64_t)(w * LPR + gl) * EPV;
            b[w] = (j < cnt && kk < p.K) ? raw_ldg<V, EPV>(brow + (EPV == 1 ? kk * p.b_cs : kk))
                                          : raw_zero<V, EPV>();
          }
#pragma unroll
          for (int w = 0; w < VPL; ++w) {
            Acc x[EPV];
            raw_unpack<V, EPV>(b[w], x);
#pragma unroll
            for (int i = 0; i < EPV; ++i) part[j] = fma(g[w][i], x[i], part[j]);
          }
        }
      }
      butterfly_reduce<Acc, LPR, NB>(part, gmask, gl);
      const int slot = gl / LPE;
      if ((gl % LPE) == 0 && slot < cnt) {
        const int64_t eo = base + slot;
        int64_t dst = eo;
        if (p.out_index) dst = (int64_t)__ldg(p.out_index + eo);
        if (dst >= 0) p.out[dst] = VT<V>::from_acc(part[0]);
      }
    }
  }
}

template <typename V, typename I, int EPV, int LPR, int VPL>
static int launch_sddmm(const SddmmParams<V, I>& p, cudaStream_t s) {
  constexpr int NB = LPR < 16 ? LPR : 16;
  const int threads = 256;
  const int64_t gpb = threads / LPR;
  int64_t blocks = (p.batch * p.n + gpb - 1) / gpb;
  if (blocks > 0x7fffffffLL) blocks = 0x7fffffffLL;
  sddmm_rowsplit_kernel<V, I, EPV, LPR, VPL, NB><<<(unsigned)blocks, threads, 0, s>>>(p);
  count_launch();
  return launch_status();
}


// =============================================================================================
// Fast path: persistent row-tile kernel; rowptr / colind staged by the bulk-copy engine (tile.cuh).
// =============================================================================================
template <typename V, typename I, int LPR, int VPL, int NB, int U, bool EXACT>
__global__ void __launch_bounds__(256, TSGU_TILE_MINB(VPL)) sddmm_tile_kernel(const SddmmParams<V, I> p, const int64_t tiles_per_item,
                                                            const int64_t num_tiles, const int64_t rowptr_len,
                                                            const int64_t nnz_len, const int tile_rows) {
  using Acc = typename VT<V>::Acc;
  using Cfg = TileCfg<V, I, 0>;
  using Smem = typename Cfg::Smem;
  constexpr int EPV = 16 / sizeof(V);
  constexpr int CAP = Cfg::CAP, AI = Cfg::Stage::AI;
  constexpr int LPE = NB <= LPR ? LPR / NB : 1;  // lanes holding the same entry after the butterfly
  constexpr int RPL = NB <= LPR ? 1 : NB / LPR;  // results per lane after the butterfly
  constexpr int QC = (NB + LPR - 1) / LPR;       // column indices each lane holds per batch
  static_assert(NB % U == 0, "batch is processed in chunks of U entries");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int gl = lane % LPR;
  const unsigned gmask = group_mask<LPR>(lane);
  const int group = tid / LPR;
  constexpr int GROUPS = 256 / LPR;
  const int kv = (int)(p.K / EPV);
  const uint32_t row_bytes = (uint32_t)(p.b_rs * sizeof(V));
  bool on[VPL];
#pragma unroll
  for (int w = 0; w < VPL; ++w) on[w] = EXACT || (w * LPR + gl < kv);

  if (tid == 0) {
    for (int s = 0; s < Cfg::STAGES; ++s) mbar_init(&sm.full[s], 1);
    mbar_fence_init();
  }
  __syncthreads();

  TileProducer<V, I, 0> prod{p.rowptr, p.colind, nullptr, nullptr, p.n, p.rowptr_bstride, p.nnz_bstride,
                             tiles_per_item, rowptr_len, nnz_len, tile_rows};
  int64_t nxt_s = 0, nxt_e = 0;
  const int64_t t0 = blockIdx.x;
  if (tid == 0 && t0 < num_tiles) {
    int64_t s0, e0;
    prod.bounds(t0, s0, e0);
    prod.issue(sm.st[0], &sm.full[0], t0, s0, e0);
    if (t0 + gridDim.x < num_tiles) prod.bounds(t0 + gridDim.x, nxt_s, nxt_e);
  }

  int it = 0;
  for (int64_t t = t0; t < num_tiles; t += gridDim.x, ++it) {
    const int stage = it & 1;
    if (tid == 0) {
      const int64_t tn = t + gridDim.x;
      if (tn < num_tiles) {
        prod.issue(sm.st[stage ^ 1], &sm.full[stage ^ 1], tn, nxt_s, nxt_e);
        if (tn + gridDim.x < num_tiles) prod.bounds(tn + gridDim.x, nxt_s, nxt_e);
      }
    }
    mbar_wait(&sm.full[stage], (uint32_t)((it >> 1) & 1));

    const TileCoord c = tile_coord(t, tiles_per_item, p.n, tile_rows);
    const auto& st = sm.st[stage];
    const int rp_shift = (int)((c.item * p.rowptr_bstride + c.r0) & (AI - 1));
    const int64_t nnz_off = c.item * p.nnz_bstride;
    const int64_t s_abs = (int64_t)st.rp[rp_shift] + nnz_off;
    const int64_t e_abs = (int64_t)st.rp[rp_shift + c.rows] + nnz_off;
    const bool staged = (e_abs - s_abs) <= CAP && e_abs > s_abs;
    const I* scol = st.col + (int)(s_abs & (AI - 1));
    const char* Bb = reinterpret_cast<const char*>(p.B + c.item * p.b_bs) + (size_t)gl * 16;

    for (int lr = group; lr < c.rows; lr += GROUPS) {
      const int64_t e0 = (int64_t)st.rp[rp_shift + lr] + nnz_off;
      const int64_t e1 = (int64_t)st.rp[rp_shift + lr + 1] + nnz_off;
      if (e0 >= e1) continue;
      // the row of the upstream gradient stays in registers for the whole row of A
      Acc g[VPL][EPV];
      const V* Grow = p.G + c.item * p.g_bs + (int64_t)(c.r0 + lr) * p.g_rs;
#pragma unroll
      for (int w = 0; w < VPL; ++w) {
        Raw<V, EPV> raw = (EXACT || on[w]) ? raw_ldg<V, EPV>(Grow + (int64_t)(w * LPR + gl) * EPV) : raw_zero<V, EPV>();
        raw_unpack<V, EPV>(raw, g[w]);
      }

      for (int64_t base = e0; base < e1; base += NB) {
        uint32_t cu[QC];
#pragma unroll
        for (int q = 0; q < QC; ++q) {
          const int64_t e = base + q * LPR + gl;
          cu[q] = 0;
          if (q * LPR + gl < NB && e < e1) cu[q] = staged ? (uint32_t)scol[(int)(e - s_abs)] : (uint32_t)__ldg(p.colind + e);
        }
        const int cnt = (int)min((int64_t)NB, e1 - base);
        Acc part[NB];
#pragma unroll
        for (int j = 0; j < NB; ++j) part[j] = Acc(0);

#pragma unroll
        for (int j0 = 0; j0 < NB; j0 += U) {
          if (j0 + U <= cnt) {  // full group (group-uniform branch): unpredicated gathers
            uint4 b[U][VPL];
#pragma unroll
            for (int u = 0; u < U; ++u) {
              const uint32_t cj = shfl_idx(gmask, cu[(j0 + u) / LPR], (j0 + u) % LPR, LPR);
              const char* brow = Bb + (uint64_t)cj * row_bytes;
#pragma unroll
              for (int w = 0; w < VPL; ++w) {
                if (EXACT || on[w]) b[u][w] = __ldg(reinterpret_cast<const uint4*>(brow + w * (LPR * 16)));
                else b[u][w] = make_uint4(0, 0, 0, 0);
              }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
#pragma unroll
              for (int w = 0; w < VPL; ++w) {
                Acc x[EPV];
                Raw<V, EPV> raw;
                raw.bits = b[u][w];
                raw_unpack<V, EPV>(raw, x);
#pragma unroll
                for (int i = 0; i < EPV; ++i) part[j0 + u] = fma(g[w][i], x[i], part[j0 + u]);
              }
            }
          } else if (j0 < cnt) {  // ragged end of the row
            uint4 b[U][VPL];
#pragma unroll
            for (int u = 0; u < U; ++u) {
              const uint32_t cj = shfl_idx(gmask, cu[(j0 + u) / LPR], (j0 + u) % LPR, LPR);
              const char* brow = Bb + (uint64_t)cj * row_bytes;
#pragma unroll
              for (int w = 0; w < VPL; ++w) {
                if (j0 + u < cnt && (EXACT || on[w])) b[u][w] = __ldg(reinterpret_cast<const uint4*>(brow + w * (LPR * 16)));
                else b[u][w] = make_uint4(0, 0, 0, 0);
              }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
#pragma unroll
              for (int w = 0; w < VPL; ++w) {
                Acc x[EPV];
                Raw<V, EPV> raw;
                raw.bits = b[u][w];
                raw_unpack<V, EPV>(raw, x);
#pragma unroll
                for (int i = 0; i < EPV; ++i) part[j0 + u] = fma(g[w][i], x[i], part[j0 + u]);
              }
            }
          }
        }
        butterfly_reduce<Acc, LPR, NB>(part, gmask, gl);
        if ((gl % LPE) == 0) {
#pragma unroll
          for (int i = 0; i < RPL; ++i) {
            const int slot = (gl / LPE) * RPL + i;
            if (slot < cnt) {
              const int64_t eo = base + slot;
              int64_t dst = eo;
              if (p.out_index) dst = (int64_t)__ldg(p.out_index + eo);
              if (dst >= 0) {
                Acc r = part[i];
                if (p.accumulate) r += VT<V>::to_acc(p.out[dst]);
                p.out[dst] = VT<V>::from_acc(r);
              }
            }
          }
        }
      }
    }
    __syncthreads();
  }
}

template <typename V, typename I, int LPR, int VPL>
static int launch_sddmm_tile(const SddmmParams<V, I>& p, int64_t nnz_total, cudaStream_t s) {
  using Cfg = TileCfg<V, I, 0>;
#ifndef TSGU_SDDMM_NB
#define TSGU_SDDMM_NB 8   // swept on the box: 8 -> no spills at the 128-register cap (config 2 SDDMM 0.282 -> 0.264 ms), 16: 24 B of spills, 32: 0.325 ms
#endif
  constexpr int NB = TSGU_SDDMM_NB;  // entries per batch (butterfly leaves NB/LPR results per lane when NB > LPR)
  constexpr int U0 = TSGU_TILE_LOADS(VPL) / VPL;
  constexpr int U = U0 < NB ? U0 : NB;
  constexpr int EPV = 16 / sizeof(V);
  const bool exact = (p.K / EPV) == (int64_t)LPR * VPL;
  auto kern = exact ? sddmm_tile_kernel<V, I, LPR, VPL, NB, U, true> : sddmm_tile_kernel<V, I, LPR, VPL, NB, U, false>;
  const int smem = (int)sizeof(typename Cfg::Smem);
  static int ctas_per_sm[2] = {0, 0};
  if (const int rc = persistent_ctas(kern, 256, smem, ctas_per_sm[exact])) return rc;
  const int tile_rows = balance_tile_rows(
      pick_tile_rows(p.batch * p.n, nnz_total, Cfg::CAP, 256 / LPR, VPL == 1 ? 256 : TSGU_TILE_ROWS_DEFAULT), p.n, p.batch,
      nnz_total, Cfg::CAP, (int64_t)kNumSMs * ctas_per_sm[exact], 256 / LPR);
  const int64_t tiles_per_item = (p.n + tile_rows - 1) / tile_rows;
  const int64_t num_tiles = tiles_per_item * p.batch;
  const int64_t rowptr_len = p.nnz_bstride > 0 ? p.batch * p.rowptr_bstride : p.batch * p.n + 1;
  return launch_persistent(kern, 256, smem, ctas_per_sm[exact], num_tiles, s, p, tiles_per_item, num_tiles, rowptr_len,
                           nnz_total, tile_rows);
}

template <typename V, typename I>
static int sddmm_tile_dispatch(const SddmmParams<V, I>& p, int64_t nnz_total, cudaStream_t s) {
  return with_tile_lanes(p.K / (16 / (int)sizeof(V)),
                         [&](auto LPR, auto VPL) { return launch_sddmm_tile<V, I, LPR, VPL>(p, nnz_total, s); });
}

template <typename V, typename I>
static int sddmm_dispatch(const SddmmParams<V, I>& p, int64_t m, int64_t nnz_total, int algo, void* ws, size_t ws_bytes,
                          cudaStream_t s) {
  constexpr int EPVF = 16 / sizeof(V);
  const bool vec_ok = p.b_cs == 1 && p.g_cs == 1 && (p.K % EPVF) == 0 && (p.b_rs % EPVF) == 0 &&
                      (p.b_bs % EPVF) == 0 && (p.g_rs % EPVF) == 0 && (p.g_bs % EPVF) == 0 &&
                      aligned16(p.B) && aligned16(p.G);
  const bool fast_ok = vec_ok && p.K / EPVF <= 128 && m < 0xffffffffLL && p.b_rs * (int64_t)sizeof(V) < 0xffffffffLL &&
                       aligned16(p.rowptr) && aligned16(p.colind);
  if (fast_ok && algo == TSGU_ALGO_MERGE && p.batch == 1)
    return sddmm_merge_dispatch<V, I>(p.rowptr, p.colind, p.out_index, p.G, p.B, p.out, p.n, p.K, nnz_total, p.g_rs, p.b_rs,
                                      ws, ws_bytes, s);
  const bool tiny = p.batch * p.n < tiny_rows_threshold();  // fewer rows than ~64 per resident CTA
  if (fast_ok && algo != TSGU_ALGO_ROWSPLIT && !tiny) {
    // L2 blocking (see pick_k_slice): partial dots of the K slices are accumulated into `out`
    const int64_t ks = pick_k_slice(m, p.K, (int)sizeof(V));
    if (ks < p.K && sizeof(V) >= 4) {  // bf16 would round the running sum at every slice: not sliced
      for (int64_t k0 = 0; k0 < p.K; k0 += ks) {
        SddmmParams<V, I> q = p;
        q.B = p.B + k0;
        q.G = p.G + k0;
        q.K = ks;
        q.accumulate = k0 > 0;
        const int rc = sddmm_tile_dispatch<V, I>(q, nnz_total, s);
        if (rc) return rc;
      }
      return 0;
    }
    return sddmm_tile_dispatch<V, I>(p, nnz_total, s);
  }
  return with_rowsplit_lanes<EPVF>(vec_ok, p.K, [&](auto EPV, auto LPR, auto VPL) { return launch_sddmm<V, I, EPV, LPR, VPL>(p, s); });
}

// ---------------------------------------------------------------------------------------------
// COO variant: entries are independent; a group of LPR lanes handles NB consecutive entries.
// ---------------------------------------------------------------------------------------------
template <typename V, int EPV, int LPR, int NB>
__global__ void __launch_bounds__(256) sddmm_coo_kernel(const int64_t* __restrict__ row,
                                                        const int64_t* __restrict__ col,
                                                        const V* __restrict__ G, const V* __restrict__ B,
                                                        V* __restrict__ out, int64_t nnz, int64_t K,
                                                        int64_t g_rs, int64_t g_cs, int64_t b_rs, int64_t b_cs) {
  using Acc = typename VT<V>::Acc;
  constexpr int CHUNK = LPR * EPV;
  constexpr int LPE = LPR / NB;
  const int lane = threadIdx.x & 31;
  const int gl = lane % LPR;
  const unsigned gmask = group_mask<LPR>(lane);
  const int64_t groups_per_block = blockDim.x / LPR;
  const int64_t ngroups = (nnz + NB - 1) / NB;
  for (int64_t grp = (int64_t)blockIdx.x * groups_per_block + threadIdx.x / LPR; grp < ngroups;
       grp += (int64_t)gridDim.x * groups_per_block) {
    const int64_t base = grp * NB;
    const int64_t e = base + gl;
    const bool ok = gl < NB && e < nnz;
    int64_t r = ok ? __ldg(row + e) : 0;
    int64_t c = ok ? __ldg(col + e) : 0;
    const int cnt = (int)min((int64_t)NB, nnz - base);
    Acc part[NB];
#pragma unroll
    for (int j = 0; j < NB; ++j) part[j] = Acc(0);
    for (int64_t k0 = 0; k0 < K; k0 += CHUNK) {
      const int64_t kk = k0 + (int64_t)gl * EPV;
#pragma unroll
      for (int j = 0; j < NB; ++j) {
        const int64_t rj = shfl_idx(gmask, r, j, LPR);
        const int64_t cj = shfl_idx(gmask, c, j, LPR);
        Raw<V, EPV> gr = raw_zero<V, EPV>(), br = raw_zero<V, EPV>();
        if (j < cnt && kk < K) {
          gr = raw_ldg<V, EPV>(G + rj * g_rs + (EPV == 1 ? kk * g_cs : kk));
          br = raw_ldg<V, EPV>(B + cj * b_rs + (EPV == 1 ? kk * b_cs : kk));
        }
        Acc x[EPV], y[EPV];
        raw_unpack<V, EPV>(gr, x);
        raw_unpack<V, EPV>(br, y);
#pragma unroll
        for (int i = 0; i < EPV; ++i) part[j] = fma(x[i], y[i], part[j]);
      }
    }
    butterfly_reduce<Acc, LPR, NB>(part, gmask, gl);
    const int slot = gl / LPE;
    if ((gl % LPE) == 0 && slot < cnt) out[base + slot] = VT<V>::from_acc(part[0]);
  }
}

template <typename V, int EPV, int LPR>
static int launch_sddmm_coo(const int64_t* row, const int64_t* col, const V* G, const V* B, V* out,
                            int64_t nnz, int64_t K, int64_t g_rs, int64_t g_cs, int64_t b_rs,
                            int64_t b_cs, cudaStream_t s) {
  constexpr int NB = LPR < 8 ? LPR : 8;
  const int threads = 256;
  const int64_t gpb = threads / LPR;
  const int64_t ngroups = (nnz + NB - 1) / NB;
  int64_t blocks = (ngroups + gpb - 1) / gpb;
  if (blocks > 0x7fffffffLL) blocks = 0x7fffffffLL;
  sddmm_coo_kernel<V, EPV, LPR, NB><<<(unsigned)blocks, threads, 0, s>>>(row, col, G, B, out, nnz, K, g_rs,
                                                                        g_cs, b_rs, b_cs);
  count_launch();
  return launch_status();
}

}  // namespace tsgu

extern "C" int tsgu_sddmm_csr(const void* rowptr, const void* colind, const void* out_index, const void* G,
                              const void* B, void* out, int64_t batch, int64_t n, int64_t m, int64_t K,
                              int64_t rowptr_bstride, int64_t nnz_bstride, int64_t nnz_total, int64_t g_bs,
                              int64_t g_rs, int64_t g_cs, int64_t b_bs, int64_t b_rs, int64_t b_cs,
                              int val_dtype, int idx_dtype, int algo, void* workspace, size_t workspace_bytes,
                              void* stream) {
  if (batch < 0 || n < 0 || K < 0) return TSGU_ERR_SHAPE;
  if (algo != TSGU_ALGO_AUTO && algo != TSGU_ALGO_ROWSPLIT && algo != TSGU_ALGO_MERGE) return TSGU_ERR_ALGO;
  if (batch == 0 || n == 0 || nnz_total == 0) return 0;
  TSGU_DISPATCH_VAL(val_dtype, TSGU_DISPATCH_IDX(idx_dtype, {
    tsgu::SddmmParams<V, I> p;
    p.rowptr = (const I*)rowptr; p.colind = (const I*)colind; p.out_index = (const I*)out_index;
    p.G = (const V*)G; p.B = (const V*)B; p.out = (V*)out;
    p.batch = batch; p.n = n; p.K = K;
    p.rowptr_bstride = rowptr_bstride; p.nnz_bstride = nnz_bstride;
    p.g_bs = g_bs; p.g_rs = g_rs; p.g_cs = g_cs; p.b_bs = b_bs; p.b_rs = b_rs; p.b_cs = b_cs;
    p.accumulate = 0;
    return tsgu::sddmm_dispatch<V, I>(p, m, nnz_total, algo, workspace, workspace_bytes, tsgu::as_stream(stream));
  }));
  return 0;
}

extern "C" size_t tsgu_sddmm_workspace_bytes(int64_t batch, int64_t n, int64_t nnz_total, int algo) {
  if (algo == TSGU_ALGO_MERGE && batch == 1) return tsgu::sddmm_merge_workspace_bytes(n, nnz_total);
  return 0;
}

extern "C" int tsgu_sddmm_coo(const int64_t* row, const int64_t* col, const void* G, const void* B, void* out,
                              int64_t nnz, int64_t K, int64_t g_rs, int64_t g_cs, int64_t b_rs, int64_t b_cs,
                              int val_dtype, void* stream) {
  if (nnz < 0 || K < 0) return TSGU_ERR_SHAPE;
  if (nnz == 0) return 0;
  cudaStream_t s = tsgu::as_stream(stream);
  TSGU_DISPATCH_VAL(val_dtype, {
    constexpr int EPVF = 16 / sizeof(V);
    const V* g = (const V*)G; const V* b = (const V*)B; V* o = (V*)out;
    const bool vec_ok = g_cs == 1 && b_cs == 1 && (K % EPVF) == 0 && (g_rs % EPVF) == 0 && (b_rs % EPVF) == 0 &&
                        tsgu::aligned16(G) && tsgu::aligned16(B);
    if (vec_ok) {
      const int64_t kv = K / EPVF;
      if (kv <= 8) return tsgu::launch_sddmm_coo<V, EPVF, 8>(row, col, g, b, o, nnz, K, g_rs, g_cs, b_rs, b_cs, s);
      return tsgu::launch_sddmm_coo<V, EPVF, 32>(row, col, g, b, o, nnz, K, g_rs, g_cs, b_rs, b_cs, s);
    }
    if (K <= 4) return tsgu::launch_sddmm_coo<V, 1, 4>(row, col, g, b, o, nnz, K, g_rs, g_cs, b_rs, b_cs, s);
    return tsgu::launch_sddmm_coo<V, 1, 32>(row, col, g, b, o, nnz, K, g_rs, g_cs, b_rs, b_cs, s);
  });
  return 0;
}
