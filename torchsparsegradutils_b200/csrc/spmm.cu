// spmm.cu -- CSR SpMM for sm_100a:  C[t] = A[t] * B[t].
//
// Replaces torch.sparse.mm at reference sparse_matmul.py:155 (forward) and :229 (grad_B, with
// the transposed structure from tsgu_csr_transpose).
//
// Three kernel families, chosen in spmm_dispatch():
//   spmm_tile_kernel      persistent row tiles, sparse operand staged by the bulk-copy engine (tile.cuh):
//                         the default whenever the dense operands are 128-bit addressable
//   spmm_merge_kernel     merge-path, nnz-balanced (merge.cu): skewed row lengths, algo = MERGE
//   spmm_rowsplit_kernel  one row per lane group, non-persistent: scalar / strided operands, K > 128
//                         vectors, and problems too small to fill the GPU with tiles
//
// Common mapping: a group of LPR lanes owns one row of A; the lanes tile the dense K dimension with
// 128-bit loads (EPV elements each), VPL vectors per lane, so one B-row fetch is one coalesced request
// per vector slot.  (col, val) pairs are broadcast inside the group with shuffles and U independent
// B-row loads are kept in flight before their FMA chain (latency hiding by ILP; no tensor cores: 2 flop
// per 4-16 B).  Accumulation is in CSR order inside a row (deterministic, no atomics).
#include <type_traits>

#include "common.cuh"
#include "merge.cuh"
#include "tile.cuh"

namespace tsgu {

template <typename V, typename I>
struct SpmmParams {
  const I* rowptr;
  const I* colind;
  const V* vals;
  const I* perm;  // nullable
  const V* B;
  V* C;
  int64_t batch, n, K;
  int64_t rowptr_bstride, nnz_bstride;
  int64_t b_bs, b_rs, b_cs, c_bs, ldc;
  const I* row_map;  // nullable: CSR row s of item t is row row_map[t*n + s] of C[t] (tsgu_spmm_csr_rowmap)
};

// EPV: elements per vector load (1 = scalar path that also honours b_cs != 1)
// LPR: lanes per row (power of two <= 32); VPL: vectors per lane
template <typename V, typename I, int EPV, int LPR, int VPL>
__global__ void __launch_bounds__(256) spmm_rowsplit_kernel(const SpmmParams<V, I> p) {
  using Acc = typename VT<V>::Acc;
  static_assert(EPV == 1 || EPV * sizeof(V) == 16, "vector path is 128-bit");
  constexpr int U = (VPL >= 4) ? 2 : (VPL == 2 ? 4 : 8);  // B-row loads in flight per lane = U*VPL
  constexpr int CHUNK = LPR * VPL * EPV;                   // K elements covered per pass

  const int lane = threadIdx.x & 31;
  const int gl = lane % LPR;
  const unsigned gmask = group_mask<LPR>(lane);
  const int64_t groups_per_block = blockDim.x / LPR;
  const int64_t total_rows = p.batch * p.n;

  for (int64_t r = (int64_t)blockIdx.x * groups_per_block + threadIdx.x / LPR; r < total_rows;
       r += (int64_t)gridDim.x * groups_per_block) {
    const int64_t item = (p.batch == 1) ? 0 : r / p.n;
    const int64_t lr = r - item * p.n;
    const I* rp = p.rowptr + item * p.rowptr_bstride + lr;
    const int64_t e0 = (int64_t)__ldg(rp) + item * p.nnz_bstride;
    const int64_t e1 = (int64_t)__ldg(rp + 1) + item * p.nnz_bstride;
    const V* Bi = p.B + item * p.b_bs;
    V* Crow = p.C + item * p.c_bs + (p.row_map ? (int64_t)p.row_map[r] : lr) * p.ldc;

    for (int64_t k0 = 0; k0 < p.K; k0 += CHUNK) {
      Acc acc[VPL][EPV];
#pragma unroll
      for (int w = 0; w < VPL; ++w)
#pragma unroll
        for (int i = 0; i < EPV; ++i) acc[w][i] = Acc(0);

      for (int64_t base = e0; base < e1; base += LPR) {
        const int64_t e = base + gl;
        const bool ok = e < e1;
        I c = ok ? __ldg(p.colind + e) : I(0);
        Acc v = Acc(0);
        if (ok) v = load_scalar<V>(p.vals + (p.perm ? (int64_t)__ldg(p.perm + e) : e));
        const int cnt = (int)min((int64_t)LPR, e1 - base);
        for (int j0 = 0; j0 < cnt; j0 += U) {
          Raw<V, EPV> b[U][VPL];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int j = j0 + u;
            const int64_t cj = (int64_t)shfl_idx(gmask, c, j, LPR);
            const V* brow = Bi + cj * p.b_rs;
#pragma unroll
            for (int w = 0; w < VPL; ++w) {
              const int64_t kk = k0 + (int64_t)(w * LPR + gl) * EPV;
              if (j < cnt && kk < p.K)
                b[u][w] = raw_ldg<V, EPV>(brow + (EPV == 1 ? kk * p.b_cs : kk));
              else
                b[u][w] = raw_zero<V, EPV>();
            }
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const Acc vj = shfl_idx(gmask, v, j0 + u, LPR);  // lanes >= cnt hold v = 0
#pragma unroll
            for (int w = 0; w < VPL; ++w) {
              Acc x[EPV];
              raw_unpack<V, EPV>(b[u][w], x);
#pragma unroll
              for (int i = 0; i < EPV; ++i) acc[w][i] = fma(vj, x[i], acc[w][i]);
            }
          }
        }
      }
#pragma unroll
      for (int w = 0; w < VPL; ++w) {
        const int64_t kk = k0 + (int64_t)(w * LPR + gl) * EPV;
        if (kk < p.K) store_vec<V, EPV>(Crow + kk, acc[w]);
      }
    }
  }
}

template <typename V, typename I, int EPV, int LPR, int VPL>
static int launch_rowsplit(const SpmmParams<V, I>& p, cudaStream_t s) {
  const int64_t total_rows = p.batch * p.n;
  const int threads = 256;
  const int64_t gpb = threads / LPR;
  int64_t blocks = (total_rows + gpb - 1) / gpb;
  if (blocks > 0x7fffffffLL) blocks = 0x7fffffffLL;
  spmm_rowsplit_kernel<V, I, EPV, LPR, VPL><<<(unsigned)blocks, threads, 0, s>>>(p);
  count_launch();
  return launch_status();
}


// =============================================================================================
// Fast path: persistent row-tile kernel, sparse operand staged by the bulk-copy engine (tile.cuh).
// Requirements (checked by the dispatcher): 128-bit addressable dense operands, no value
// permutation, K <= 32*4 vectors, m < 2^32.
// =============================================================================================
template <typename V, typename I, int LPR, int VPL, int U, bool EXACT, bool PERM>
__global__ void __launch_bounds__(256, TSGU_TILE_MINB(VPL)) spmm_tile_kernel(const SpmmParams<V, I> p, const int64_t tiles_per_item,
                                                        const int64_t num_tiles, const int64_t rowptr_len,
                                                        const int64_t nnz_len, const int tile_rows) {
  using Acc = typename VT<V>::Acc;
  using Cfg = TileCfg<V, I, PERM ? 2 : 1>;
  using Smem = typename Cfg::Smem;
  constexpr int EPV = 16 / sizeof(V);
  constexpr int CAP = Cfg::CAP, AI = Cfg::Stage::AI, AV = Cfg::Stage::AV;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int gl = lane % LPR;
  const unsigned gmask = group_mask<LPR>(lane);
  const int group = tid / LPR;
  constexpr int GROUPS = 256 / LPR;
  const int kv = (int)(p.K / EPV);                      // vectors per dense row
  const uint32_t row_bytes = (uint32_t)(p.b_rs * sizeof(V));  // dense row pitch in bytes (< 4 GiB)
  // lane validity per vector slot (all true when EXACT: K fills LPR*VPL vectors)
  bool on[VPL];
#pragma unroll
  for (int w = 0; w < VPL; ++w) on[w] = EXACT || (w * LPR + gl < kv);

  if (tid == 0) {
    for (int s = 0; s < Cfg::STAGES; ++s) mbar_init(&sm.full[s], 1);
    mbar_fence_init();
  }
  __syncthreads();

  TileProducer<V, I, PERM ? 2 : 1> prod{p.rowptr, p.colind, p.vals, p.perm, p.n, p.rowptr_bstride, p.nnz_bstride,
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
    const V* sval = st.val + (int)(s_abs & (AV - 1));
    const I* sprm = st.prm + (int)(s_abs & (AI - 1));
    // this lane's 16-byte column slice of the item's dense operand
    const char* Bb = reinterpret_cast<const char*>(p.B + c.item * p.b_bs) + (size_t)gl * 16;

    for (int lr = group; lr < c.rows; lr += GROUPS) {
      const int64_t e0 = (int64_t)st.rp[rp_shift + lr] + nnz_off;
      const int64_t e1 = (int64_t)st.rp[rp_shift + lr + 1] + nnz_off;
      Acc acc[VPL][EPV];
#pragma unroll
      for (int w = 0; w < VPL; ++w)
#pragma unroll
        for (int i = 0; i < EPV; ++i) acc[w][i] = Acc(0);

      // a batch is 32 entries: every lane holds Q = 32/LPR (col, val) pairs, broadcast by shuffle;
      // U dense-row gathers (x VPL vectors) are issued back to back before their FMAs
      constexpr int Q = 32 / LPR;
      for (int64_t base = e0; base < e1; base += 32) {
        uint32_t cu[Q];
        Acc v[Q];
#pragma unroll
        for (int q = 0; q < Q; ++q) {
          const int64_t e = base + q * LPR + gl;
          cu[q] = 0;
          v[q] = Acc(0);
          if (e < e1) {
            if (staged) {
              cu[q] = (uint32_t)scol[(int)(e - s_abs)];
              if constexpr (PERM) v[q] = load_scalar<V>(p.vals + (int64_t)sprm[(int)(e - s_abs)]);
              else v[q] = VT<V>::to_acc(sval[(int)(e - s_abs)]);
            } else {
              cu[q] = (uint32_t)__ldg(p.colind + e);
              v[q] = load_scalar<V>(p.vals + (PERM ? (int64_t)__ldg(p.perm + e) : e));
            }
          }
        }
        const int cnt = (int)min((int64_t)32, e1 - base);
#pragma unroll
        for (int j0 = 0; j0 < 32; j0 += U) {
          if (j0 + U <= cnt) {  // full group (group-uniform branch): no predicates on the loads
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
              const Acc vj = shfl_idx(gmask, v[(j0 + u) / LPR], (j0 + u) % LPR, LPR);
#pragma unroll
              for (int w = 0; w < VPL; ++w) {
                Acc x[EPV];
                Raw<V, EPV> raw;
                raw.bits = b[u][w];
                raw_unpack<V, EPV>(raw, x);
#pragma unroll
                for (int i = 0; i < EPV; ++i) acc[w][i] = fma(vj, x[i], acc[w][i]);
              }
            }
          } else if (j0 < cnt) {  // ragged end of the row: same batch, loads predicated
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
              const Acc vj = shfl_idx(gmask, v[(j0 + u) / LPR], (j0 + u) % LPR, LPR);  // 0 past the row end
#pragma unroll
              for (int w = 0; w < VPL; ++w) {
                Acc x[EPV];
                Raw<V, EPV> raw;
                raw.bits = b[u][w];
                raw_unpack<V, EPV>(raw, x);
#pragma unroll
                for (int i = 0; i < EPV; ++i) acc[w][i] = fma(vj, x[i], acc[w][i]);
              }
            }
          }
        }
      }
      int64_t dest = c.r0 + lr;
      if (p.row_map) dest = (int64_t)p.row_map[c.item * p.n + dest];
      V* Crow = p.C + c.item * p.c_bs + dest * p.ldc;
#pragma unroll
      for (int w = 0; w < VPL; ++w)
        if (EXACT || on[w]) store_vec<V, EPV>(Crow + (int64_t)(w * LPR + gl) * EPV, acc[w]);
    }
    __syncthreads();  // everyone is done with this stage before it is refilled
  }
}

template <typename V, typename I, int LPR, int VPL, bool PERM>
static int launch_tile(const SpmmParams<V, I>& p, int64_t nnz_total, cudaStream_t s) {
  using Cfg = TileCfg<V, I, PERM ? 2 : 1>;
  constexpr int U0 = TSGU_TILE_LOADS(VPL) / VPL;  // independent 128-bit loads in flight per lane ...
  constexpr int U = U0 < 32 ? U0 : 32;        // ... (a batch is 32 entries)
  constexpr int EPV = 16 / sizeof(V);
  const bool exact = (p.K / EPV) == (int64_t)LPR * VPL;
  auto kern = exact ? spmm_tile_kernel<V, I, LPR, VPL, U, true, PERM> : spmm_tile_kernel<V, I, LPR, VPL, U, false, PERM>;
  const int smem = (int)sizeof(typename Cfg::Smem);
  static int ctas_per_sm[2] = {0, 0};  // per instantiation; same answer on every B200 of the box
  if (const int rc = persistent_ctas(kern, 256, smem, ctas_per_sm[exact])) return rc;
  const int tile_rows = balance_tile_rows(pick_tile_rows(p.batch * p.n, nnz_total, Cfg::CAP, 256 / LPR), p.n, p.batch,
                                          nnz_total, Cfg::CAP, (int64_t)kNumSMs * ctas_per_sm[exact], 256 / LPR);
  const int64_t tiles_per_item = (p.n + tile_rows - 1) / tile_rows;
  const int64_t num_tiles = tiles_per_item * p.batch;
  const int64_t rowptr_len = p.nnz_bstride > 0 ? p.batch * p.rowptr_bstride : p.batch * p.n + 1;
  return launch_persistent(kern, 256, smem, ctas_per_sm[exact], num_tiles, s, p, tiles_per_item, num_tiles, rowptr_len,
                           nnz_total, tile_rows);
}

template <typename V, typename I>
static int spmm_tile_dispatch(const SpmmParams<V, I>& p, int64_t nnz_total, cudaStream_t s) {
  return with_tile_lanes(p.K / (16 / (int)sizeof(V)), [&](auto LPR, auto VPL) {
    return p.perm ? launch_tile<V, I, LPR, VPL, true>(p, nnz_total, s) : launch_tile<V, I, LPR, VPL, false>(p, nnz_total, s);
  });
}

template <typename V, typename I>
static int spmm_dispatch(const SpmmParams<V, I>& p, int64_t m, int64_t nnz_total, int algo_flags, void* ws, size_t ws_bytes,
                         cudaStream_t s) {
  const int algo = algo_flags & ~TSGU_ALGO_FLAG_KSLICE;
  const bool uniform_rows = (algo_flags & TSGU_ALGO_FLAG_KSLICE) != 0;
  constexpr int EPVF = 16 / sizeof(V);
  const bool vec_ok = p.b_cs == 1 && (p.K % EPVF) == 0 && (p.b_rs % EPVF) == 0 && (p.b_bs % EPVF) == 0 &&
                      (p.ldc % EPVF) == 0 && (p.c_bs % EPVF) == 0 && aligned16(p.B) && aligned16(p.C);
  const bool fast_ok = vec_ok && p.K / EPVF <= 128 && m < 0xffffffffLL && p.b_rs * (int64_t)sizeof(V) < 0xffffffffLL &&
                       aligned16(p.rowptr) && aligned16(p.colind) && aligned16(p.vals) && aligned16(p.perm);
  if (fast_ok && algo == TSGU_ALGO_MERGE && p.batch == 1 && p.ldc == p.K)
    return spmm_merge_dispatch<V, I>(p.rowptr, p.colind, p.vals, p.perm, p.B, p.C, p.n, p.K, nnz_total, p.b_rs, p.ldc, ws,
                                     ws_bytes, s);
  // small problems cannot fill 148 SMs with 64-row tiles: one row per lane group, one CTA per 256/LPR rows
  const bool tiny = p.batch * p.n < tiny_rows_threshold();  // fewer rows than ~64 per resident CTA
  if (fast_ok && algo != TSGU_ALGO_ROWSPLIT && !tiny) {
    // L2 blocking: run K in slices whose dense footprint stays L2-resident (see pick_k_slice)
    const int64_t ks = pick_k_slice(m, p.K, (int)sizeof(V), uniform_rows);
    if (ks < p.K) {
      for (int64_t k0 = 0; k0 < p.K; k0 += ks) {
        SpmmParams<V, I> q = p;
        q.B = p.B + k0;
        q.C = p.C + k0;
        q.K = ks;
        const int rc = spmm_tile_dispatch<V, I>(q, nnz_total, s);
        if (rc) return rc;
      }
      return 0;
    }
    return spmm_tile_dispatch<V, I>(p, nnz_total, s);
  }
  return with_rowsplit_lanes<EPVF>(vec_ok, p.K, [&](auto EPV, auto LPR, auto VPL) { return launch_rowsplit<V, I, EPV, LPR, VPL>(p, s); });
}

}  // namespace tsgu

// the shared body of the two SpMM entry points
static int spmm_csr(const void* rowptr, const void* colind, const void* vals, const void* perm, const void* row_map, const void* B,
                    void* C, int64_t batch, int64_t n, int64_t m, int64_t K, int64_t rowptr_bstride, int64_t nnz_bstride,
                    int64_t nnz_total, int64_t b_bs, int64_t b_rs, int64_t b_cs, int64_t c_bs, int64_t ldc, int val_dtype,
                    int idx_dtype, int algo, void* workspace, size_t workspace_bytes, void* stream) {
  TSGU_DISPATCH_VAL(val_dtype, TSGU_DISPATCH_IDX(idx_dtype, {
    const tsgu::SpmmParams<V, I> p{(const I*)rowptr, (const I*)colind, (const V*)vals, (const I*)perm, (const V*)B, (V*)C,
                                   batch, n, K, rowptr_bstride, nnz_bstride, b_bs, b_rs, b_cs, c_bs, ldc, (const I*)row_map};
    return tsgu::spmm_dispatch<V, I>(p, m, nnz_total, algo, workspace, workspace_bytes, tsgu::as_stream(stream));
  }));
  return 0;
}

extern "C" int tsgu_spmm_csr(const void* rowptr, const void* colind, const void* vals, const void* perm,
                             const void* B, void* C, int64_t batch, int64_t n, int64_t m, int64_t K,
                             int64_t rowptr_bstride, int64_t nnz_bstride, int64_t nnz_total,
                             int64_t b_bs, int64_t b_rs, int64_t b_cs, int64_t c_bs, int64_t ldc,
                             int val_dtype, int idx_dtype, int algo, void* workspace,
                             size_t workspace_bytes, void* stream) {
  if (batch < 0 || n < 0 || K < 0) return TSGU_ERR_SHAPE;
  {
    const int family = algo & ~TSGU_ALGO_FLAG_KSLICE;
    if (family != TSGU_ALGO_AUTO && family != TSGU_ALGO_ROWSPLIT && family != TSGU_ALGO_MERGE) return TSGU_ERR_ALGO;
  }
  if (batch == 0 || n == 0 || K == 0) return 0;
  return spmm_csr(rowptr, colind, vals, perm, nullptr, B, C, batch, n, m, K, rowptr_bstride, nnz_bstride, nnz_total, b_bs,
                  b_rs, b_cs, c_bs, ldc, val_dtype, idx_dtype, algo, workspace, workspace_bytes, stream);
}

extern "C" int tsgu_spmm_csr_rowmap(const void* rowptr, const void* colind, const void* vals, const void* perm,
                                    const void* row_map, const void* B, void* C, int64_t batch, int64_t n, int64_t m,
                                    int64_t K, int64_t rowptr_bstride, int64_t nnz_bstride, int64_t nnz_total, int64_t b_bs,
                                    int64_t b_rs, int64_t b_cs, int64_t c_bs, int64_t ldc, int val_dtype, int idx_dtype,
                                    int algo, void* stream) {
  if (batch < 0 || n < 0 || K < 0) return TSGU_ERR_SHAPE;
  const int family = algo & ~TSGU_ALGO_FLAG_KSLICE;
  if (family != TSGU_ALGO_AUTO && family != TSGU_ALGO_ROWSPLIT) return TSGU_ERR_ALGO;  // merge-path has no row map
  if (batch == 0 || n == 0 || K == 0) return 0;
  return spmm_csr(rowptr, colind, vals, perm, row_map, B, C, batch, n, m, K, rowptr_bstride, nnz_bstride, nnz_total, b_bs,
                  b_rs, b_cs, c_bs, ldc, val_dtype, idx_dtype, algo, nullptr, 0, stream);
}

extern "C" size_t tsgu_spmm_workspace_bytes(int64_t batch, int64_t n, int64_t K, int64_t nnz_total,
                                            int val_dtype, int algo) {
  if ((algo & ~TSGU_ALGO_FLAG_KSLICE) == TSGU_ALGO_MERGE && batch == 1) return tsgu::spmm_merge_workspace_bytes(n, K, nnz_total, val_dtype);
  return 0;
}
