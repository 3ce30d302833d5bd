/*
 * tsgu_b200.h -- C ABI of the B200-native sparse_mm hot path.
 *
 * Drop-in boundary for cai4cai/torchsparsegradutils' `sparse_mm` (reference
 * torchsparsegradutils/sparse_matmul.py:8-234).  The reference has no FFI of its
 * own: its boundary is the Python function `sparse_mm` + `SparseMatMul.apply`
 * (sparse_matmul.py:129,132) whose arithmetic is delegated to torch ATen.  Each
 * entry point below replaces one of those ATen call sites; the citation on each
 * declaration names it.  INTEGRATION.md shows the ctypes binding a maintainer of
 * the reference would add.
 *
 * Conventions
 *   - Plain pointers and sizes only; no torch types.  All pointers are DEVICE
 *     pointers on the current CUDA device; `stream` is a cudaStream_t passed as
 *     void*.  Every call is asynchronous on `stream`; nothing synchronises.
 *   - The caller owns every buffer (inputs, outputs, workspace).  The library
 *     never allocates, frees or retains pointers past return.
 *   - Return value: 0 = OK; > 0 = a cudaError_t from launch; < 0 = argument
 *     error (TSGU_ERR_*).  tsgu_error_string() decodes both ranges.
 *   - Strides are in ELEMENTS.  Dense operands are addressed as
 *       X[item, r, k] = X + item*bs + r*rs + k*cs.
 *   - Sparse operands are "CSR batches":
 *       row r of item t spans entries [ rowptr[t*rowptr_bstride + r]     + t*nnz_bstride,
 *                                       rowptr[t*rowptr_bstride + r + 1] + t*nnz_bstride )
 *     of colind / vals.  torch batched CSR (crow (b,n+1), col (b,nnz)) is
 *     rowptr_bstride = n+1, nnz_bstride = nnz; one flat CSR over batch*n rows
 *     (what the COO->CSR and transpose builders emit) is rowptr_bstride = n,
 *     nnz_bstride = 0.  Column indices are local to the item (0 <= col < m).
 *   - Re-entrant and thread-safe; no static per-process device.
 */
#ifndef TSGU_B200_H
#define TSGU_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TSGU_ABI_VERSION 2

#if defined(__GNUC__)
#define TSGU_API __attribute__((visibility("default")))
#else
#define TSGU_API
#endif

/* value dtypes */
enum { TSGU_F32 = 0, TSGU_F64 = 1, TSGU_BF16 = 2 };
/* index dtypes */
enum { TSGU_I32 = 0, TSGU_I64 = 1 };
/* kernel selection (AUTO: nnz-imbalance heuristic done by the caller; see DESIGN.md) */
enum { TSGU_ALGO_AUTO = 0, TSGU_ALGO_ROWSPLIT = 1, TSGU_ALGO_MERGE = 2 };
/* hint OR-ed into `algo` of tsgu_spmm_csr: the rows of this pattern have (near-)uniform length, so when one item
 * of the dense operand exceeds L2 the K dimension may be processed in L2-resident slices (same results: the
 * slices are independent columns of C).  Ignored by every other entry point. */
#define TSGU_ALGO_FLAG_KSLICE 0x100
/* argument errors */
enum {
  TSGU_ERR_DTYPE = -1,      /* unknown value / index dtype enum              */
  TSGU_ERR_SHAPE = -2,      /* negative size, K <= 0 with rows > 0, ...      */
  TSGU_ERR_WORKSPACE = -3,  /* workspace pointer null or too small           */
  TSGU_ERR_ALGO = -4,       /* unknown algo enum                             */
  TSGU_ERR_RANGE = -5       /* sizes do not fit the requested index dtype    */
};

TSGU_API int tsgu_version(void);
TSGU_API const char* tsgu_error_string(int code);
/* Number of kernels this library has launched in the calling process (monotonic;
 * bench.py reports the delta over the timed region as `gpu_launches`). */
TSGU_API int64_t tsgu_launch_count(void);
/* SMs the persistent kernels launched from the CALLING THREAD leave free from now on (0 = use all 148); returns the
 * previous value.  Used while a collective must run concurrently with a kernel of this library (row-sharded
 * grad_B reduction overlapped with the SDDMM, SURVEY 8(e)): a persistent grid that owns every SM would otherwise
 * keep NCCL's kernels waiting until it drains. */
TSGU_API int tsgu_set_sm_margin(int sms);
/* Host mailbox: `bytes` of mapped pinned host memory (host_ptr for the host to read, dev_ptr for kernels to write) and
 * tsgu_publish(), a one-block kernel that stores `bytes` (multiple of 4) of device memory `src` into a mailbox on
 * `stream`.  Synchronise the stream, then read host_ptr.  This is how the host side learns the few scalars a new
 * sparsity pattern produces (longest row, window-plan verdict, padded size).  Replaces the `.item()` / `int(tensor)`
 * host reads of the reference's index plumbing (utils/utils.py:766-767 in sparse_block_diag_split, and the nnz / shape
 * reads inside the torch.sparse.mm calls of sparse_matmul.py:155 and :229): unlike a cudaMemcpy the store does not queue
 * behind bulk D2H transfers on the copy engines. */
TSGU_API int tsgu_mailbox_create(size_t bytes, void** host_ptr, void** dev_ptr);
TSGU_API int tsgu_mailbox_destroy(void* host_ptr);
TSGU_API int tsgu_publish(const void* src, void* mailbox_dev, size_t bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * SpMM:  C[t] = A[t] * B[t]                 replaces torch.sparse.mm(A, B)
 *   forward   sparse_matmul.py:155   (A in CSR, or COO via tsgu_coo_to_csr + perm)
 *   grad_B    sparse_matmul.py:229   (A^T via tsgu_csr_transpose: rowptrT/colindT + perm)
 * `perm` (nullable, idx_dtype): value of stored entry e is vals[perm[e]] instead of vals[e].
 * C is written row-major: C[t, r, k] = C + t*c_bs + r*ldc + k; every row is written (empty
 * rows get zeros), so C needs no initialisation.
 * algo: AUTO / ROWSPLIT pick the row-split kernels (persistent bulk-copy-staged tiles when the
 * operands are 128-bit addressable); MERGE (batch = 1 only, else ignored) the nnz-balanced merge-path
 * kernel for skewed row lengths.  Workspace: tsgu_spmm_workspace_bytes() (0 unless algo = MERGE).
 * ---------------------------------------------------------------------------------- */
TSGU_API int tsgu_spmm_csr(const void* rowptr, const void* colind, const void* vals, const void* perm,
                  const void* B, void* C,
                  int64_t batch, int64_t n, int64_t m, int64_t K,
                  int64_t rowptr_bstride, int64_t nnz_bstride, int64_t nnz_total,
                  int64_t b_bs, int64_t b_rs, int64_t b_cs,
                  int64_t c_bs, int64_t ldc,
                  int val_dtype, int idx_dtype, int algo,
                  void* workspace, size_t workspace_bytes, void* stream);
/* Same product over a structure whose rows were PERMUTED (the cached transpose keeps its rows sorted by length so that
 * the rows a warp works on together are equally long): CSR row s of item t is row row_map[t*n + s] of C[t]
 * (idx_dtype, a permutation of 0..n-1 per item).  Row-tile and row-split kernels only (algo AUTO / ROWSPLIT). */
TSGU_API int tsgu_spmm_csr_rowmap(const void* rowptr, const void* colind, const void* vals, const void* perm,
                         const void* row_map, const void* B, void* C, int64_t batch, int64_t n, int64_t m, int64_t K,
                         int64_t rowptr_bstride, int64_t nnz_bstride, int64_t nnz_total, int64_t b_bs, int64_t b_rs,
                         int64_t b_cs, int64_t c_bs, int64_t ldc, int val_dtype, int idx_dtype, int algo, void* stream);

TSGU_API size_t tsgu_spmm_workspace_bytes(int64_t batch, int64_t n, int64_t K, int64_t nnz_total,
                                 int val_dtype, int algo);

/* ------------------------------------------------------------------------------------
 * SDDMM:  out[dst(e)] = < G[t, r_e, :], B[t, c_e, :] >     for every stored entry e
 *   replaces index_select x2 + mul + sum, sparse_matmul.py:201-205, and the row expansion
 *   repeat_interleave(arange(n), diff(crow)) of sparse_matmul.py:190-192 (never materialised).
 * `out_index` (nullable, idx_dtype): dst(e) = out_index[e], entries with out_index[e] < 0 are
 * skipped (used to write COO gradients back in A's storage order); null: dst(e) = e.
 * Workspace: tsgu_sddmm_workspace_bytes() (0 unless algo = MERGE).
 * ---------------------------------------------------------------------------------- */
TSGU_API int tsgu_sddmm_csr(const void* rowptr, const void* colind, const void* out_index,
                   const void* G, const void* B, void* out,
                   int64_t batch, int64_t n, int64_t m, int64_t K,
                   int64_t rowptr_bstride, int64_t nnz_bstride, int64_t nnz_total,
                   int64_t g_bs, int64_t g_rs, int64_t g_cs,
                   int64_t b_bs, int64_t b_rs, int64_t b_cs,
                   int val_dtype, int idx_dtype, int algo,
                   void* workspace, size_t workspace_bytes, void* stream);
TSGU_API size_t tsgu_sddmm_workspace_bytes(int64_t batch, int64_t n, int64_t nnz_total, int algo);

/* Order-agnostic COO variant: row/col are int64 arrays of length nnz (torch COO indices,
 * sparse_matmul.py:184-185); out[e] = <G[row[e],:], B[col[e],:]>.  Also the kernel the
 * solve/lstsq backwards would reuse (sparse_solve.py:216-235, sparse_lstsq.py:239-256). */
TSGU_API int tsgu_sddmm_coo(const int64_t* row, const int64_t* col, const void* G, const void* B, void* out,
                   int64_t nnz, int64_t K,
                   int64_t g_rs, int64_t g_cs, int64_t b_rs, int64_t b_cs,
                   int val_dtype, void* stream);

/* ------------------------------------------------------------------------------------
 * Index builders (bit-exact integer work).
 * ---------------------------------------------------------------------------------- */

/* Stable lexicographic sort of COO coordinates; replaces torch.unique(sorted)+argsort,
 * utils/utils.py:148-149 (_sort_coo_indices).  idx is int64 (ndim, nnz) with row stride idx_ld;
 * dims[d] is the extent of coordinate d (ndim = 2: row,col; 3: batch,row,col).
 * key_dims <= ndim: only the leading key_dims coordinates form the key (ndim-1 = sort by
 * (batch,)row only, keeping storage order inside a row).  Outputs: perm (perm_dtype; position in
 * the input of the k-th sorted entry) and, if non-null, sorted_idx (int64, (ndim, nnz), ld nnz). */
TSGU_API int tsgu_coo_sort(const int64_t* idx, int ndim, int64_t nnz, int64_t idx_ld, const int64_t* dims,
                  int key_dims, int64_t* sorted_idx, void* perm, int perm_dtype,
                  void* workspace, size_t workspace_bytes, void* stream);
TSGU_API size_t tsgu_coo_sort_workspace_bytes(int ndim, int64_t nnz, int perm_dtype);

/* COO (already sorted, or sorted through `perm`) -> flat CSR over batch*n rows; replaces
 * bincount+cumsum (utils/utils.py:228-231) and the per-batch Python loop of
 * convert_coo_to_csr_indices_values (utils/utils.py:327-344).  rowptr_out has batch*n+1 entries
 * (absolute offsets), colind_out[k] is the item-local column of the k-th sorted entry. */
TSGU_API int tsgu_coo_to_csr(const int64_t* idx, int ndim, int64_t nnz, int64_t idx_ld,
                    int64_t batch, int64_t n, const void* perm,
                    void* rowptr_out, void* colind_out, int out_idx_dtype, void* stream);

/* Histogram + scan: row indices (any order) -> crow; replaces _compress_row_indices
 * (utils/utils.py:152-233).  Output dtype = input dtype. */
TSGU_API int tsgu_compress_rows(const void* rows, int64_t nnz, int64_t n, void* crow_out, int idx_dtype,
                       void* workspace, size_t workspace_bytes, void* stream);
TSGU_API size_t tsgu_compress_rows_workspace_bytes(int64_t n, int idx_dtype);

/* crow -> per-entry row index; replaces _demcompress_crow_indices (utils/utils.py:413-470). */
TSGU_API int tsgu_decompress_crow(const void* crow, int64_t n, int64_t nnz, void* rows_out, int idx_dtype,
                         void* stream);

/* CSR batch -> CSR of the transposes, as one flat CSR over batch*m rows: rowptrT (batch*m+1,
 * absolute), colindT (item-local row of A), permT (absolute position of the entry in A's
 * colind/vals storage).  Stable (ties keep A's storage order), so for duplicate-free input it is
 * the unique answer A.t().to_sparse_csr() gives.  No reference function exists: the transpose is
 * implicit in A.t() at sparse_matmul.py:229 and redone by ATen on every backward. */
TSGU_API int tsgu_csr_transpose(const void* rowptr, const void* colind,
                       int64_t batch, int64_t n, int64_t m,
                       int64_t rowptr_bstride, int64_t nnz_bstride, int64_t nnz_total, int idx_dtype,
                       void* rowptrT, void* colindT, void* permT, int out_idx_dtype,
                       void* workspace, size_t workspace_bytes, void* stream);
TSGU_API size_t tsgu_csr_transpose_workspace_bytes(int64_t batch, int64_t m, int64_t nnz_total,
                                          int out_idx_dtype);

/* out[k] = in[perm[k]] for the value array (values[permutation], utils/utils.py:327,340). */
TSGU_API int tsgu_gather_values(const void* in, const void* perm, void* out, int64_t count,
                       int val_dtype, int idx_dtype, void* stream);

/* out[perm[k]] = in[k], every other element of out (out_count elements) zero: the adjoint of tsgu_gather_values for an
 * injective perm -- the backward of the PairwiseEncoder value assembly (encoders/pairwise_encoder.py:744-749, :837). */
TSGU_API int tsgu_scatter_values(const void* in, const void* perm, void* out, int64_t count, int64_t out_count,
                        int val_dtype, int idx_dtype, void* stream);

/* *out (uint64, zeroed by the caller) += position-weighted checksum of an index array of `count` elements.  The host
 * side keeps one per cached sparsity pattern and re-checks it on a thinning schedule of cache hits, so index buffers that
 * were rewritten in place under a cached pattern raise instead of silently reusing the old structure.  No reference
 * counterpart: the reference re-derives all index structure on every call (sparse_matmul.py:190-192 row expansion,
 * :229 re-sort inside torch.sparse.mm(A.t(), .)), so it has nothing to invalidate; this is the guard that makes caching
 * those structures safe. */
TSGU_API int tsgu_fingerprint(const void* data, int64_t count, int idx_dtype, void* out, void* stream);

/* Batched CSR (crow (b, n+1), col (b, nnz)) -> block-diagonal CSR over b*n rows / b*m columns in one pass: the index
 * arithmetic of sparse_block_diag (utils/utils.py:604-645) as the solves need it (sparse_solve.py:172-174). */
TSGU_API int tsgu_block_diag_csr(const void* crow, const void* col, int64_t batch, int64_t n, int64_t m, int64_t nnz,
                        void* crow_out, void* col_out, int idx_dtype, void* stream);

/* Segmented sum of duplicate coordinates: out[u] = sum_{k in [seg[u], seg[u+1])} in[perm[k]]
 * (what coalesce() does to values, utils/utils.py:580). */
TSGU_API int tsgu_segment_sum_values(const void* in, const void* perm, const void* seg, void* out,
                            int64_t nseg, int val_dtype, int idx_dtype, void* stream);

/* Strided dense -> strided dense layout change, coalesced on both sides.  Used for the
 * B.reshape(-1,K) copy of sparse_matmul.py:153 when B is a transposed / permuted view (e.g. from
 * _batch_sparse_mv, distributions/sparse_multivariate_normal.py:96,100) and to hand grad_B back in
 * B's own memory layout (what autograd would otherwise re-stride with a generic copy). */
TSGU_API int tsgu_pack_dense(const void* src, void* dst, int64_t batch, int64_t rows, int64_t cols,
                    int64_t s_bs, int64_t s_rs, int64_t s_cs, int64_t d_bs, int64_t d_rs, int64_t d_cs,
                    int val_dtype, void* stream);

/* tsgu_pack_dense with an additive epilogue: dst[t, r, c] = src[t, r, c] + add[t, r, c] + rowvec[t, r], `add` (nullable)
 * addressed with the destination's strides, `rowvec` (nullable) with (v_bs, v_rs).  One pass for the layout change
 * and the two elementwise adds that follow sparse_mm in SparseMultivariateNormal.rsample
 * (distributions/sparse_multivariate_normal.py:362 "+ eta", :389 "loc +", after the .t() / permute of :96-100). */
TSGU_API int tsgu_pack_dense_add(const void* src, const void* add, const void* rowvec, void* dst, int64_t batch,
                        int64_t rows, int64_t cols, int64_t s_bs, int64_t s_rs, int64_t s_cs, int64_t d_bs,
                        int64_t d_rs, int64_t d_cs, int64_t v_bs, int64_t v_rs, int val_dtype, void* stream);

/* ------------------------------------------------------------------------------------
 * Column-window kernels for structured (banded / stencil) patterns -- same products as
 * tsgu_spmm_csr / tsgu_sddmm_csr (sparse_matmul.py:155, :229, :190-205), for patterns
 * whose tiles of consecutive rows touch few contiguous runs of columns (the 27-point
 * PairwiseEncoder matrices of encoders/pairwise_encoder.py:383-505).
 *
 * tsgu_window_plan (once per pattern): for tiles of `tile_rows` rows writes
 *   lcol  uint16 per stored entry (same indexing as colind): slot of the entry's column in
 *         its tile's window (the dense rank of the column among the tile's distinct columns)
 *   desc  32 int32 per tile: [0] number of column runs (-1: tile does not fit the limits of
 *         tsgu_window_limits), [1] distinct columns, then per run {first column, slot | len << 16}
 *   stats int32[4]: tiles that do not fit, max distinct columns, max runs, max entries per tile
 * The plan is usable iff stats[0] == 0.  32-bit index structures only (idx_dtype == TSGU_I32
 * for the compute entry points).  The compute kernels need K * sizeof(value) in {64, 128, 256}
 * bytes and 16-byte aligned dense rows; `out` of the SDDMM is written exactly like tsgu_sddmm_csr; the SpMM writes element
 * (r, k) of item t at C + t*c_bs + r*ldc + k*c_cs: c_cs == 1 is the row-major result of tsgu_spmm_csr, ldc == 1 a
 * column-major one (grad_B in the layout of a column-major B, without a separate layout pass).  The SpMM reads `vals` in
 * pattern order (entry e has value vals[e]); callers whose values are permuted run tsgu_gather_values first. */
TSGU_API int tsgu_window_limits(int* tile_rows_max, int* entries_max, int* window_rows, int* runs_max);
TSGU_API int tsgu_window_plan(const void* rowptr, const void* colind, int64_t batch, int64_t n,
                     int64_t rowptr_bstride, int64_t nnz_bstride, int idx_dtype, int tile_rows,
                     void* lcol_out, void* desc_out, void* stats_out, void* stream);
TSGU_API int tsgu_spmm_window(const void* rowptr, const void* lcol, const void* desc, const void* vals,
                     const void* B, void* C, int64_t batch, int64_t n, int64_t K,
                     int64_t rowptr_bstride, int64_t nnz_bstride, int64_t nnz_len, int tile_rows,
                     int64_t b_bs, int64_t b_rs, int64_t c_bs, int64_t ldc, int64_t c_cs, int val_dtype,
                     int idx_dtype, void* stream);
TSGU_API int tsgu_sddmm_window(const void* rowptr, const void* lcol, const void* desc, const void* out_index,
                      const void* G, const void* B, void* out, int64_t batch, int64_t n, int64_t K,
                      int64_t rowptr_bstride, int64_t nnz_bstride, int64_t nnz_len, int tile_rows,
                      int64_t g_bs, int64_t g_rs, int64_t b_bs, int64_t b_rs, int val_dtype, int idx_dtype,
                      void* stream);

/* ------------------------------------------------------------------------------------
 * Sparse triangular solve  op(A) X = B  (op(A) = A or A^T), level-scheduled and sync-free.
 *   replaces the torch.triangular_solve / linalg_solve_triangular_compat calls of sparse_solve.py
 *   SparseTriangularSolve.forward (op(A) x = B) and .backward (op(A)^T gradB = grad), which run
 *   cuSPARSE's analysis again inside every call; here the analysis is a per-pattern plan.
 *
 * The solved matrix is a CSR batch in the conventions above, square (m = n); for op(A) = A^T the
 * caller passes the CSR of the transposes (tsgu_csr_transpose) and the opposite triangle.  Only
 * the strictly off-diagonal entries of the requested triangle (`lower`: col < row, else col > row)
 * and the diagonal are read; entries of the other triangle are ignored, like torch's sparse CSR
 * triangular_solve.  Rows are addressed flat: row g = t*n + r of item t.
 *
 * tsgu_trisolve_levels (once per pattern and triangle): level_out[g] = level of row g - 1
 *   (int64, 0-based), count_out[g] = number of its off-diagonal dependencies (int64),
 *   stats_out = uint64[3] {number of levels, total dependencies, status (0 = ok)}; stats_out is
 *   zeroed on `stream` first.  Sorting the rows stably by level (tsgu_coo_sort on (level, row),
 *   key_dims = 1) gives `order`, the plan's row order.
 * tsgu_trisolve_plan: for slot s (row order[s]), with plan_rowptr the exclusive prefix sum of the
 *   dependency counts in slot order (rows + 1 entries, idx_dtype), writes plan_col (flat row of
 *   each dependency), plan_pos (position of its value: perm[e] if `perm` is given, else the
 *   absolute entry position e), and plan_diag[s] (value position of the diagonal entry, -1 if none).
 * tsgu_trisolve: X (row-major (batch, n, K), contiguous) from B (any strides) over a plan.  `vals`
 *   is indexed by plan_pos / plan_diag.  unitriangular: the diagonal is taken as 1 (a stored one is
 *   ignored).  A missing diagonal divides by zero, as the dense solve does.  fp32 and fp64 only
 *   (TSGU_ERR_DTYPE otherwise).  Results are bit-identical from run to run.
 * Workspace (tsgu_trisolve_workspace_bytes, both levels and solve): ticket counter, per-row ready
 *   flags and, as the uint32 at byte offset 8, the status word; each call zeroes it on `stream`.
 *   Every dependency wait is bounded (about one second): a row whose wait expired is written as NaN
 *   and the status word (levels: stats_out[2]) becomes non-zero, so the kernels always terminate.
 * ---------------------------------------------------------------------------------- */
TSGU_API size_t tsgu_trisolve_workspace_bytes(int64_t batch, int64_t n);
TSGU_API int tsgu_trisolve_levels(const void* rowptr, const void* colind, int64_t batch, int64_t n,
                         int64_t rowptr_bstride, int64_t nnz_bstride, int idx_dtype, int lower,
                         void* level_out, void* count_out, void* stats_out, void* workspace,
                         size_t workspace_bytes, void* stream);
TSGU_API int tsgu_trisolve_plan(const void* rowptr, const void* colind, const void* perm, int64_t batch, int64_t n,
                       int64_t rowptr_bstride, int64_t nnz_bstride, int idx_dtype, int lower,
                       const void* order, const void* plan_rowptr, void* plan_col, void* plan_pos,
                       void* plan_diag, void* stream);
TSGU_API int tsgu_trisolve(const void* plan_rowptr, const void* plan_col, const void* plan_pos,
                  const void* plan_diag, const void* order, const void* vals, const void* B, void* X,
                  int64_t batch, int64_t n, int64_t K, int64_t b_bs, int64_t b_rs, int64_t b_cs,
                  int unitriangular, int val_dtype, int idx_dtype, void* workspace, size_t workspace_bytes,
                  void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TSGU_B200_H */
