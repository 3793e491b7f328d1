/* sparse_b200.h — C ABI of libsparse_b200: the B200 (sm_100a) backend for the
 * column-sweep hot path of zdebruine/RcppSparse.
 *
 * Plain C, plain pointers and sizes, no exceptions, no torch/Rcpp types.  Every entry
 * point returns an int status (0 = SB200_OK, negative = category below); the message for
 * the calling thread's last failure is sb200_last_error().  The library never calls the R
 * API and never longjmps, so it is safe under BEGIN_RCPP/END_RCPP (reference
 * src/RcppExports.cpp:17,23): the C++ header turns a non-zero status into an exception.
 *
 * "reference" below = /root/reference (zdebruine/RcppSparse); RcppSparse.h =
 * inst/include/RcppSparse.h.  Layout everywhere is the dgCMatrix slot layout of
 * RcppSparse.h:29-30: x double[nnz], i int32[nnz] (0-based rows, strictly ascending inside
 * a column), p int32[ncol+1] (p[0]=0, p[ncol]=nnz), Dim = (nrow, ncol).
 *
 * There is NO CPU fallback: without a CUDA device every compute entry returns
 * SB200_E_NODEVICE.
 */
#ifndef SPARSE_B200_H
#define SPARSE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SB200_ABI_VERSION 1

/* status codes */
#define SB200_OK 0
#define SB200_E_INVALID (-1)   /* bad argument (null pointer, negative size, wrong handle) */
#define SB200_E_CUDA (-2)      /* a CUDA runtime call or kernel failed; message has the CUDA text */
#define SB200_E_NOMEM (-3)     /* device or host allocation failed */
#define SB200_E_STRUCTURE (-4) /* i/p violate the dgCMatrix invariants (what the reference turns into
                                  Rcpp::index_out_of_bounds at RcppSparse.h:135,142, or silent UB) */
#define SB200_E_NODEVICE (-5)  /* no CUDA device / requested device absent */
#define SB200_E_UNSUPPORTED (-6)

/* flags for sb200_matrix_create* */
#define SB200_PIN_HOST 1u    /* cudaHostRegister i/x for the upload, unregister after; measured SLOWER than the default
                                * for pageable memory (pinned-chunk worker threads): 123-170 ms vs 30 ms for 1.2 GB */
#define SB200_NO_VALIDATE 2u /* skip the structure-validation kernel (trusted producer, benchmarks) */
#define SB200_NO_ROW_PLAN 4u /* sb200_matrix_create: do not prepare the row-band plan during the upload (column sweeps only) */
#define SB200_LAZY_ROWS 8u   /* sb200_matrix_create: leave the row indices `i` on the host until an op reads them.  columnSums /
                                * colSums / colMeans never read `i` (reference src/example.cpp:28-30, RcppSparse.h:133-135), so a
                                * one-shot call uploads 8 of the 12 bytes per entry; `i` is uploaded (and, unless SB200_NO_VALIDATE,
                                * checked) by the first entry point that needs it.  The caller keeps `i` alive and unchanged until
                                * then or until destroy (true for the drop-in header's per-call mirror: R protects the slots for
                                * the lifetime of the Matrix).  Ignored by sb200_sharded_create. */

/* Opaque device-resident mirror of one dgCMatrix (or of one column block of it, which is
 * itself a valid dgCMatrix with the same nrow — the unit of multi-GPU sharding).
 * Replaces the four Rcpp handles of RcppSparse.h:29-30 as the thing kernels read. */
typedef struct sb200_matrix sb200_matrix;

/* ---- library / errors ------------------------------------------------------------------ */
int sb200_abi_version(void);
const char* sb200_last_error(void);      /* thread-local, never NULL */
int sb200_device_count(int* count);      /* SB200_E_NODEVICE when there is none */

/* ---- mirror lifecycle -------------------------------------------------------------------
 * sb200_matrix_create: what Exporter::get() / the 4-vector constructor do in the reference
 * (RcppSparse.h:33,417-419) plus the one-time upload.  The host arrays are BORROWED for the
 * duration of the call only (copied to HBM); they may be R-owned pageable memory (staged through pinned
 * chunks by worker threads, SB200_COPY_THREADS) or
 * already pinned.  Structure is validated on the device unless SB200_NO_VALIDATE. */
int sb200_matrix_create(const int32_t* i, const int32_t* p, const double* x, int32_t nrow, int32_t ncol,
                        int64_t nnz, int device, unsigned flags, sb200_matrix** out);
/* Adopt arrays that already live in HBM on `device` (a generator's output, a torch tensor,
 * a rank's column shard).  Not copied, not freed by destroy; must outlive the handle.
 * d_i and d_x must be 16-byte aligned and readable up to the next 16-byte boundary past
 * their last element; d_p likewise (cudaMalloc / torch allocations satisfy this). */
int sb200_matrix_adopt_device(const int32_t* d_i, const int32_t* d_p, const double* d_x, int32_t nrow,
                              int32_t ncol, int64_t nnz, int device, unsigned flags, sb200_matrix** out);
int sb200_matrix_destroy(sb200_matrix* m);
int sb200_matrix_dims(const sb200_matrix* m, int32_t* nrow, int32_t* ncol, int64_t* nnz);
/* The view aliases R memory and users may mutate x in place (reference
 * vignettes/Documentation.Rmd:325-347); this re-uploads x[nnz] into the mirror. */
int sb200_matrix_refresh_values(sb200_matrix* m, const double* x);
/* Run this handle's work on a caller-owned CUDA stream (a cudaStream_t passed as void*,
 * e.g. torch.cuda.current_stream().cuda_stream) so the caller's events bracket it. */
int sb200_matrix_set_stream(sb200_matrix* m, void* cuda_stream);
int sb200_matrix_sync(sb200_matrix* m);
/* Device pointers of the mirror (for callers that shard or inspect it). */
int sb200_matrix_device_arrays(const sb200_matrix* m, const int32_t** d_i, const int32_t** d_p,
                               const double** d_x);

/* ---- the sweeps, host-buffer form (what the C++ header calls) -----------------------------
 * Output buffers are caller-allocated host memory of the stated length (the NumericVector
 * the header allocates); the call returns after the result is in `out`.
 *   sb200_col_sums   replaces Matrix::colSums()  RcppSparse.h:131-137 and columnSums() src/example.cpp:26-32
 *   sb200_row_sums   replaces Matrix::rowSums()  RcppSparse.h:138-144
 *   sb200_col_means  replaces Matrix::colMeans() RcppSparse.h:145-150 (sum / nrow, true division)
 *   sb200_row_means  replaces Matrix::rowMeans() RcppSparse.h:151-156 (sum / ncol)
 *   sb200_spmv       y[nrow] = A v[ncol]   — the InnerIterator sweep y[it.row()] += it.value()*v[col]
 *   sb200_spmv_t     y[ncol] = A^T v[nrow] — the sweep y[col] += it.value()*v[it.row()]
 *                    (idiom of src/example.cpp:28-30; the reference has no SpMV function)
 *   sb200_transpose  replaces Matrix::transpose() RcppSparse.h:375-385: canonical CSC of A^T,
 *                    p_out[nrow+1], i_out[nnz] ascending inside each new column, x_out[nnz] */
int sb200_col_sums(sb200_matrix* m, double* out /* ncol */);
int sb200_row_sums(sb200_matrix* m, double* out /* nrow */);
int sb200_col_means(sb200_matrix* m, double* out /* ncol */);
int sb200_row_means(sb200_matrix* m, double* out /* nrow */);
int sb200_spmv(sb200_matrix* m, const double* v /* ncol */, double* y /* nrow */);
int sb200_spmv_t(sb200_matrix* m, const double* v /* nrow */, double* y /* ncol */);
int sb200_transpose(sb200_matrix* m, int32_t* p_out, int32_t* i_out, double* x_out);

/* Column and row variances (sparseMatrixStats::colVars / rowVars; the reference has none): out[c] is the sample variance
 * of the nrow values of column c — its stored entries and its nrow - nnz_c implicit zeros — over nrow - 1, as R's
 * var(A[, c]); out[r] the same over the ncol values of row r, over ncol - 1.  Two passes: the mean m is exactly what
 * sb200_col_means / sb200_row_means return (same sweep, same division), then S = sum over the stored entries of
 * (x - m)^2, and the result is (S + (n - cnt) m^2) / (n - 1) with cnt the stored entries (explicit zeros count).  No
 * one-pass formula: within 1e-12 * exact + 2 * spacing(m)^2 of the exact variance of the double inputs, also on nearly
 * constant data (mean 1e9, variance 1).  colVars is bit-stable run to run; rowVars is where rowSums is (on the
 * row-ordered copy; the plan-free and banded paths add with FP64 atomics), and like rowSums it runs on that copy when
 * the mirror has one, else on the path sb200_matrix_row_path reports; one call counts once toward building the copy.
 * NaN or +-Inf among the entries of a column / row make that output NaN and no other.  An empty column / row gives +0.0.
 * A dimension below 2 gives NaN for every output (R gives NA there); an output dimension of 0 writes nothing.  Scratch
 * (8 bytes per output, 16 for rowVars) comes from the device: SB200_E_NOMEM when it does not fit.  A NULL output of
 * non-empty shape: SB200_E_INVALID. */
int sb200_col_vars(sb200_matrix* m, double* out /* ncol */);
int sb200_row_vars(sb200_matrix* m, double* out /* nrow */);

/* ---- the sweeps, device-buffer form (asynchronous on the handle's stream) ------------------
 * Operands and results are device pointers on the handle's device.  Used by the sharding
 * layer (results feed NCCL collectives without touching the host) and by bench.py.
 * `divisor` of the *_scaled forms: result = sum / divisor (0 = no scaling); a sharded
 * rowMeans/colMeans passes the GLOBAL dimension here. */
int sb200_col_sums_dev(sb200_matrix* m, double divisor, double* d_out /* ncol */);
int sb200_row_sums_dev(sb200_matrix* m, double divisor, double* d_out /* nrow */);
int sb200_spmv_dev(sb200_matrix* m, const double* d_v /* ncol */, double* d_y /* nrow */);
int sb200_spmv_t_dev(sb200_matrix* m, const double* d_v /* nrow */, double* d_y /* ncol */);
/* sb200_col_vars / sb200_row_vars into a device buffer, asynchronous on the handle's stream (tools/vars_bench.py). */
int sb200_col_vars_dev(sb200_matrix* m, double* d_out /* ncol */);
int sb200_row_vars_dev(sb200_matrix* m, double* d_out /* nrow */);
/* Result stays in HBM as a new handle that owns its arrays (Dim swapped). */
int sb200_transpose_dev(sb200_matrix* m, sb200_matrix** out);
/* The same transpose (RcppSparse.h:375-385) written into a result that sb200_transpose_dev produced earlier for a matrix
 * of this structure (t: Dim swapped, same nnz, owns its arrays): nothing is allocated, t's tile plans stay (they depend on
 * the structure only), its cached layouts are dropped.  For mirrors whose values change and whose transpose is wanted
 * again (sb200_matrix_refresh_values + this).  Blocking. */
int sb200_transpose_into(sb200_matrix* m, sb200_matrix* t);
/* d[k] /= divisor for k < n, on the handle's stream (mean scaling after a cross-rank reduce). */
int sb200_vec_div_dev(sb200_matrix* m, double* d, int64_t n, double divisor);

/* Dense A^T A (reference Matrix::crossprod(), RcppSparse.h:158-194): ncol x ncol doubles, column-major, exactly
 * symmetric.  Computed as the sum over rows of (row)^T (row) on the row-ordered copy of the mirror (built, and
 * kept, for mirrors that own their arrays; temporary otherwise).  Entries agree with the reference within
 * 1e-12 * sum |a_ri a_rj| (the additions inside an entry are not in the reference's ascending-row order). */
int sb200_crossprod(sb200_matrix* m, double* out /* ncol*ncol, host */);
int sb200_crossprod_dev(sb200_matrix* m, double* d_out /* ncol*ncol, device */);

/* Sparse x dense block: Y = A B (sb200_spmm) and Y = A^T B (sb200_spmm_t) for k right-hand sides in one sweep of the
 * matrix, where k calls of sb200_spmv / sb200_spmv_t would stream it k times (NMF, randomized SVD / PCA, block
 * Lanczos, subspace iteration, several least-squares right-hand sides).  B and Y are dense and COLUMN-major (R's
 * NumericMatrix): A B takes B ncol x k and fills Y nrow x k, A^T B takes B nrow x k and fills Y ncol x k.  Column j
 * of Y is what sb200_spmv / sb200_spmv_t gives for column j of B, within 1e-12 * sum |a b| per entry; NaN and Inf in
 * B reach exactly the outputs whose stored entries touch them.  k = 0 writes nothing and launches nothing; k = 1 is
 * sb200_spmv / sb200_spmv_t.  A^T B is bit-stable run to run (no atomics).  A B runs on the row-ordered copy when the
 * mirror holds one (then also bit-stable; a k-wide call counts once toward building it, like one A v call), else
 * with FP64 reductions at L2.  Scratch for a row-major copy of B and Y (8 k (nrow + ncol) bytes) comes from the
 * device; SB200_E_NOMEM when it does not fit.  k < 0, or a NULL B / Y of non-empty shape: SB200_E_INVALID.
 * Host form: B and Y are host memory; returns when Y is complete.  Device form: device pointers, asynchronous on
 * the handle's stream. */
int sb200_spmm(sb200_matrix* m, const double* B /* ncol x k, col-major, host */, int64_t k, double* Y /* nrow x k */);
int sb200_spmm_t(sb200_matrix* m, const double* B /* nrow x k */, int64_t k, double* Y /* ncol x k */);
int sb200_spmm_dev(sb200_matrix* m, const double* d_B, int64_t k, double* d_Y);
int sb200_spmm_t_dev(sb200_matrix* m, const double* d_B, int64_t k, double* d_Y);

/* Which kernel serves the row-indexed sweeps of this matrix: *banded = 1 shared-memory row bands
 * (a band plan is built on first use and cached with the mirror), 0 = plan-free L2 atomics.
 * Decided once per handle from the shape (see DESIGN.md 4.2); SB200_ROW_PLAN=0/1 overrides. */
int sb200_matrix_row_path(sb200_matrix* m, int* banded);

/* Row-major companion of a RESIDENT mirror.  rowSums / rowMeans / A v scatter by row index when they run on
 * the CSC arrays (the reference's loop, RcppSparse.h:137-143, 153-160); a mirror that is asked for them more
 * than SB200_ROW_COMPANION_AFTER times (default 8; 0 = never) and owns its arrays (created from host
 * buffers, generated or transposed here — not adopted device arrays, whose values the caller may change
 * behind the mirror) keeps a row-ordered copy of itself (one device transpose, + 12 B per entry of HBM) and
 * serves the row sums as streaming segmented sums and A v as a gather sweep from then on;
 * sb200_matrix_row_path reports 2.  sb200_matrix_refresh_values drops the copy.  action: 1 = build now (also
 * for adopted arrays: the caller promises to call this again, or refresh, after changing values), 0 = drop,
 * -1 = drop and never build. */
int sb200_matrix_row_companion(sb200_matrix* m, int action);

/* Band-major companion of a RESIDENT mirror, for the two products.  A^T v gathers v[i[k]] once per stored entry; on
 * the CSC arrays those gathers go to L2 (8 MB of operand does not fit shared memory) and its request rate, not
 * HBM, bounds the sweep.  A mirror that is asked for A^T v more than SB200_ROW_COMPANION_AFTER times (default 8) and
 * owns its arrays keeps a copy of its entries regrouped by (row band of <= 12288 rows, column) with 16-bit
 * in-band row ids (+10 B per entry of HBM, one pass to build): the operand's slice of a band then sits in shared
 * memory while the band's entries stream through, and a (column, band) run leaves as one FP64 reduction on
 * y[column].  A v is the same sweep on the row-ordered copy's own companion (which = 1 builds both).  Same
 * arithmetic every call: only the layout is kept.  sb200_matrix_refresh_values drops it.
 * which: 0 = the layout A^T v runs on, 1 = the layout A v runs on; action: 1 build now, 0 drop, -1 drop and never build. */
int sb200_matrix_band_companion(sb200_matrix* m, int which, int action);
/* Bit mask of the cached layouts this mirror holds: 1 row-ordered copy, 2 band-major companion (A^T v),
 * 4 band-major companion of the row-ordered copy (A v), 8 transpose plan. */
int sb200_matrix_layouts(sb200_matrix* m, int* mask);
/* HBM bytes the cached layouts of this mirror occupy (row-ordered copy, band-major companions, transpose plan),
 * beside its i/p/x. */
int sb200_matrix_layout_bytes(sb200_matrix* m, int64_t* bytes);

/* ---- cross-GPU exchange for column-sharded matrices (one process per GPU, GPUs of one node) ---------
 * The reference is single-process; a column-sharded deployment (SURVEY.md 8e) needs two exchange steps:
 * assembling column-indexed results from disjoint slices, and summing full-length row-indexed partials.
 * Both run as this library's kernels over NVLink peer memory.  Each rank creates a window of device memory,
 * the 64-byte handles are exchanged by the host side (any transport; rcppsparse_b200/shard.py uses
 * torch.distributed), every rank connects, and result vectors are placed INSIDE the window (offsets in
 * bytes from the window base, 16-byte aligned, at or after *data_offset).  Every rank must issue the same
 * sequence of gather / reduce / barrier calls.  All calls are asynchronous on the given stream. */
typedef struct sb200_exchange sb200_exchange;
int sb200_exchange_create(int device, int64_t data_bytes, sb200_exchange** out, void* ipc_handle_out /* 64 bytes */);
int sb200_exchange_connect(sb200_exchange* x, int rank, int world, const void* all_handles /* world x 64 bytes, by rank */);
int sb200_exchange_destroy(sb200_exchange* x);
int sb200_exchange_window(const sb200_exchange* x, void** base, int64_t* data_offset, int64_t* bytes);
/* Column-indexed result: this rank has written doubles [slice_begin, slice_begin+slice_len) of the vector at
 * full_offset in ITS window; copy them to the same place in every peer's window and wait until every
 * rank's slice has landed here. */
int sb200_exchange_gather(sb200_exchange* x, void* cuda_stream, int64_t full_offset, int64_t slice_begin, int64_t slice_len);
/* Row-indexed result: every rank holds an n-vector of partial sums at partial_offset of its window; on return
 * (in stream order) the vector at result_offset of EVERY window holds their sum, added in rank order (bit-
 * identical on all ranks and run to run), divided by divisor when divisor != 0 (rowMeans: the global ncol,
 * RcppSparse.h:154). partial and result must not overlap. */
int sb200_exchange_reduce(sb200_exchange* x, void* cuda_stream, int64_t partial_offset, int64_t result_offset, int64_t n,
                          double divisor);
/* Sharded transpose: every rank has transposed its own column block (d_p_loc[nrow+1], d_cols local column ids, d_vals);
 * output row r belongs to the rank q with row_bounds[q] <= r < row_bounds[q+1] and is the concatenation, in rank order, of
 * the ranks' segments of row r.  Writes MY segment of every row straight into its owner's window — column ids (made global
 * with col_offset) at byte offset cols_offsets[q], values at vals_offsets[q], segment of row r starting d_dst_off[r]
 * entries into those regions — and waits until every rank's segments have landed here. */
int sb200_exchange_push_rows(sb200_exchange* x, void* cuda_stream, const int32_t* d_p_loc, const int32_t* d_cols,
                             const double* d_vals, const int64_t* d_dst_off, int32_t nrow, int32_t col_offset,
                             const int32_t* row_bounds /* world + 1, host */, const int64_t* cols_offsets /* world, host */,
                             const int64_t* vals_offsets /* world, host */);
int sb200_exchange_barrier(sb200_exchange* x, void* cuda_stream);
/* Synchronises the device; SB200_E_CUDA if a barrier gave up waiting for a peer.  A barrier that sees no signal
 * from a peer for SB200_EXCHANGE_TIMEOUT_S seconds (default 600) raises the window's error word and traps its kernel: the
 * stream and every later CUDA call fail, no result computed from partial data is ever returned. */
int sb200_exchange_status(sb200_exchange* x);

/* ---- range cursors and dense extraction as batched device ops (SURVEY.md 8f N4) ----------------------------------
 * sb200_col_sums_in_rows: for every column c at once, out[c] = the sum a user loop over
 * InnerIteratorInRange(A, c, s) (negate = 0, reference RcppSparse.h:238-264) or InnerIteratorNotInRange(A, c, s)
 * (negate = 1, :270-321) accumulates: the entries of column c whose row is / is not in the index set rows[n] (host
 * array; order and duplicates do not matter; indices outside [0, nrow) select nothing).  Entries outside the
 * selection are skipped, not multiplied by zero: an Inf or NaN outside it does not reach the sum.
 * sb200_gather_block: out[jc * nr + ir] = A(rows[ir], cols[jc]), dense column-major nr x nc (reference :76-92
 * operator()(IntegerVector, IntegerVector)); rows = NULL takes every row (:95-107 col(...)), cols = NULL every column
 * (:110-128 row(...)); indices outside the matrix give 0. */
int sb200_col_sums_in_rows(sb200_matrix* m, const int32_t* rows, int64_t n, int negate, double* out /* ncol */);
int sb200_gather_block(sb200_matrix* m, const int32_t* rows, int64_t nr, const int32_t* cols, int64_t nc,
                       double* out /* nr * nc, column-major, host */);

/* ---- one process, several GPUs (SURVEY.md 8e behind the shim) --------------------------------------------------
 * The reference is ONE R process calling Matrix methods (RcppSparse.h:131-156); a drop-in cannot be launched as one
 * process per GPU.  sb200_sharded_create cuts the dgCMatrix into n_gpus nnz-balanced contiguous column blocks
 * (columns are independent units; a block is a dgCMatrix with the full row count), uploads block k to devices[k]
 * (NULL = devices 0..n_gpus-1; the devices need peer access to each other when n_gpus > 1) and returns one handle.
 * The ops take and fill HOST vectors like the single-GPU entry points: column-indexed results are disjoint slices
 * copied straight to their place; row-indexed results are full-length partials summed in block order by the
 * library's P2P reduction kernel on all devices at once (bit-identical run to run for deterministic partials).
 * The drop-in header uses this form when SB200_GPUS > 1.  Error behaviour as sb200_matrix_create. */
typedef struct sb200_sharded sb200_sharded;
int sb200_sharded_create(const int32_t* i, const int32_t* p, const double* x, int32_t nrow, int32_t ncol, int64_t nnz,
                         int n_gpus, const int* devices, unsigned flags, sb200_sharded** out);
int sb200_sharded_destroy(sb200_sharded* s);
int sb200_sharded_info(const sb200_sharded* s, int* n_gpus, int64_t* bounds /* n_gpus + 1 first columns, or NULL */);
int sb200_sharded_block(const sb200_sharded* s, int k, sb200_matrix** block /* borrowed: block k's mirror */);
int sb200_sharded_col_sums(sb200_sharded* s, double* out /* ncol */);
int sb200_sharded_row_sums(sb200_sharded* s, double* out /* nrow */);
int sb200_sharded_col_means(sb200_sharded* s, double* out /* ncol */);
int sb200_sharded_row_means(sb200_sharded* s, double* out /* nrow */);
int sb200_sharded_spmv(sb200_sharded* s, const double* v /* ncol */, double* y /* nrow */);
int sb200_sharded_spmv_t(sb200_sharded* s, const double* v /* nrow */, double* y /* ncol */);
/* Y = A B and Y = A^T B for k right-hand sides (sb200_spmm / sb200_spmm_t) on every device of the handle.  Same contract
 * as the one-GPU host form: B and Y are column-major host buffers, the call returns when Y is complete, column j of Y is
 * what sb200_sharded_spmv / sb200_sharded_spmv_t gives for column j of B within 1e-12 * sum |a b| per entry, NaN and Inf
 * in B reach exactly the outputs they touch, k = 0 writes and launches nothing, k < 0 or a NULL B / Y of non-empty
 * shape is SB200_E_INVALID, scratch that does not fit is SB200_E_NOMEM (the handle stays usable).
 * A^T B: every device gets all of B, runs the one-GPU block product on its block and copies its rows of Y home; bit-
 * stable run to run, and at n_gpus = 1 bit-identical to sb200_spmm_t.  A B: device w gets its block's rows of B and
 * leaves a full-height partial A_w B_w (8 nrow k bytes of device memory per block, kept between calls); device q sums
 * rows [q nrow / n_gpus, (q+1) nrow / n_gpus) of all partials over peer memory in block order and copies them home.
 * Bit-stable run to run when every block serves A B from its row-ordered copy; a k-wide call counts once per block
 * toward building that copy, like one A v call.  Devices are ordered by CUDA events only, so blocks may share a device. */
int sb200_sharded_spmm(sb200_sharded* s, const double* B /* ncol x k, col-major, host */, int64_t k, double* Y /* nrow x k */);
int sb200_sharded_spmm_t(sb200_sharded* s, const double* B /* nrow x k */, int64_t k, double* Y /* ncol x k */);
/* Matrix::transpose() (RcppSparse.h:375-385) of the whole matrix into host arrays: local transposes on every device, row
 * pieces exchanged over peer memory in block (= column) order, every device copies its rows home (SURVEY.md 8e).
 * Bit-exact like the one-GPU transpose.  Blocking. */
int sb200_sharded_transpose(sb200_sharded* s, int32_t* p_out /* nrow + 1 */, int32_t* i_out /* nnz */, double* x_out /* nnz */);
/* Matrix::crossprod() (RcppSparse.h:158-194) on every device of the handle: dense A^T A into the column-major host buffer
 * `out`.  Every entry res(a, b) is the sum over rows r of x_ra * x_rb, from +0.0, added in ascending row order with no
 * contraction and no atomics: the reference's result bit for bit (NaN payloads aside; NaN positions match), exactly
 * symmetric, and the same bits run to run, for any n_gpus and any placement.  Device w computes the result columns of its
 * block, a contiguous range of `out` (8 ncol ncol_w bytes of device memory, plus a 12 nnz byte row-ordered copy of the
 * whole matrix built per call over peer memory), and copies it home over its own link.  ncol = 0 writes nothing; nnz = 0
 * or nrow = 0 gives zeros.  A NULL `out` with ncol > 0 is SB200_E_INVALID; device memory that does not fit is
 * SB200_E_NOMEM before anything is written (the handle stays usable).  Devices are ordered by CUDA events and host
 * synchronisation only, so blocks may share a device.  Blocking. */
int sb200_sharded_crossprod(sb200_sharded* s, double* out /* ncol*ncol, column-major, host */);
/* sb200_col_vars / sb200_row_vars on every device of the handle, same contract and bar.  colVars: every block runs the
 * one-GPU two-pass sweep on its columns and its slice goes straight home; bit-stable, and bit-identical to
 * sb200_col_vars at n_gpus = 1.  rowVars: the global row means as sb200_sharded_row_means computes them, then every
 * block's sums of squares and entry counts over its own columns (16 nrow bytes of device memory per block, kept
 * between calls; SB200_E_NOMEM when they do not fit), added in block order over peer memory, device q finishing rows
 * [q nrow / n_gpus, (q+1) nrow / n_gpus) and copying them home.  Bit-stable where every block serves its row sums
 * from its row-ordered copy.  That reduce is ordered by CUDA events only, so blocks may share a device.  Blocking. */
int sb200_sharded_col_vars(sb200_sharded* s, double* out /* ncol */);
int sb200_sharded_row_vars(sb200_sharded* s, double* out /* nrow */);

/* Scratch, results and cached layouts come from the device's stream-ordered memory pool, which keeps freed blocks
 * for reuse (a multi-GB cudaMalloc/cudaFree pair costs as much as a sweep).  sb200_trim synchronises the device and
 * hands everything the pool holds but does not use back to the driver (e.g. before another library allocates). */
int sb200_trim(int device);

/* ---- introspection for benchmarks ----------------------------------------------------------
 * Number of kernel launches this library has issued in this process (all handles). */
int64_t sb200_launch_count(void);
/* Name and per-launch algorithmic bytes (SURVEY.md 8d figures) of the dominant kernel of an op:
 * op = "col_sums" | "row_sums" | "col_means" | "row_means" | "spmv" | "spmv_t" | "transpose" |
 * "row_sums_companion" | "row_means_companion" (what the row sums read once the row-ordered copy exists) |
 * "col_vars" | "row_vars" (compulsory: every array once, as for the sums; the two passes read x twice). */
int sb200_algorithmic_bytes(const sb200_matrix* m, const char* op, int64_t* bytes);

/* ---- synthetic matrices generated straight into HBM (tests and benchmarks) -----------------
 * Integer-exact recipe shared with rcppsparse_b200/synth.py (bit-identical output).
 * len_table: int64[4097] quantile table; bands: K ascending row bands [lo,hi) with weights.
 * Columns [col_begin, col_end) are generated; p is rebased to 0.  The new handle owns its arrays. */
int sb200_synth_create(int32_t nrow, int64_t col_begin, int64_t col_end, uint64_t seed,
                       const int64_t* len_table, int32_t empty_permille, int32_t n_bands,
                       const int64_t* band_lo, const int64_t* band_hi, const int64_t* band_w, int device,
                       sb200_matrix** out);
/* v[k] for k in [begin, begin+n): the dense SpMV operand of the recipe (seed+1 stream). */
int sb200_synth_vector_dev(sb200_matrix* m, uint64_t seed, int64_t begin, int64_t n, double* d_out);
/* Copy a column block [c0, c1) of the mirror back to host buffers (p rebased to 0);
 * sizes: p_out[c1-c0+1]; i_out/x_out sized by the block's nnz (query with i_out = NULL:
 * only *nnz_out is written). */
int sb200_matrix_download_columns(sb200_matrix* m, int64_t c0, int64_t c1, int32_t* i_out, int32_t* p_out,
                                  double* x_out, int64_t* nnz_out);

#ifdef __cplusplus
}
#endif
#endif /* SPARSE_B200_H */
