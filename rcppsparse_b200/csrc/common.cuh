// Shared declarations of libsparse_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <atomic>
#include <chrono>
#include <initializer_list>
#include <string>

#include "../../include/sparse_b200.h"

namespace sb200 {

// ---------------------------------------------------------------------------------------------
// error plumbing: the C ABI never throws; every internal step returns a status.
// ---------------------------------------------------------------------------------------------
void set_error(const std::string& msg);
int fail(int code, const std::string& msg);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define SB_CUDA(expr)                                                        \
  do {                                                                       \
    cudaError_t sb_e_ = (expr);                                              \
    if (sb_e_ != cudaSuccess) return ::sb200::cuda_fail(sb_e_, #expr, __FILE__, __LINE__); \
  } while (0)

#define SB_TRY(expr)              \
  do {                            \
    int sb_rc_ = (expr);          \
    if (sb_rc_ != SB200_OK) return sb_rc_; \
  } while (0)

extern std::atomic<int64_t> g_launches;  // kernels launched by this library (sb200_launch_count)
inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---------------------------------------------------------------------------------------------
// geometry of the merge-path sweep (sweep.cu) — one "item" is either one stored entry or one
// column end; a tile is SWEEP_TILE consecutive items on the merge path of (p[1..ncol], 0..nnz).
// ---------------------------------------------------------------------------------------------
constexpr int SWEEP_THREADS = 256;
// items per thread, odd => conflict-free 8-byte shared-memory reads at stride IPT.  Two geometries
// (measured, profiles/r01): the plain column sums want 11 (34 KB stages, 3 CTAs/SM: 83-101 % of peak),
// the gather/scatter sweeps want 7 (29 KB stages, 3 CTAs/SM: more warps to hide the L2 gathers).
constexpr int SWEEP_IPT = 11;
constexpr int SWEEP_TILE = SWEEP_THREADS * SWEEP_IPT;  // 2816 items per tile (also the band-pointer tiling)
constexpr int GATHER_IPT = 7;
constexpr int GATHER_TILE = SWEEP_THREADS * GATHER_IPT;  // 1792 items per tile

constexpr int NUM_SMS_B200 = 148;

// ---------------------------------------------------------------------------------------------
// the device-resident mirror
// ---------------------------------------------------------------------------------------------
struct BandPlan;       // bands.cu
struct BandCompanion;  // bmc.cu
struct SplitPlan;      // transpose_split.cu

}  // namespace sb200

struct sb200_matrix {
  uint32_t magic;
  int device;
  int sm_count;
  cudaStream_t stream;
  bool owns_stream;
  bool owns_arrays;
  int32_t nrow, ncol;
  int64_t nnz;
  // mirror of the dgCMatrix slots (RcppSparse.h:29-30); allocations are padded so that 16-byte
  // bulk copies starting at any 16-byte-aligned element may run to the next 16-byte boundary.
  int32_t* d_i;
  int32_t* d_p;
  double* d_x;
  // merge-path plan: plan[t] = number of column ends before diagonal t*SWEEP_TILE (t = 0..n_tiles)
  int32_t* d_plan;
  int64_t n_tiles;
  int32_t* d_plan_g;  // same, every GATHER_TILE items
  int64_t n_tiles_g;
  // per-launch workspace (carries, tickets), zeroed where the kernels expect zero
  void* d_ws;
  size_t ws_bytes;
  // device staging for the host-buffer entry points
  double* d_stage_in;
  double* d_stage_out;
  int64_t stage_len;
  // row-band plan for the row-indexed sweeps (bands.cu); structure-only, built on first use
  sb200::BandPlan* plan_scatter;
  int row_path;  // -1 undecided, 0 plan-free L2 atomics, 1 banded (decide_row_path)
  sb200::BandPlan* plan_gather;  // wider bands (v's slice in shared memory) for A^T v, built on first use
  int gather_path;               // -1 undecided, 0 sweep_kernel<SPMV_T> (L2 gathers), 1 banded gather
  // Row-major companion for rowSums / rowMeans / A v on a resident mirror (capi.cu, build_row_companion): the
  // transposed copy.  Built after `row_companion_after()` row-indexed calls on a mirror that owns its arrays,
  // dropped by refresh_values.
  sb200_matrix* rows;
  int rows_state;     // 0 not built, 1 built, -1 never (disabled, or the build failed once)
  int row_sum_calls;  // row-indexed calls served by the scatter kernels since the last (re)build decision
  // Band-major companion for A^T v (bmc.cu): the entries regrouped by (row band, column), local 16-bit row ids, so
  // that the operand's slice of a band sits in shared memory while the band's entries stream through the TMA ring.
  // Built after `row_companion_after()` A^T v calls on a mirror that owns its arrays (A v: the same on `rows`).
  sb200::BandCompanion* bmc;
  int bmc_state;      // 0 not built, 1 built, -1 never
  int spmv_t_calls;   // A^T v calls served by the L2-gather sweep since the last (re)build decision
  sb200::BandPlan* plan_transpose;  // band plan of the transpose, kept between calls (structure only)
  sb200::SplitPlan* plan_split;     // same for the two-split transpose of tall matrices (transpose_split.cu)
  // SB200_LAZY_ROWS: the caller's row indices, still on the host; d_i is allocated but not filled until ensure_rows()
  const int32_t* lazy_i;
  bool lazy_validate;
};

namespace sb200 {

constexpr uint32_t MATRIX_MAGIC = 0x5B200C5Cu;

inline int check_handle(const sb200_matrix* m) {
  if (m == nullptr || m->magic != MATRIX_MAGIC) return fail(SB200_E_INVALID, "not a live sb200_matrix handle");
  return SB200_OK;
}

// RAII device switch for entry points
struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

// SB200_TRACE=1: host wall clock of the phases of an entry point on stderr, one line per phase
struct WallTrace {
  bool on = getenv("SB200_TRACE") != nullptr;
  const char* title;
  std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
  explicit WallTrace(const char* what) : title(what) {}
  void phase(const char* what) {
    if (!on) return;
    const auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[sb200 trace] %s: %s %.2f ms\n", title, what, std::chrono::duration<double, std::milli>(now - t).count());
    t = now;
  }
};

// SB200_TRACE=1: device time between marks on one stream, one line on stderr.  mark(name) records an event; report()
// prints the caller's header and then " name ms;" for the gap that ends at every mark after the first.
struct PhaseTrace {
  static constexpr int MAX_MARKS = 8;
  bool on = getenv("SB200_TRACE") != nullptr;
  cudaStream_t st;
  cudaEvent_t ev[MAX_MARKS];
  const char* name[MAX_MARKS];
  int n = 0;
  explicit PhaseTrace(cudaStream_t s) : st(s) {}
  ~PhaseTrace() {
    for (int k = 0; k < n; ++k) cudaEventDestroy(ev[k]);
  }
  void mark(const char* what) {
    if (!on || n >= MAX_MARKS) return;
    cudaEventCreate(&ev[n]);
    cudaEventRecord(ev[n], st);
    name[n++] = what;
  }
  __attribute__((format(printf, 2, 3))) void report(const char* header, ...) {
    if (!on) return;
    cudaStreamSynchronize(st);
    char buf[256];
    va_list ap;
    va_start(ap, header);
    vsnprintf(buf, sizeof(buf), header, ap);
    va_end(ap);
    std::string line = std::string("[sb200 trace] ") + buf;
    for (int k = 1; k < n; ++k) {
      float ms = 0;
      cudaEventElapsedTime(&ms, ev[k - 1], ev[k]);
      snprintf(buf, sizeof(buf), " %s %.3f ms;", name[k], ms);
      line += buf;
    }
    fprintf(stderr, "%s\n", line.c_str());  // one write: concurrent plans on other threads do not cut into the line
  }
};

// sweep.cu
// COLVAR / ROWVAR: colVars / rowVars through launch_sweep (vars.cu); COLVAR is also the kernel mode of their second pass
enum SweepMode { SWEEP_COLSUM = 0, SWEEP_SPMV_T = 1, SWEEP_ROWSUM = 2, SWEEP_SPMV = 3, SWEEP_COLVAR = 4, SWEEP_ROWVAR = 5 };
int build_sweep_plan(sb200_matrix* m);
int launch_sweep(sb200_matrix* m, SweepMode mode, const double* d_v, double divisor, double* d_out);
int launch_vec_div(cudaStream_t s, double* d, int64_t n, double divisor);
int launch_col_var_sweep(sb200_matrix* m, const double* d_mean, double n, double* d_out);  // n = 0: raw sums of squares

// vars.cu: two-pass variances.  The variance of n values (n >= 2) of which cnt are stored entries whose squared
// deviations from the mean mu sum to S and n - cnt are zeros, over n - 1 (R's var()).
__device__ __forceinline__ double var_from_sums(double S, double cnt, double mu, double n) {
  return __ddiv_rn(__dadd_rn(S, __dmul_rn(__dsub_rn(n, cnt), __dmul_rn(mu, mu))), __dsub_rn(n, 1.0));
}
int launch_col_vars(sb200_matrix* m, double* d_out);  // ncol outputs, NaN when nrow < 2
int launch_row_vars(sb200_matrix* m, double* d_out);  // nrow outputs, NaN when ncol < 2
// Second pass of rowVars without the formula, for the sharded reduce: d_S[r] = sum over row r's stored entries of
// (x - d_mean[r])^2, d_cnt[r] = their number (as a double), on the path rowSums takes on this mirror.
int launch_row_var_sums(sb200_matrix* m, const double* d_mean, double* d_S, double* d_cnt);
int launch_fill_nan(cudaStream_t s, double* d, int64_t n);

// validate.cu
int validate_structure(sb200_matrix* m, bool rows = true);  // p always; i (range, ascending inside a column) when rows
int validate_rows(sb200_matrix* m);                         // i alone, once p is known to be sound
int ensure_rows(sb200_matrix* m);                           // capi.cu: upload and check a lazily kept `i` (SB200_LAZY_ROWS)

// scan.cu — exclusive prefix sum of u32 counts into int32 offsets (out has n+1 entries);
// d_total (optional) receives the 64-bit grand total.  ws must hold scan_workspace_bytes(n).
size_t scan_workspace_bytes(int64_t n);
int exclusive_scan_u32(cudaStream_t s, const uint32_t* d_in, int32_t* d_out, int64_t n, unsigned long long* d_total,
                       void* d_ws, size_t ws_bytes);

// bands.cu
int transpose_device(sb200_matrix* m, int32_t* d_p_out, int32_t* d_i_out, double* d_x_out);
int ensure_scatter_plan(sb200_matrix* m);
int decide_row_path(sb200_matrix* m);
int decide_gather_path(sb200_matrix* m);
int launch_band_gather(sb200_matrix* m, const double* d_v, double* d_out);
int launch_band_scatter(sb200_matrix* m, const double* d_v, double* d_out);  // d_v null = rowSums
// rowVars' second pass on the row bands: d_S[r] = sum of (x - d_mean[r])^2 over row r; *d_rowptr = the plan's row pointer
int launch_band_var(sb200_matrix* m, const double* d_mean, double* d_S, const int32_t** d_rowptr);
int launch_band_ptr(sb200_matrix* m, const int32_t* d_rb, int nb, int32_t* d_bpt);
// bmc.cu
int build_band_companion(sb200_matrix* m);  // non-fatal: leaves bmc_state = -1 when it cannot be built
void drop_band_companion(sb200_matrix* m, cudaStream_t s);
int launch_bandsweep(sb200_matrix* m, const double* d_v, double* d_out);  // y[ncol] = A^T v from the companion
int64_t band_companion_bytes(const sb200_matrix* m);                    // HBM the companion occupies (0 without one)
void free_matrix_plans(sb200_matrix* m, cudaStream_t s);
// transpose_split.cu: two stable stream splits (tall matrices)
bool split_transpose_fits(const sb200_matrix* m);
int transpose_split_device(sb200_matrix* m, int32_t* d_p_out, int32_t* d_i_out, double* d_x_out);
void free_split_plan(SplitPlan* sp, cudaStream_t s);
int64_t split_plan_bytes(const SplitPlan* sp);
// hostcopy.cu: copies between host and device memory.  One copy is `runs` runs of `width` bytes, hpitch / dpitch bytes
// apart on the host / the device (runs = 1: a contiguous range).
struct HostCopy {
  void* host;
  void* dev;
  size_t width;
  size_t runs = 1;
  size_t hpitch = 0, dpitch = 0;
  const char* phase = nullptr;  // SB200_TRACE: the WallTrace phase that ends when this copy has arrived
};
// Whether a copy of `bytes` from or to `host` goes through the pinned-chunk workers: large, and in pageable memory (what
// R owns), which the driver would stage through one pinned buffer from one thread.
bool copy_is_staged(const void* host, size_t bytes);
// Copies in one direction between host memory and `device`, for work on stream `st`.  The copies the driver does well
// are enqueued on the stream first; then, if any copy is staged, the stream is synchronised and the staged copies run
// through the pinned-chunk workers.  Returns when the staged copies have arrived; the others are only enqueued.  With a
// trace that is on, the stream is synchronised in any case and reported as `synced`, then every copy's `phase`.
int host_copies(int device, cudaStream_t st, cudaMemcpyKind kind, std::initializer_list<HostCopy> copies, WallTrace* tr = nullptr,
                const char* synced = nullptr);
int launch_crossprod(const sb200_matrix* T, int32_t ncol_a, double* d_res, cudaStream_t st);  // crossprod.cu
// crossprod.cu: slab (ncol x blk->ncol, column-major) = A^T A_blk in ascending row order, on blk's stream; rp / rc / rv are
// the row-ordered copy of the WHOLE matrix (global column ids) on blk's device
int launch_crossprod_slab(const sb200_matrix* blk, const int32_t* rp, const int32_t* rc, const double* rv, int64_t ncol, double* slab);
// capi.cu: the row-ordered copy crossprod runs on, built now if the mirror owns its arrays and has room (null if not)
const sb200_matrix* crossprod_row_copy(sb200_matrix* m);
// spmm.cu: d_Y = A d_B (transposed = false) or A^T d_B, k right-hand sides, both column-major; k = 1 is launch_sweep
int launch_spmm(sb200_matrix* m, bool transposed, const double* d_B, int64_t k, double* d_Y);
// the same up to the final transpose: d_Yrm is ROW-major (y_rows x k); a block without entries or columns gives zeros
int launch_spmm_rm(sb200_matrix* m, bool transposed, const double* d_B, int64_t k, double* d_Yrm);
int build_row_companion(sb200_matrix* m);  // capi.cu; non-fatal: leaves rows_state = -1 when it cannot be built
void drop_row_companion(sb200_matrix* m);
int row_companion_after();                 // SB200_ROW_COMPANION_AFTER (default 8, 0 = never build on its own)

// exchange.cu (single-process form used by sharded.cu)
int exchange_connect_local(sb200_exchange** xs, int world);
unsigned char* exchange_window_base(const sb200_exchange* x);
// mirror.cu
int alloc_matrix(int device, int32_t nrow, int32_t ncol, int64_t nnz, sb200_matrix** out);  // owns arrays, uninitialised
int finish_matrix(sb200_matrix* m, unsigned flags);  // validate + plan + workspace
size_t padded_bytes(size_t bytes);
int pool_alloc(void** out, size_t bytes, cudaStream_t s);  // stream-ordered, from a retaining pool
void pool_free(void* ptr, cudaStream_t s);
size_t pool_idle_bytes(int device);     // freed blocks the library's cache holds on that device (blockcache.cu)
void pool_release_idle(int device);     // hand them back to the driver pool; the device is current and synchronised
size_t device_free_bytes();  // driver-free plus what the pool holds unused

}  // namespace sb200
