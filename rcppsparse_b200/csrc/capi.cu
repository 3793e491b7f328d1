// extern "C" surface of libsparse_b200 (declared in include/sparse_b200.h) and the mirror's lifecycle.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <atomic>
#include <thread>
#include <new>
#include <string>

#include "bandplan.cuh"
#include "common.cuh"

namespace sb200 {

static thread_local std::string t_last_error;
std::atomic<int64_t> g_launches{0};

void set_error(const std::string& msg) { t_last_error = msg; }
int fail(int code, const std::string& msg) {
  t_last_error = msg;
  return code;
}
int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  const char* base = strrchr(file, '/');
  t_last_error = std::string(cudaGetErrorName(e)) + ": " + cudaGetErrorString(e) + " at " + (base ? base + 1 : file) +
                 ":" + std::to_string(line) + " (" + what + ")";
  if (e == cudaErrorMemoryAllocation) return SB200_E_NOMEM;
  if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver || e == cudaErrorInvalidDevice) return SB200_E_NODEVICE;
  return SB200_E_CUDA;
}

size_t padded_bytes(size_t bytes) { return ((bytes + 15) / 16) * 16 + 16; }

static int require_device(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    cudaGetLastError();
    return fail(SB200_E_NODEVICE, "no CUDA device available: libsparse_b200 has no CPU fallback");
  }
  if (device < 0 || device >= n) return fail(SB200_E_NODEVICE, "requested CUDA device " + std::to_string(device) + " not present");
  return SB200_OK;
}

static void free_matrix(sb200_matrix* m) {
  if (!m) return;
  // frees are ordered after the handle's own work; a caller-owned stream may be gone already
  cudaStream_t fs = m->owns_stream ? m->stream : static_cast<cudaStream_t>(0);
  if (!m->owns_stream && m->stream) cudaStreamSynchronize(m->stream), cudaGetLastError();
  if (m->rows) {
    m->rows->stream = m->stream;  // shares the owner's stream (owns_stream == false)
    free_matrix(m->rows);
    m->rows = nullptr;
  }
  if (m->owns_arrays) {
    pool_free(m->d_i, fs);
    pool_free(m->d_p, fs);
    pool_free(m->d_x, fs);
  }
  free_matrix_plans(m, fs);
  drop_band_companion(m, fs);
  pool_free(m->d_plan, fs);
  pool_free(m->d_plan_g, fs);
  pool_free(m->d_ws, fs);
  pool_free(m->d_stage_in, fs);
  pool_free(m->d_stage_out, fs);
  if (m->owns_stream && m->stream) {
    cudaStreamSynchronize(m->stream);
    cudaStreamDestroy(m->stream);
  }
  m->magic = 0;
  delete m;
}

static int new_handle(int device, int32_t nrow, int32_t ncol, int64_t nnz, sb200_matrix** out) {
  if (nrow < 0 || ncol < 0 || nnz < 0) return fail(SB200_E_INVALID, "negative dimension");
  if (nnz > 2147483647LL) return fail(SB200_E_INVALID, "nnz exceeds int32: dgCMatrix p/i are int32 (reference RcppSparse.h:30)");
  SB_TRY(require_device(device));
  sb200_matrix* m = new (std::nothrow) sb200_matrix();
  if (!m) return fail(SB200_E_NOMEM, "host allocation failed");
  memset(m, 0, sizeof(*m));
  m->magic = MATRIX_MAGIC;
  m->row_path = -1;
  m->gather_path = -1;
  m->device = device;
  m->nrow = nrow;
  m->ncol = ncol;
  m->nnz = nnz;
  int sms = 0;
  cudaError_t e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  if (e != cudaSuccess) {
    free_matrix(m);
    return cuda_fail(e, "cudaDeviceGetAttribute", __FILE__, __LINE__);
  }
  m->sm_count = sms;
  e = cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    free_matrix(m);
    return cuda_fail(e, "cudaStreamCreateWithFlags", __FILE__, __LINE__);
  }
  m->owns_stream = true;
  *out = m;
  return SB200_OK;
}

int alloc_matrix(int device, int32_t nrow, int32_t ncol, int64_t nnz, sb200_matrix** out) {
  sb200_matrix* m = nullptr;
  SB_TRY(new_handle(device, nrow, ncol, nnz, &m));
  m->owns_arrays = true;
  int rc = pool_alloc(reinterpret_cast<void**>(&m->d_i), padded_bytes(sizeof(int32_t) * static_cast<size_t>(nnz)), m->stream);
  if (rc == SB200_OK)
    rc = pool_alloc(reinterpret_cast<void**>(&m->d_p), padded_bytes(sizeof(int32_t) * (static_cast<size_t>(ncol) + 1)), m->stream);
  if (rc == SB200_OK)
    rc = pool_alloc(reinterpret_cast<void**>(&m->d_x), padded_bytes(sizeof(double) * static_cast<size_t>(nnz)), m->stream);
  if (rc != SB200_OK) {
    free_matrix(m);
    return rc;
  }
  *out = m;
  return SB200_OK;
}

// Everything the sweeps need besides i/p/x, on the handle's stream: workspace, staging vectors, structure
// check (reads its verdict back, so it waits for p and i), tile plan.  finish_matrix() = this + a stream sync.
static int enqueue_finish(sb200_matrix* m, unsigned flags) {
  m->ws_bytes = 16 + 4 * 1024 + 8 * 1024 + 4 * 1024;  // sweep ticket + carries, then lockstep counters
  SB_TRY(pool_alloc(&m->d_ws, m->ws_bytes, m->stream));
  SB_CUDA(cudaMemsetAsync(m->d_ws, 0, m->ws_bytes, m->stream));
  m->stage_len = (m->nrow > m->ncol ? m->nrow : m->ncol);
  if (m->stage_len < 1) m->stage_len = 1;
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&m->d_stage_in), padded_bytes(sizeof(double) * static_cast<size_t>(m->stage_len)), m->stream));
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&m->d_stage_out), padded_bytes(sizeof(double) * static_cast<size_t>(m->stage_len)), m->stream));
  if (!(flags & SB200_NO_VALIDATE)) SB_TRY(validate_structure(m, m->lazy_i == nullptr));
  SB_TRY(build_sweep_plan(m));
  return SB200_OK;
}

// Free device memory as an allocation from the pool sees it: what the driver reports plus what the pool has
// reserved but is not using (the release threshold keeps freed blocks in the pool).
size_t device_free_bytes() {
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  int dev = 0;
  cudaMemPool_t pool;
  if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
    uint64_t reserved = 0, used = 0;
    if (cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &reserved) == cudaSuccess &&
        cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used) == cudaSuccess && reserved > used)
      free_b += static_cast<size_t>(reserved - used);
    free_b += pool_idle_bytes(dev);  // blocks the library's own cache holds: handed back to the driver when it runs short
  }
  cudaGetLastError();
  return free_b;
}

int row_companion_after() {
  static const int after = [] {
    const char* ev = getenv("SB200_ROW_COMPANION_AFTER");
    return ev ? atoi(ev) : 8;
  }();
  return after;
}

void drop_row_companion(sb200_matrix* m) {
  if (m->rows) {
    m->rows->stream = m->stream;
    free_matrix(m->rows);
    m->rows = nullptr;
  }
  if (m->rows_state == 1) m->rows_state = 0;
  m->row_sum_calls = 0;
}

// Transposed copy on the owner's stream (row pointer, column ids and values in row order, tile plans).  Costs
// one transpose (DESIGN.md 4.3) and 12 B per entry of HBM; skipped when that would not leave room to spare.
// Failure is not the caller's problem: the scatter kernels keep serving the mirror.
int build_row_companion(sb200_matrix* m) {
  if (m->rows_state == 1) return SB200_OK;
  m->rows_state = -1;
  if (m->nnz == 0 || m->nrow == 0) return SB200_OK;
  const size_t need = 12ull * static_cast<size_t>(m->nnz) + 64ull * static_cast<size_t>(m->nrow);
  if (device_free_bytes() < 2 * need) return SB200_OK;  // the copy plus the transpose's own scratch
  const std::string saved = t_last_error;
  sb200_matrix* t = nullptr;
  int rc = alloc_matrix(m->device, m->ncol, m->nrow, m->nnz, &t);
  if (rc == SB200_OK) {
    cudaStreamSynchronize(t->stream);  // its arrays were allocated in that stream's order
    cudaStreamDestroy(t->stream);
    t->stream = m->stream;
    t->owns_stream = false;
    t->rows_state = -1;
    rc = transpose_device(m, t->d_p, t->d_i, t->d_x);
    if (rc == SB200_OK) rc = finish_matrix(t, SB200_NO_VALIDATE);
  }
  if (rc != SB200_OK) {
    if (t) free_matrix(t);
    cudaGetLastError();
    t_last_error = saved;
    return SB200_OK;
  }
  m->rows = t;
  m->rows_state = 1;
  return SB200_OK;
}

const sb200_matrix* crossprod_row_copy(sb200_matrix* m) {
  if (m->owns_arrays && m->rows_state != 1) {
    const int keep = m->rows_state;
    m->rows_state = 0;
    build_row_companion(m);
    if (m->rows_state != 1) m->rows_state = keep;
  }
  if (m->rows_state != 1) return nullptr;
  m->rows->stream = m->stream;
  return m->rows;
}

int finish_matrix(sb200_matrix* m, unsigned flags) {
  SB_TRY(enqueue_finish(m, flags));
  SB_CUDA(cudaStreamSynchronize(m->stream));
  return SB200_OK;
}

// SB200_LAZY_ROWS: the row indices are still in the caller's array.  Bring them over (and check them, unless the mirror
// was created with SB200_NO_VALIDATE) before the first op that reads d_i.  A failed check leaves the mirror as it was:
// the next row-indexed call tries again and fails the same way; the column sweeps keep working, like the reference's
// colSums on a matrix whose `i` is garbage (it never reads it, RcppSparse.h:133-135).
int ensure_rows(sb200_matrix* m) {
  if (!m->lazy_i) return SB200_OK;
  SB_TRY(host_copies(m->device, m->stream, cudaMemcpyHostToDevice,
                     {{const_cast<int32_t*>(m->lazy_i), m->d_i, sizeof(int32_t) * static_cast<size_t>(m->nnz)}}));
  SB_CUDA(cudaStreamSynchronize(m->stream));  // the caller's array is not needed after this call
  if (m->lazy_validate) SB_TRY(validate_rows(m));
  m->lazy_i = nullptr;
  return SB200_OK;
}

}  // namespace sb200

using namespace sb200;

// ENTER_COLS: entry points that never read the row indices (column sweeps, bookkeeping).  ENTER: everything else — a
// mirror created with SB200_LAZY_ROWS gets its `i` now.
#define ENTER_COLS(m)                   \
  SB_TRY(check_handle(m));              \
  DeviceGuard guard_((m)->device);      \
  if (!guard_.ok) return fail(SB200_E_CUDA, "cudaSetDevice failed")
#define ENTER(m)  \
  ENTER_COLS(m);  \
  SB_TRY(ensure_rows(m))

extern "C" {

int sb200_abi_version(void) { return SB200_ABI_VERSION; }
const char* sb200_last_error(void) { return t_last_error.c_str(); }

int sb200_device_count(int* count) {
  if (!count) return fail(SB200_E_INVALID, "count is NULL");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    cudaGetLastError();
    *count = 0;
    return fail(SB200_E_NODEVICE, "no CUDA device available");
  }
  *count = n;
  return SB200_OK;
}

int sb200_trim(int device) {
  SB_TRY(require_device(device));
  DeviceGuard guard(device);
  if (!guard.ok) return fail(SB200_E_CUDA, "cudaSetDevice failed");
  SB_CUDA(cudaDeviceSynchronize());
  pool_release_idle(device);
  SB_CUDA(cudaDeviceSynchronize());
  cudaMemPool_t pool;
  SB_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
  SB_CUDA(cudaMemPoolTrimTo(pool, 0));
  return SB200_OK;
}

int64_t sb200_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int sb200_matrix_create(const int32_t* i, const int32_t* p, const double* x, int32_t nrow, int32_t ncol, int64_t nnz,
                        int device, unsigned flags, sb200_matrix** out) {
  if (!out) return fail(SB200_E_INVALID, "out is NULL");
  *out = nullptr;
  if (!p || (nnz > 0 && (!i || !x))) return fail(SB200_E_INVALID, "NULL slot array");
  SB_TRY(require_device(device));
  DeviceGuard guard(device);
  if (!guard.ok) return fail(SB200_E_CUDA, "cudaSetDevice failed");
  sb200_matrix* m = nullptr;
  SB_TRY(alloc_matrix(device, nrow, ncol, nnz, &m));
  const bool lazy = (flags & SB200_LAZY_ROWS) && nnz > 0;  // `i` stays with the caller until an op reads it
  m->lazy_i = lazy ? i : nullptr;
  m->lazy_validate = !(flags & SB200_NO_VALIDATE);
  const size_t bi = sizeof(int32_t) * static_cast<size_t>(nnz), bp = sizeof(int32_t) * (static_cast<size_t>(ncol) + 1),
               bx = sizeof(double) * static_cast<size_t>(nnz);
  bool pinned_i = false, pinned_x = false;
  if ((flags & SB200_PIN_HOST) && nnz > 0) {
    // R owns these pages; pinning the enclosing pages lets the copy engine stream them directly
    if (!lazy) pinned_i = cudaHostRegister(const_cast<int32_t*>(i), bi, cudaHostRegisterReadOnly) == cudaSuccess;
    if (!lazy && !pinned_i) pinned_i = cudaHostRegister(const_cast<int32_t*>(i), bi, cudaHostRegisterDefault) == cudaSuccess;
    pinned_x = cudaHostRegister(const_cast<double*>(x), bx, cudaHostRegisterReadOnly) == cudaSuccess;
    if (!pinned_x) pinned_x = cudaHostRegister(const_cast<double*>(x), bx, cudaHostRegisterDefault) == cudaSuccess;
    cudaGetLastError();
  }
  // The value array is two thirds of the bytes and nothing at create time reads it: it goes up on a second
  // stream while the structure check, the tile plan and (for matrices that take the banded row path) the row
  // histogram of the band plan run on p and i behind their own, shorter copies.
  const bool trace = getenv("SB200_TRACE") != nullptr;
  const auto t0 = std::chrono::steady_clock::now();
  std::string x_err_text;  // sb200_last_error() is per thread: the values-upload thread reports through this
  // Pageable arrays (what R owns) go through the worker threads of hostcopy.cu; pinned or registered ones are
  // handed to the copy engine directly.
  const bool stage_i = nnz > 0 && !lazy && !pinned_i && copy_is_staged(i, bi);
  const bool stage_x = nnz > 0 && !pinned_x && copy_is_staged(x, bx);
  cudaStream_t xs = nullptr;
  cudaError_t e = cudaStreamCreateWithFlags(&xs, cudaStreamNonBlocking);
  int rc = SB200_OK, rc_x = SB200_OK;
  std::thread x_thread;
  // i/p/x were allocated in m->stream's order; every other stream or thread that writes them waits for that
  if (e == cudaSuccess && (stage_i || stage_x)) {
    e = cudaStreamSynchronize(m->stream);
  } else if (e == cudaSuccess) {
    cudaEvent_t allocated = nullptr;
    e = cudaEventCreateWithFlags(&allocated, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventRecord(allocated, m->stream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(xs, allocated, 0);
    if (allocated) cudaEventDestroy(allocated);
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(m->d_p, p, bp, cudaMemcpyHostToDevice, m->stream);
  if (e == cudaSuccess && nnz > 0 && !lazy) rc = host_copies(device, m->stream, cudaMemcpyHostToDevice, {{const_cast<int32_t*>(i), m->d_i, bi}});
  if (e == cudaSuccess && rc == SB200_OK && nnz > 0) {
    if (stage_x) {
      x_thread = std::thread([&] {
        rc_x = host_copies(device, xs, cudaMemcpyHostToDevice, {{const_cast<double*>(x), m->d_x, bx}});
        if (rc_x != SB200_OK) x_err_text = sb200_last_error();
      });
    } else {
      e = cudaMemcpyAsync(m->d_x, x, bx, cudaMemcpyHostToDevice, xs);
    }
  }
  if (e == cudaSuccess && rc == SB200_OK) rc = enqueue_finish(m, flags);
  if (e == cudaSuccess && rc == SB200_OK && nnz > 0 && m->nrow > 0 && !lazy && !(flags & SB200_NO_ROW_PLAN)) {
    // plan failures here are not fatal: the row sweeps retry (or fall back to the L2 path) on first use
    const std::string keep = t_last_error;
    if (decide_row_path(m) == SB200_OK && m->row_path == 1) ensure_scatter_plan(m);
    t_last_error = keep;
  }
  const auto t1 = std::chrono::steady_clock::now();
  if (e == cudaSuccess) e = cudaStreamSynchronize(m->stream);
  const auto t2 = std::chrono::steady_clock::now();
  if (x_thread.joinable()) x_thread.join();
  if (rc == SB200_OK && rc_x != SB200_OK) {
    rc = rc_x;
    set_error(x_err_text);
  }
  if (xs) {
    const cudaError_t ex = cudaStreamSynchronize(xs);
    if (e == cudaSuccess) e = ex;
    cudaStreamDestroy(xs);
  }
  if (pinned_i) cudaHostUnregister(const_cast<int32_t*>(i));
  if (pinned_x) cudaHostUnregister(const_cast<double*>(x));
  if (trace) {
    const auto t3 = std::chrono::steady_clock::now();
    auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
    fprintf(stderr, "[sb200 trace] create: enqueue %.2f ms; structure stream %.2f ms; values %.2f ms\n", ms(t0, t1), ms(t1, t2), ms(t2, t3));
  }
  if (e != cudaSuccess) {
    free_matrix(m);
    return cuda_fail(e, "upload of i/p/x", __FILE__, __LINE__);
  }
  if (rc != SB200_OK) {
    free_matrix(m);
    return rc;
  }
  *out = m;
  return SB200_OK;
}

int sb200_matrix_adopt_device(const int32_t* d_i, const int32_t* d_p, const double* d_x, int32_t nrow, int32_t ncol,
                              int64_t nnz, int device, unsigned flags, sb200_matrix** out) {
  if (!out) return fail(SB200_E_INVALID, "out is NULL");
  *out = nullptr;
  if (!d_p || (nnz > 0 && (!d_i || !d_x))) return fail(SB200_E_INVALID, "NULL device array");
  if ((reinterpret_cast<uintptr_t>(d_i) | reinterpret_cast<uintptr_t>(d_p) | reinterpret_cast<uintptr_t>(d_x)) & 15)
    return fail(SB200_E_INVALID, "device arrays must be 16-byte aligned");
  SB_TRY(require_device(device));
  DeviceGuard guard(device);
  if (!guard.ok) return fail(SB200_E_CUDA, "cudaSetDevice failed");
  sb200_matrix* m = nullptr;
  SB_TRY(new_handle(device, nrow, ncol, nnz, &m));
  m->owns_arrays = false;
  m->d_i = const_cast<int32_t*>(d_i);
  m->d_p = const_cast<int32_t*>(d_p);
  m->d_x = const_cast<double*>(d_x);
  const int rc = finish_matrix(m, flags);
  if (rc != SB200_OK) {
    free_matrix(m);
    return rc;
  }
  *out = m;
  return SB200_OK;
}

int sb200_matrix_destroy(sb200_matrix* m) {
  if (!m) return SB200_OK;
  SB_TRY(check_handle(m));
  DeviceGuard guard(m->device);
  if (m->stream) cudaStreamSynchronize(m->stream);
  free_matrix(m);
  return SB200_OK;
}

int sb200_matrix_dims(const sb200_matrix* m, int32_t* nrow, int32_t* ncol, int64_t* nnz) {
  SB_TRY(check_handle(m));
  if (nrow) *nrow = m->nrow;
  if (ncol) *ncol = m->ncol;
  if (nnz) *nnz = m->nnz;
  return SB200_OK;
}

int sb200_matrix_refresh_values(sb200_matrix* m, const double* x) {
  ENTER_COLS(m);
  if (m->nnz == 0) return SB200_OK;
  if (!x) return fail(SB200_E_INVALID, "x is NULL");
  drop_row_companion(m);  // its values are the old ones; the call count starts over
  drop_band_companion(m, m->stream);
  SB_TRY(host_copies(m->device, m->stream, cudaMemcpyHostToDevice,
                     {{const_cast<double*>(x), m->d_x, sizeof(double) * static_cast<size_t>(m->nnz)}}));
  SB_CUDA(cudaStreamSynchronize(m->stream));
  return SB200_OK;
}

int sb200_matrix_set_stream(sb200_matrix* m, void* cuda_stream) {
  ENTER_COLS(m);
  SB_CUDA(cudaStreamSynchronize(m->stream));
  if (m->owns_stream && m->stream) cudaStreamDestroy(m->stream);
  m->stream = static_cast<cudaStream_t>(cuda_stream);
  m->owns_stream = false;
  return SB200_OK;
}

int sb200_matrix_sync(sb200_matrix* m) {
  ENTER_COLS(m);
  SB_CUDA(cudaStreamSynchronize(m->stream));
  return SB200_OK;
}

int sb200_matrix_device_arrays(const sb200_matrix* m, const int32_t** d_i, const int32_t** d_p, const double** d_x) {
  SB_TRY(check_handle(m));
  if (d_i && m->lazy_i) {  // the caller is about to read the row indices on the device
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(SB200_E_CUDA, "cudaSetDevice failed");
    SB_TRY(ensure_rows(const_cast<sb200_matrix*>(m)));
  }
  if (d_i) *d_i = m->d_i;
  if (d_p) *d_p = m->d_p;
  if (d_x) *d_x = m->d_x;
  return SB200_OK;
}

// ---- device-buffer form ---------------------------------------------------------------------------------
int sb200_col_sums_dev(sb200_matrix* m, double divisor, double* d_out) {
  ENTER_COLS(m);
  if (m->ncol > 0 && !d_out) return fail(SB200_E_INVALID, "d_out is NULL");
  return launch_sweep(m, SWEEP_COLSUM, nullptr, divisor, d_out);
}
int sb200_row_sums_dev(sb200_matrix* m, double divisor, double* d_out) {
  ENTER(m);
  if (m->nrow > 0 && !d_out) return fail(SB200_E_INVALID, "d_out is NULL");
  return launch_sweep(m, SWEEP_ROWSUM, nullptr, divisor, d_out);
}
int sb200_spmv_dev(sb200_matrix* m, const double* d_v, double* d_y) {
  ENTER(m);
  if ((m->ncol > 0 && !d_v) || (m->nrow > 0 && !d_y)) return fail(SB200_E_INVALID, "NULL operand");
  return launch_sweep(m, SWEEP_SPMV, d_v, 0.0, d_y);
}
int sb200_spmv_t_dev(sb200_matrix* m, const double* d_v, double* d_y) {
  ENTER(m);
  if ((m->nrow > 0 && !d_v) || (m->ncol > 0 && !d_y)) return fail(SB200_E_INVALID, "NULL operand");
  return launch_sweep(m, SWEEP_SPMV_T, d_v, 0.0, d_y);
}
int sb200_col_vars_dev(sb200_matrix* m, double* d_out) {
  ENTER_COLS(m);
  if (m->ncol > 0 && !d_out) return fail(SB200_E_INVALID, "d_out is NULL");
  return launch_col_vars(m, d_out);
}
int sb200_row_vars_dev(sb200_matrix* m, double* d_out) {
  ENTER(m);
  if (m->nrow > 0 && !d_out) return fail(SB200_E_INVALID, "d_out is NULL");
  return launch_row_vars(m, d_out);
}
int sb200_vec_div_dev(sb200_matrix* m, double* d, int64_t n, double divisor) {
  ENTER_COLS(m);
  return launch_vec_div(m->stream, d, n, divisor);
}

int sb200_transpose_dev(sb200_matrix* m, sb200_matrix** out) {
  if (!out) return fail(SB200_E_INVALID, "out is NULL");
  *out = nullptr;
  ENTER(m);
  sb200_matrix* t = nullptr;
  SB_TRY(alloc_matrix(m->device, m->ncol, m->nrow, m->nnz, &t));
  cudaStreamSynchronize(t->stream);  // t's arrays were allocated in its own stream's order, written in m's
  int rc = transpose_device(m, t->d_p, t->d_i, t->d_x);
  if (rc == SB200_OK) rc = cudaStreamSynchronize(m->stream) == cudaSuccess ? SB200_OK : fail(SB200_E_CUDA, "transpose: stream sync failed");
  // the result is canonical by construction; skip re-validation
  if (rc == SB200_OK) rc = finish_matrix(t, SB200_NO_VALIDATE);
  if (rc != SB200_OK) {
    cudaStreamSynchronize(m->stream);  // kernels on m's stream may still be writing t's arrays
    cudaGetLastError();
    free_matrix(t);
    return rc;
  }
  *out = t;
  return SB200_OK;
}

int sb200_transpose_into(sb200_matrix* m, sb200_matrix* t) {
  ENTER(m);
  SB_TRY(check_handle(t));
  if (t == m || !t->owns_arrays || t->device != m->device || t->nrow != m->ncol || t->ncol != m->nrow || t->nnz != m->nnz)
    return fail(SB200_E_INVALID, "transpose_into: the target is not a transpose of this shape that owns its arrays");
  // t's own work first (its stream may differ from m's), then the kernels on m's stream write its arrays
  if (t->stream != m->stream && cudaStreamSynchronize(t->stream) != cudaSuccess) return fail(SB200_E_CUDA, "transpose_into: stream sync failed");
  drop_row_companion(t);
  drop_band_companion(t, t->stream);
  int rc = transpose_device(m, t->d_p, t->d_i, t->d_x);
  if (cudaStreamSynchronize(m->stream) != cudaSuccess && rc == SB200_OK) rc = fail(SB200_E_CUDA, "transpose_into: stream sync failed");
  return rc;
}

// ---- host-buffer form: stage through the handle's device buffers ---------------------------------------------
static int run_to_host(sb200_matrix* m, SweepMode mode, const double* v_host, int64_t v_len, double divisor,
                       double* out_host, int64_t out_len) {
  if (out_len > 0 && !out_host) return fail(SB200_E_INVALID, "output buffer is NULL");
  if (v_len > 0) {
    if (!v_host) return fail(SB200_E_INVALID, "operand vector is NULL");
    SB_CUDA(cudaMemcpyAsync(m->d_stage_in, v_host, sizeof(double) * static_cast<size_t>(v_len), cudaMemcpyHostToDevice,
                            m->stream));
  }
  SB_TRY(launch_sweep(m, mode, m->d_stage_in, divisor, m->d_stage_out));
  if (out_len > 0)
    SB_CUDA(cudaMemcpyAsync(out_host, m->d_stage_out, sizeof(double) * static_cast<size_t>(out_len),
                            cudaMemcpyDeviceToHost, m->stream));
  SB_CUDA(cudaStreamSynchronize(m->stream));
  return SB200_OK;
}

int sb200_col_sums(sb200_matrix* m, double* out) {
  ENTER_COLS(m);
  return run_to_host(m, SWEEP_COLSUM, nullptr, 0, 0.0, out, m->ncol);
}
int sb200_row_sums(sb200_matrix* m, double* out) {
  ENTER(m);
  return run_to_host(m, SWEEP_ROWSUM, nullptr, 0, 0.0, out, m->nrow);
}
int sb200_col_means(sb200_matrix* m, double* out) {
  ENTER_COLS(m);
  // RcppSparse.h:148: sums[i] / Dim[0]; Dim[0] == 0 gives 0/0 = NaN there and here
  if (m->nrow == 0) {
    for (int32_t c = 0; c < m->ncol; ++c) out[c] = 0.0 / static_cast<double>(m->nrow);
    return SB200_OK;
  }
  return run_to_host(m, SWEEP_COLSUM, nullptr, 0, static_cast<double>(m->nrow), out, m->ncol);
}
int sb200_row_means(sb200_matrix* m, double* out) {
  ENTER(m);
  if (m->ncol == 0) {
    for (int32_t r = 0; r < m->nrow; ++r) out[r] = 0.0 / static_cast<double>(m->ncol);
    return SB200_OK;
  }
  return run_to_host(m, SWEEP_ROWSUM, nullptr, 0, static_cast<double>(m->ncol), out, m->nrow);
}
int sb200_col_vars(sb200_matrix* m, double* out) {
  ENTER_COLS(m);
  return run_to_host(m, SWEEP_COLVAR, nullptr, 0, 0.0, out, m->ncol);
}
int sb200_row_vars(sb200_matrix* m, double* out) {
  ENTER(m);
  return run_to_host(m, SWEEP_ROWVAR, nullptr, 0, 0.0, out, m->nrow);
}
int sb200_spmv(sb200_matrix* m, const double* v, double* y) {
  ENTER(m);
  return run_to_host(m, SWEEP_SPMV, v, m->ncol, 0.0, y, m->nrow);
}
int sb200_spmv_t(sb200_matrix* m, const double* v, double* y) {
  ENTER(m);
  return run_to_host(m, SWEEP_SPMV_T, v, m->nrow, 0.0, y, m->ncol);
}

int sb200_transpose(sb200_matrix* m, int32_t* p_out, int32_t* i_out, double* x_out) {
  ENTER(m);
  if (!p_out || (m->nnz > 0 && (!i_out || !x_out))) return fail(SB200_E_INVALID, "NULL output array");
  WallTrace tr("transpose to host");
  sb200_matrix* t = nullptr;
  SB_TRY(alloc_matrix(m->device, m->ncol, m->nrow, m->nnz, &t));
  cudaStreamSynchronize(t->stream);  // t's arrays were allocated in its own stream's order, written in m's
  tr.phase("result allocated");
  int rc = transpose_device(m, t->d_p, t->d_i, t->d_x);
  cudaError_t e = cudaSuccess;
  if (rc == SB200_OK) {
    const size_t bi = sizeof(int32_t) * static_cast<size_t>(m->nnz), bx = sizeof(double) * static_cast<size_t>(m->nnz);
    e = cudaMemcpyAsync(p_out, t->d_p, sizeof(int32_t) * (static_cast<size_t>(m->nrow) + 1), cudaMemcpyDeviceToHost, m->stream);
    // the result goes back into the caller's (R-allocated, pageable) vectors: large ones through the pinned-chunk workers,
    // once the transposed arrays are complete
    if (e == cudaSuccess)
      rc = host_copies(m->device, m->stream, cudaMemcpyDeviceToHost,
                       {{i_out, t->d_i, bi, 1, 0, 0, "i' to the host"}, {x_out, t->d_x, bx, 1, 0, 0, "x' to the host"}}, &tr,
                       "transposed on the device (plan + kernels, p' copied)");
    if (e == cudaSuccess && rc == SB200_OK) e = cudaStreamSynchronize(m->stream);
  }
  if (rc != SB200_OK || e != cudaSuccess) {
    cudaStreamSynchronize(m->stream);  // nothing on m's stream still touches t's arrays when they are freed
    cudaGetLastError();
  }
  free_matrix(t);
  tr.phase("result freed");
  if (rc != SB200_OK) return rc;
  if (e != cudaSuccess) return cuda_fail(e, "download of the transposed matrix", __FILE__, __LINE__);
  return SB200_OK;
}

// ---- sparse x dense block (spmm.cu) -------------------------------------------------------------------------
// Arguments of the four spmm entry points.  k = 0 is an empty result: it reads nothing (not even a lazily kept `i`)
// and launches nothing.
static int spmm_args(const sb200_matrix* m, bool transposed, const void* B, int64_t k, const void* Y) {
  if (k < 0) return fail(SB200_E_INVALID, "spmm: k must not be negative");
  const int64_t b_rows = transposed ? m->nrow : m->ncol, y_rows = transposed ? m->ncol : m->nrow;
  if (k > 0 && ((b_rows > 0 && !B) || (y_rows > 0 && !Y))) return fail(SB200_E_INVALID, "spmm: NULL operand or result");
  return SB200_OK;
}

static int spmm_to_host(sb200_matrix* m, bool transposed, const double* B, int64_t k, double* Y) {
  const int64_t b_rows = transposed ? m->nrow : m->ncol, y_rows = transposed ? m->ncol : m->nrow;
  if (k == 1) return run_to_host(m, transposed ? SWEEP_SPMV_T : SWEEP_SPMV, B, b_rows, 0.0, Y, y_rows);
  if ((b_rows > 0 && k > INT64_MAX / 8 / b_rows) || (y_rows > 0 && k > INT64_MAX / 8 / y_rows))
    return fail(SB200_E_NOMEM, "spmm: the dense operand or result does not fit in device memory");
  const size_t b_bytes = sizeof(double) * static_cast<size_t>(b_rows * k), y_bytes = sizeof(double) * static_cast<size_t>(y_rows * k);
  double *d_B = nullptr, *d_Y = nullptr;
  int rc = pool_alloc(reinterpret_cast<void**>(&d_B), b_bytes > 0 ? b_bytes : 16, m->stream);
  if (rc == SB200_OK) rc = pool_alloc(reinterpret_cast<void**>(&d_Y), y_bytes > 0 ? y_bytes : 16, m->stream);
  // R's matrices are pageable: large ones go through the pinned-chunk workers
  if (rc == SB200_OK) rc = host_copies(m->device, m->stream, cudaMemcpyHostToDevice, {{const_cast<double*>(B), d_B, b_bytes}});
  if (rc == SB200_OK) rc = launch_spmm(m, transposed, d_B, k, d_Y);
  if (rc == SB200_OK) rc = host_copies(m->device, m->stream, cudaMemcpyDeviceToHost, {{Y, d_Y, y_bytes}});
  const cudaError_t es = cudaStreamSynchronize(m->stream);
  if (rc == SB200_OK && es != cudaSuccess) rc = cuda_fail(es, "spmm: stream sync", __FILE__, __LINE__);
  if (rc == SB200_E_NOMEM) cudaGetLastError();
  pool_free(d_B, m->stream);
  pool_free(d_Y, m->stream);
  return rc;
}

// ---- crossprod (dense A^T A) -------------------------------------------------------------------------------
// Runs on the row-ordered copy: the cached one of a mirror that owns its arrays (built now if need be), a
// temporary one otherwise (adopted arrays: the caller may have changed the values since any earlier copy).
static int crossprod_into(sb200_matrix* m, double* d_res) {
  if (m->nnz == 0 || m->nrow == 0) {  // no products at all: the result is the zero matrix
    if (m->ncol > 0)
      SB_CUDA(cudaMemsetAsync(d_res, 0, sizeof(double) * static_cast<size_t>(m->ncol) * static_cast<size_t>(m->ncol), m->stream));
    return SB200_OK;
  }
  if (const sb200_matrix* rows = crossprod_row_copy(m)) return launch_crossprod(rows, m->ncol, d_res, m->stream);
  sb200_matrix* t = nullptr;
  SB_TRY(alloc_matrix(m->device, m->ncol, m->nrow, m->nnz, &t));
  cudaStreamSynchronize(t->stream);
  int rc = transpose_device(m, t->d_p, t->d_i, t->d_x);
  if (rc == SB200_OK) {
    t->sm_count = m->sm_count;
    rc = launch_crossprod(t, m->ncol, d_res, m->stream);
  }
  if (cudaStreamSynchronize(m->stream) != cudaSuccess && rc == SB200_OK) rc = fail(SB200_E_CUDA, "crossprod: stream sync failed");
  free_matrix(t);
  return rc;
}

int sb200_crossprod_dev(sb200_matrix* m, double* d_out) {
  ENTER(m);
  if (m->ncol > 0 && !d_out) return fail(SB200_E_INVALID, "d_out is NULL");
  return crossprod_into(m, d_out);
}

int sb200_crossprod(sb200_matrix* m, double* out) {
  ENTER(m);
  if (m->ncol == 0) return SB200_OK;
  if (!out) return fail(SB200_E_INVALID, "output buffer is NULL");
  const size_t bytes = sizeof(double) * static_cast<size_t>(m->ncol) * static_cast<size_t>(m->ncol);
  double* d_res = nullptr;
  if (pool_alloc(reinterpret_cast<void**>(&d_res), bytes, m->stream) != SB200_OK) {
    cudaGetLastError();
    return fail(SB200_E_NOMEM, "crossprod: the dense ncol x ncol result does not fit on the device");
  }
  int rc = crossprod_into(m, d_res);
  if (rc == SB200_OK) {
    cudaError_t e = cudaMemcpyAsync(out, d_res, bytes, cudaMemcpyDeviceToHost, m->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(m->stream);
    if (e != cudaSuccess) rc = cuda_fail(e, "crossprod: result copy", __FILE__, __LINE__);
  }
  pool_free(d_res, m->stream);
  return rc;
}

int sb200_spmm(sb200_matrix* m, const double* B, int64_t k, double* Y) {
  ENTER_COLS(m);
  SB_TRY(spmm_args(m, false, B, k, Y));
  if (k == 0) return SB200_OK;
  SB_TRY(ensure_rows(m));
  return spmm_to_host(m, false, B, k, Y);
}
int sb200_spmm_t(sb200_matrix* m, const double* B, int64_t k, double* Y) {
  ENTER_COLS(m);
  SB_TRY(spmm_args(m, true, B, k, Y));
  if (k == 0) return SB200_OK;
  SB_TRY(ensure_rows(m));
  return spmm_to_host(m, true, B, k, Y);
}
int sb200_spmm_dev(sb200_matrix* m, const double* d_B, int64_t k, double* d_Y) {
  ENTER_COLS(m);
  SB_TRY(spmm_args(m, false, d_B, k, d_Y));
  if (k == 0) return SB200_OK;
  SB_TRY(ensure_rows(m));
  return launch_spmm(m, false, d_B, k, d_Y);
}
int sb200_spmm_t_dev(sb200_matrix* m, const double* d_B, int64_t k, double* d_Y) {
  ENTER_COLS(m);
  SB_TRY(spmm_args(m, true, d_B, k, d_Y));
  if (k == 0) return SB200_OK;
  SB_TRY(ensure_rows(m));
  return launch_spmm(m, true, d_B, k, d_Y);
}

int sb200_matrix_row_path(sb200_matrix* m, int* banded) {
  ENTER(m);
  if (!banded) return fail(SB200_E_INVALID, "banded is NULL");
  SB_TRY(decide_row_path(m));
  *banded = m->rows_state == 1 ? 2 : m->row_path;
  return SB200_OK;
}

int sb200_matrix_row_companion(sb200_matrix* m, int action) {
  ENTER(m);
  if (action > 0) {
    if (m->rows_state != 1) {
      m->rows_state = 0;
      SB_TRY(build_row_companion(m));
    }
    if (m->rows_state != 1 && m->nnz > 0 && m->nrow > 0)
      return fail(SB200_E_NOMEM, "row companion could not be built (memory, or the transpose does not support this shape)");
    return SB200_OK;
  }
  drop_row_companion(m);
  m->rows_state = action < 0 ? -1 : 0;
  return SB200_OK;
}

int sb200_matrix_band_companion(sb200_matrix* m, int which, int action) {
  ENTER(m);
  if (which != 0 && which != 1) return fail(SB200_E_INVALID, "which must be 0 (A^T v) or 1 (A v)");
  sb200_matrix* t = m;
  if (which == 1) {  // A v runs on the row-ordered copy: that copy's own companion
    if (action > 0 && m->rows_state != 1) {
      m->rows_state = 0;
      SB_TRY(build_row_companion(m));
    }
    if (m->rows_state != 1) {
      if (action > 0 && m->nnz > 0 && m->nrow > 0)
        return fail(SB200_E_NOMEM, "row companion could not be built (memory, or the transpose does not support this shape)");
      return SB200_OK;
    }
    t = m->rows;
    t->stream = m->stream;
  }
  if (action > 0) {
    if (t->bmc_state != 1) {
      t->bmc_state = 0;
      SB_TRY(build_band_companion(t));
    }
    if (t->bmc_state != 1 && t->nnz > 0 && t->nrow > 0 && t->ncol > 0)
      return fail(SB200_E_NOMEM, "band-major companion could not be built (memory, or too many (band, column) runs)");
    return SB200_OK;
  }
  drop_band_companion(t, m->stream);
  t->bmc_state = action < 0 ? -1 : 0;
  return SB200_OK;
}

int sb200_matrix_layouts(sb200_matrix* m, int* mask) {
  ENTER_COLS(m);
  if (!mask) return fail(SB200_E_INVALID, "mask is NULL");
  *mask = (m->rows_state == 1 ? 1 : 0) | (m->bmc_state == 1 ? 2 : 0) |
          ((m->rows_state == 1 && m->rows && m->rows->bmc_state == 1) ? 4 : 0) | ((m->plan_transpose || m->plan_split) ? 8 : 0);
  return SB200_OK;
}

int sb200_matrix_layout_bytes(sb200_matrix* m, int64_t* bytes) {
  ENTER_COLS(m);
  if (!bytes) return fail(SB200_E_INVALID, "bytes is NULL");
  int64_t total = band_companion_bytes(m);
  if (m->rows_state == 1 && m->rows) {
    total += 12 * m->rows->nnz + 4 * (static_cast<int64_t>(m->rows->ncol) + 1);  // row-ordered copy: x', i', p'
    total += band_companion_bytes(m->rows);
  }
  // transpose plans kept between calls (structure only): band pointers + per-(row, split) offsets, or the destination
  // tables of the two stream splits
  total += split_plan_bytes(m->plan_split);
  if (const BandPlan* bp = m->plan_transpose) {
    total += 4 * (static_cast<int64_t>(bp->nb > 0 ? bp->nb - 1 : 0) * m->ncol + static_cast<int64_t>(m->nrow) * bp->S + 1 + bp->nb + 1 + bp->S + 1);
    if (bp->S > 1) total += 4 * (static_cast<int64_t>(m->nrow) + 1);
  }
  *bytes = total;
  return SB200_OK;
}

int sb200_algorithmic_bytes(const sb200_matrix* m, const char* op, int64_t* bytes) {
  SB_TRY(check_handle(m));
  if (!op || !bytes) return fail(SB200_E_INVALID, "NULL argument");
  const int64_t N = m->nnz, n = m->ncol, r = m->nrow;
  const std::string s(op);
  // SURVEY.md section 8(d): compulsory traffic only — every array once, the output once
  if (s == "col_sums" || s == "col_means" || s == "col_vars")  // colVars: the two passes read x twice (16N + ...)
    *bytes = 8 * N + 4 * (n + 1) + 8 * n;
  else if (s == "row_sums" || s == "row_means" || s == "row_vars")
    *bytes = 12 * N + 8 * r;
  else if (s == "row_sums_companion" || s == "row_means_companion")  // row-ordered x once, row pointer, output
    *bytes = 8 * N + 4 * (r + 1) + 8 * r;
  else if (s == "spmv" || s == "spmv_t")
    *bytes = 12 * N + 4 * (n + 1) + 8 * n + 8 * r;
  else if (s == "transpose")
    *bytes = 24 * N + 4 * (n + 1) + 4 * (r + 1);
  else
    return fail(SB200_E_INVALID, "unknown op '" + s + "'");
  return SB200_OK;
}

int sb200_matrix_download_columns(sb200_matrix* m, int64_t c0, int64_t c1, int32_t* i_out, int32_t* p_out, double* x_out,
                                  int64_t* nnz_out) {
  ENTER(m);
  if (c0 < 0 || c1 < c0 || c1 > m->ncol) return fail(SB200_E_INVALID, "column range outside the matrix");
  int32_t ends[2] = {0, 0};
  SB_CUDA(cudaMemcpyAsync(&ends[0], m->d_p + c0, sizeof(int32_t), cudaMemcpyDeviceToHost, m->stream));
  SB_CUDA(cudaMemcpyAsync(&ends[1], m->d_p + c1, sizeof(int32_t), cudaMemcpyDeviceToHost, m->stream));
  SB_CUDA(cudaStreamSynchronize(m->stream));
  const int64_t k0 = ends[0], k1 = ends[1];
  if (nnz_out) *nnz_out = k1 - k0;
  if (!i_out) return SB200_OK;  // size query
  if (!p_out || !x_out) return fail(SB200_E_INVALID, "NULL output array");
  SB_CUDA(cudaMemcpyAsync(p_out, m->d_p + c0, sizeof(int32_t) * static_cast<size_t>(c1 - c0 + 1), cudaMemcpyDeviceToHost, m->stream));
  if (k1 > k0) {
    SB_CUDA(cudaMemcpyAsync(i_out, m->d_i + k0, sizeof(int32_t) * static_cast<size_t>(k1 - k0), cudaMemcpyDeviceToHost, m->stream));
    SB_CUDA(cudaMemcpyAsync(x_out, m->d_x + k0, sizeof(double) * static_cast<size_t>(k1 - k0), cudaMemcpyDeviceToHost, m->stream));
  }
  SB_CUDA(cudaStreamSynchronize(m->stream));
  for (int64_t c = 0; c <= c1 - c0; ++c) p_out[c] -= static_cast<int32_t>(k0);
  return SB200_OK;
}

}  // extern "C"
