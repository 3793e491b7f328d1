// colVars / rowVars: the sample variance of every column or row of the dgCMatrix, its implicit zeros included, over
// n - 1 (R's var(A[, c]) and var(A[r, ])), in two passes.
//
// Pass 1 is colMeans / rowMeans exactly (the same sweep and the same IEEE division), so the mean m used is theirs bit
// for bit.  Pass 2 sums S = sum over the stored entries of (x - m)^2, and the result is var_from_sums (common.cuh):
// (S + (n - cnt) m^2) / (n - 1), cnt = the stored entries of the column or row.  The one-pass sum(x^2)/n - m^2 (or its
// rewrite sum x (x - 2m) + n m^2) cancels catastrophically on nearly constant data, and a running (Welford) mean puts
// its own rounding into every term; two passes read x twice instead.
//
//   colVars               pass 2 = sweep_kernel<SWEEP_COLVAR> (sweep.cu), the formula applied at the column's store
//   rowVars, row copy     the same two passes on the mirror's row-ordered copy (where rowSums runs as a column sweep)
//   rowVars, CSC arrays   pass 1 = rowMeans on the path rowSums takes.  Pass 2 on the same path: band_var_kernel
//                         (bands.cu: the band's slice of the means in shared memory beside its accumulators, the counts
//                         from the band plan's row pointer) or rowvar_stream_kernel (L2 reductions of (x - m)^2 and of
//                         the counts); then var_finish_kernel.
// NaN or Inf among the entries of a column or row make its mean non-finite and its variance NaN, and nothing else.
// n < 2 gives NaN everywhere (R gives NA).
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"
#include "ptx.cuh"

namespace sb200 {
namespace {

__global__ void fill_nan_kernel(double* __restrict__ d, int64_t n) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; k < n; k += stride)
    d[k] = __longlong_as_double(0x7ff8000000000000LL);
}

// rowvar_stream_kernel: rowsum_stream_kernel (sweep.cu) for the second pass — S[i] += (x - mean[i])^2 and cnt[i] += 1
// as FP64 reductions at L2.  The means of a group's rows are gathered before its reductions are fired.
template <int THREADS, int UNROLL>
__global__ void __launch_bounds__(THREADS) rowvar_stream_kernel(const int32_t* __restrict__ gi, const double* __restrict__ gx,
                                                                int64_t nnz, const double* __restrict__ mean,
                                                                double* __restrict__ S, double* __restrict__ cnt) {
  const int64_t n4 = nnz >> 2;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * THREADS;
  const int4* __restrict__ i4 = reinterpret_cast<const int4*>(gi);
  const double2* __restrict__ x2 = reinterpret_cast<const double2*>(gx);
  auto add = [&](int32_t r, double x, double m) {
    const double d = __dsub_rn(x, m);
    ptx::red_add_f64(S + r, __dmul_rn(d, d));
    ptx::red_add_f64(cnt + r, 1.0);
  };
  int64_t g = static_cast<int64_t>(blockIdx.x) * THREADS + threadIdx.x;
  for (; g + (UNROLL - 1) * stride < n4; g += UNROLL * stride) {
    int4 r[UNROLL];
    double2 a[UNROLL], b[UNROLL];
    double mu[UNROLL][4];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      r[u] = ptx::ld_stream_v4s32(i4 + g + u * stride);
      a[u] = ptx::ld_stream_v2f64(x2 + 2 * (g + u * stride));
      b[u] = ptx::ld_stream_v2f64(x2 + 2 * (g + u * stride) + 1);
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      mu[u][0] = __ldg(mean + r[u].x);
      mu[u][1] = __ldg(mean + r[u].y);
      mu[u][2] = __ldg(mean + r[u].z);
      mu[u][3] = __ldg(mean + r[u].w);
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      add(r[u].x, a[u].x, mu[u][0]);
      add(r[u].y, a[u].y, mu[u][1]);
      add(r[u].z, b[u].x, mu[u][2]);
      add(r[u].w, b[u].y, mu[u][3]);
    }
  }
  for (; g < n4; g += stride) {
    const int4 r = ptx::ld_stream_v4s32(i4 + g);
    const double2 a = ptx::ld_stream_v2f64(x2 + 2 * g);
    const double2 b = ptx::ld_stream_v2f64(x2 + 2 * g + 1);
    const double m0 = __ldg(mean + r.x), m1 = __ldg(mean + r.y), m2 = __ldg(mean + r.z), m3 = __ldg(mean + r.w);
    add(r.x, a.x, m0);
    add(r.y, a.y, m1);
    add(r.z, b.x, m2);
    add(r.w, b.y, m3);
  }
  // tail (nnz % 4 entries)
  const int64_t k = (n4 << 2) + static_cast<int64_t>(blockIdx.x) * THREADS + threadIdx.x;
  if (k < nnz) add(gi[k], gx[k], __ldg(mean + gi[k]));
}

// cnt[r] = ptr[r + 1] - ptr[r]: a row pointer's counts as doubles (the sharded reduce sums them)
__global__ void row_counts_kernel(const int32_t* __restrict__ ptr, int64_t n, double* __restrict__ cnt) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < n; r += stride)
    cnt[r] = static_cast<double>(ptr[r + 1] - ptr[r]);
}

// out[r] = var_from_sums(out[r], count of row r, mean[r], n); the count from the row pointer `ptr` when it is set,
// from `cnt` otherwise
__global__ void var_finish_kernel(double* __restrict__ out, const double* __restrict__ mean, const int32_t* __restrict__ ptr,
                                  const double* __restrict__ cnt, int64_t len, double n) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < len; r += stride) {
    const double c = ptr ? static_cast<double>(ptr[r + 1] - ptr[r]) : cnt[r];
    out[r] = var_from_sums(out[r], c, mean[r], n);
  }
}

unsigned elementwise_blocks(int64_t n) {
  int64_t blocks = (n + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  return static_cast<unsigned>(blocks);
}

// rowVars' second pass on the CSC arrays, on the path decide_row_path chose for rowSums (and, like rowSums, on the L2
// kernel when no band plan can be built for the shape).  *d_rowptr = the band plan's row pointer on the banded path
// (the counts are its differences), null on the L2 path, which counts into d_cnt.
int row_var_csc(sb200_matrix* m, const double* d_mean, double* d_S, double* d_cnt, const int32_t** d_rowptr) {
  *d_rowptr = nullptr;
  SB_TRY(decide_row_path(m));
  if (m->row_path == 1) {
    const int rc = launch_band_var(m, d_mean, d_S, d_rowptr);
    if (rc == SB200_OK) return SB200_OK;
    if (rc != SB200_E_UNSUPPORTED && rc != SB200_E_NOMEM) return rc;
    cudaGetLastError();
    m->row_path = 0;
  }
  const size_t bytes = sizeof(double) * static_cast<size_t>(m->nrow);
  SB_CUDA(cudaMemsetAsync(d_S, 0, bytes, m->stream));
  SB_CUDA(cudaMemsetAsync(d_cnt, 0, bytes, m->stream));
  if (m->nnz > 0) {
    constexpr int T = 256, U = 4;
    int64_t blocks = ((m->nnz >> 2) + static_cast<int64_t>(T) * U - 1) / (static_cast<int64_t>(T) * U);
    const int64_t cap = static_cast<int64_t>(m->sm_count) * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    rowvar_stream_kernel<T, U><<<static_cast<unsigned>(blocks), T, 0, m->stream>>>(m->d_i, m->d_x, m->nnz, d_mean, d_S, d_cnt);
    count_launch();
    SB_CUDA(cudaGetLastError());
  }
  return SB200_OK;
}

int launch_row_counts(cudaStream_t st, const int32_t* d_ptr, int64_t n, double* d_cnt) {
  if (n <= 0) return SB200_OK;
  row_counts_kernel<<<elementwise_blocks(n), 256, 0, st>>>(d_ptr, n, d_cnt);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return SB200_OK;
}

}  // namespace

int launch_fill_nan(cudaStream_t s, double* d, int64_t n) {
  if (n <= 0) return SB200_OK;
  fill_nan_kernel<<<elementwise_blocks(n), 256, 0, s>>>(d, n);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return SB200_OK;
}

int launch_col_vars(sb200_matrix* m, double* d_out) {
  if (m->ncol == 0) return SB200_OK;
  if (m->nrow < 2) return launch_fill_nan(m->stream, d_out, m->ncol);
  const double n = static_cast<double>(m->nrow);
  double* d_mean = nullptr;
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&d_mean), sizeof(double) * static_cast<size_t>(m->ncol), m->stream));
  int rc = launch_sweep(m, SWEEP_COLSUM, nullptr, n, d_mean);  // pass 1: colMeans
  if (rc == SB200_OK) rc = launch_col_var_sweep(m, d_mean, n, d_out);
  pool_free(d_mean, m->stream);
  return rc;
}

int launch_row_vars(sb200_matrix* m, double* d_out) {
  if (m->nrow == 0) return SB200_OK;
  if (m->ncol < 2) return launch_fill_nan(m->stream, d_out, m->nrow);
  const double n = static_cast<double>(m->ncol);
  const size_t bytes = sizeof(double) * static_cast<size_t>(m->nrow);
  double *d_mean = nullptr, *d_cnt = nullptr;
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&d_mean), bytes, m->stream));
  int rc = pool_alloc(reinterpret_cast<void**>(&d_cnt), bytes, m->stream);
  // pass 1: rowMeans (it counts toward the row-ordered copy, and may build it, like one rowMeans call)
  if (rc == SB200_OK) rc = launch_sweep(m, SWEEP_ROWSUM, nullptr, n, d_mean);
  if (rc == SB200_OK && m->rows_state == 1 && m->nnz > 0) {
    m->rows->stream = m->stream;
    rc = launch_col_var_sweep(m->rows, d_mean, n, d_out);  // the counts are the copy's column lengths
  } else if (rc == SB200_OK) {
    const int32_t* d_rowptr = nullptr;
    rc = row_var_csc(m, d_mean, d_out, d_cnt, &d_rowptr);
    if (rc == SB200_OK) {
      var_finish_kernel<<<elementwise_blocks(m->nrow), 256, 0, m->stream>>>(d_out, d_mean, d_rowptr, d_cnt, m->nrow, n);
      count_launch();
      const cudaError_t e = cudaGetLastError();
      if (e != cudaSuccess) rc = cuda_fail(e, "var_finish_kernel", __FILE__, __LINE__);
    }
  }
  pool_free(d_mean, m->stream);
  pool_free(d_cnt, m->stream);
  return rc;
}

int launch_row_var_sums(sb200_matrix* m, const double* d_mean, double* d_S, double* d_cnt) {
  if (m->nrow == 0) return SB200_OK;
  if (m->rows_state == 1 && m->nnz > 0) {
    m->rows->stream = m->stream;
    SB_TRY(launch_col_var_sweep(m->rows, d_mean, 0.0, d_S));
    return launch_row_counts(m->stream, m->rows->d_p, m->nrow, d_cnt);
  }
  const int32_t* d_rowptr = nullptr;
  SB_TRY(row_var_csc(m, d_mean, d_S, d_cnt, &d_rowptr));
  if (d_rowptr) return launch_row_counts(m->stream, d_rowptr, m->nrow, d_cnt);
  return SB200_OK;
}

}  // namespace sb200
