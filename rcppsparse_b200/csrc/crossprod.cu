// crossprod(): dense A^T A (reference inst/include/RcppSparse.h:158-194; SURVEY.md 8f N2).
//
// The reference merges the sorted row lists of every PAIR of columns — n(n+1)/2 two-pointer merges, OpenMP over
// the first column.  On the device the sum is turned inside out: A^T A = sum over rows r of (row r)^T (row r),
// and the row-ordered copy of the mirror (capi.cu, build_row_companion) has every row as a contiguous list of
// (column id ascending, value).  A warp takes a row, stages it in shared memory, and for every pair a <= b of its
// entries fires one FP64 reduction at L2 into res(c_a, c_b) — sum_r k_r^2 / 2 reductions in all, nothing per
// column pair.  Only the upper triangle is accumulated; a tiled mirror pass then copies it below the diagonal,
// so the result is exactly symmetric like the reference's (which assigns res(col2, col1) = res(col1, col2)).
// The order of the additions inside one entry is not the reference's ascending-row order: results agree within
// the 1e-12 * sum|terms| bar, not bitwise.  The sharded form (crossprod_slab_kernel below) keeps that order instead.
#include <algorithm>

#include "common.cuh"
#include "ptx.cuh"

namespace sb200 {
namespace {

constexpr int CP_THREADS = 256;
constexpr int CP_WARPS = CP_THREADS / 32;
constexpr int CP_CAP = 480;  // entries of a row staged per warp (45 KB per CTA); longer rows are walked in pieces

__global__ void __launch_bounds__(CP_THREADS) crossprod_rows_kernel(const int32_t* __restrict__ pt, const int32_t* __restrict__ ct,
                                                                     const double* __restrict__ xt, int32_t nrow, int64_t n,
                                                                     double* __restrict__ res) {
  __shared__ int32_t s_c[CP_WARPS][CP_CAP];
  __shared__ double s_x[CP_WARPS][CP_CAP];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t warps_total = static_cast<int64_t>(gridDim.x) * CP_WARPS;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * CP_WARPS + warp; r < nrow; r += warps_total) {
    const int32_t k0 = __ldg(pt + r), k1 = __ldg(pt + r + 1);
    // pieces of the row: (piece A, piece B >= A); inside a diagonal piece only pairs a <= b
    for (int32_t a0 = k0; a0 < k1; a0 += CP_CAP) {
      const int32_t an = min(CP_CAP, k1 - a0);
      __syncwarp();
      for (int32_t t = lane; t < an; t += 32) {
        s_c[warp][t] = __ldg(ct + a0 + t);
        s_x[warp][t] = __ldg(xt + a0 + t);
      }
      __syncwarp();
      // diagonal piece
      for (int32_t a = 0; a < an; ++a) {
        const int64_t ca = s_c[warp][a];
        const double xa = s_x[warp][a];
        for (int32_t b = a + lane; b < an; b += 32)
          ptx::red_add_f64(res + ca + static_cast<int64_t>(s_c[warp][b]) * n, __dmul_rn(xa, s_x[warp][b]));
      }
      // pieces to the right (rows longer than CP_CAP entries): b from global memory
      for (int32_t b = a0 + an + lane; b < k1; b += 32) {
        const int64_t cb = __ldg(ct + b);
        const double xb = __ldg(xt + b);
        for (int32_t a = 0; a < an; ++a) ptx::red_add_f64(res + s_c[warp][a] + cb * n, __dmul_rn(s_x[warp][a], xb));
      }
    }
  }
}

// res(j, i) = res(i, j) for i < j, 32 x 32 tiles through shared memory (both sides coalesced)
__global__ void __launch_bounds__(256) mirror_upper_kernel(double* __restrict__ res, int64_t n) {
  __shared__ double tile[32][33];
  const int64_t bi = blockIdx.x, bj = blockIdx.y;
  if (bi > bj) return;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int c = ty; c < 32; c += 8) {
    const int64_t row = bi * 32 + tx, col = bj * 32 + c;
    tile[c][tx] = (row < n && col < n) ? res[row + col * n] : 0.0;  // element (row, col) of the upper part
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int64_t row = bi * 32 + r, col = bj * 32 + tx;  // write (col, row) = below the diagonal when row < col
    if (row < n && col < n && row < col) res[col + row * n] = tile[tx][r];
  }
}

// ---- the ordered column sweep of the sharded crossprod (sharded.cu, sb200_sharded_crossprod) ------------------------
// slab(a, b) = sum over the rows r of column b, in ascending r, of x_ra * x_rb, from +0.0 with __dmul_rn / __dadd_rn:
// the reference's order of additions (RcppSparse.h:178-188), so res(a, b) and res(b, a) come out bitwise equal.
// A warp owns (local column b, output rows [a0, a0 + SLAB_SPAN)) with that span's accumulators in shared memory.  It
// takes column b's entries 32 rows at a time: every lane binary-searches its row of the whole-matrix row-ordered copy
// for the piece inside the span and prefetches up to SLAB_PREFETCH of its entries; then the rows are applied one after
// another, lanes on distinct slots, a __syncwarp between rows.  The span is stored once, coalesced: no memset.
constexpr int SLAB_THREADS = 256;
constexpr int SLAB_WARPS = SLAB_THREADS / 32;
constexpr int SLAB_SPAN = 512;      // accumulators per warp (32 KB per CTA)
constexpr int SLAB_PREFETCH = 2;    // entries of a row's piece that travel in registers; longer pieces are read in the apply

__device__ __forceinline__ int32_t lower_bound_i32(const int32_t* __restrict__ a, int32_t lo, int32_t hi, int32_t key) {
  while (lo < hi) {
    const int32_t mid = lo + ((hi - lo) >> 1);
    if (__ldg(a + mid) < key)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(SLAB_THREADS) crossprod_slab_kernel(const int32_t* __restrict__ bp, const int32_t* __restrict__ bi,
                                                                     const double* __restrict__ bx, int64_t ncol_w,
                                                                     const int32_t* __restrict__ rp, const int32_t* __restrict__ rc,
                                                                     const double* __restrict__ rv, int64_t ncol,
                                                                     double* __restrict__ slab) {
  __shared__ double s_acc[SLAB_WARPS][SLAB_SPAN];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* acc = s_acc[warp];
  const int64_t spans = (ncol + SLAB_SPAN - 1) / SLAB_SPAN;
  const int64_t warps_total = static_cast<int64_t>(gridDim.x) * SLAB_WARPS;
  for (int64_t task = static_cast<int64_t>(blockIdx.x) * SLAB_WARPS + warp; task < ncol_w * spans; task += warps_total) {
    const int64_t b = task / spans;
    const int64_t a0 = (task % spans) * SLAB_SPAN;
    const int32_t lo_key = static_cast<int32_t>(a0);
    const int32_t width = static_cast<int32_t>(ncol - a0 < SLAB_SPAN ? ncol - a0 : SLAB_SPAN);
    const int32_t hi_key = lo_key + width;
    for (int t = lane; t < SLAB_SPAN; t += 32) acc[t] = 0.0;
    __syncwarp();
    const int32_t e0 = __ldg(bp + b), e1 = __ldg(bp + b + 1);
    for (int32_t base = e0; base < e1; base += 32) {
      int32_t lo = 0, hi = 0;
      double xb = 0.0;
      int32_t pc[SLAB_PREFETCH];
      double pv[SLAB_PREFETCH];
#pragma unroll
      for (int u = 0; u < SLAB_PREFETCH; ++u) {
        pc[u] = 0;
        pv[u] = 0.0;
      }
      if (base + lane < e1) {
        const int32_t r = __ldg(bi + base + lane);
        xb = __ldg(bx + base + lane);
        const int32_t s0 = __ldg(rp + r), s1 = __ldg(rp + r + 1);
        lo = lower_bound_i32(rc, s0, s1, lo_key);
        hi = lower_bound_i32(rc, lo, lo + min(s1 - lo, width), hi_key);  // at most `width` distinct columns fall inside
#pragma unroll
        for (int u = 0; u < SLAB_PREFETCH; ++u)
          if (lo + u < hi) {
            pc[u] = __ldg(rc + lo + u) - lo_key;
            pv[u] = __ldg(rv + lo + u);
          }
      }
      const int rows = min(32, e1 - base);
      for (int j = 0; j < rows; ++j) {  // ascending r: the rows of a column are sorted
        const int32_t lj = __shfl_sync(0xffffffffu, lo, j);
        const int32_t n = __shfl_sync(0xffffffffu, hi, j) - lj;
        const double xj = __shfl_sync(0xffffffffu, xb, j);
        if (n == 0) continue;  // uniform: the piece of row j misses the span
        if (n <= SLAB_PREFETCH) {
#pragma unroll
          for (int u = 0; u < SLAB_PREFETCH; ++u) {
            const int32_t c = __shfl_sync(0xffffffffu, pc[u], j);
            const double v = __shfl_sync(0xffffffffu, pv[u], j);
            if (lane == u && u < n) acc[c] = __dadd_rn(acc[c], __dmul_rn(v, xj));
          }
        } else {
          for (int32_t t = lj + lane; t < lj + n; t += 32) {
            const int32_t c = __ldg(rc + t) - lo_key;
            acc[c] = __dadd_rn(acc[c], __dmul_rn(__ldg(rv + t), xj));
          }
        }
        __syncwarp();  // the next row may add to the same slots
      }
    }
    double* out = slab + b * ncol + a0;
    for (int t = lane; t < width; t += 32) out[t] = acc[t];
    __syncwarp();
  }
}

}  // namespace

int launch_crossprod_slab(const sb200_matrix* blk, const int32_t* rp, const int32_t* rc, const double* rv, int64_t ncol, double* slab) {
  if (blk->ncol == 0 || ncol == 0) return SB200_OK;
  const int64_t tasks = static_cast<int64_t>(blk->ncol) * ((ncol + SLAB_SPAN - 1) / SLAB_SPAN);
  const int64_t blocks = std::min<int64_t>((tasks + SLAB_WARPS - 1) / SLAB_WARPS, static_cast<int64_t>(blk->sm_count) * 8);
  crossprod_slab_kernel<<<static_cast<unsigned>(blocks), SLAB_THREADS, 0, blk->stream>>>(blk->d_p, blk->d_i, blk->d_x, blk->ncol, rp, rc,
                                                                                          rv, ncol, slab);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return SB200_OK;
}

// T = the row-ordered copy of the mirror (its "columns" are the rows of A, its i the column ids of A)
int launch_crossprod(const sb200_matrix* T, int32_t ncol_a, double* d_res, cudaStream_t st) {
  const int64_t n = ncol_a;
  if (n == 0) return SB200_OK;
  SB_CUDA(cudaMemsetAsync(d_res, 0, sizeof(double) * static_cast<size_t>(n) * static_cast<size_t>(n), st));
  if (T->nnz > 0 && T->ncol > 0) {
    int64_t blocks = (static_cast<int64_t>(T->ncol) + CP_WARPS - 1) / CP_WARPS;
    const int64_t cap = static_cast<int64_t>(T->sm_count) * 8;
    if (blocks > cap) blocks = cap;
    crossprod_rows_kernel<<<static_cast<unsigned>(blocks), CP_THREADS, 0, st>>>(T->d_p, T->d_i, T->d_x, T->ncol, n, d_res);
    count_launch();
    SB_CUDA(cudaGetLastError());
  }
  const unsigned tiles = static_cast<unsigned>((n + 31) / 32);
  if (tiles > 65535) return fail(SB200_E_UNSUPPORTED, "crossprod: more than 2M columns");
  mirror_upper_kernel<<<dim3(tiles, tiles), 256, 0, st>>>(d_res, n);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return SB200_OK;
}

}  // namespace sb200
