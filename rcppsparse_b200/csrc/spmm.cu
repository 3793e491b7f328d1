// Sparse x dense-block products on B200: Y = A B and Y = A^T B for k right-hand sides in one sweep.
//
// What a user otherwise writes as k calls of spmv / spmv_t (NMF, randomized range finders, block Lanczos, subspace
// iteration): each of those streams the whole matrix again.  Here the matrix is streamed once per 32 right-hand
// sides, and the k values a stored entry needs are contiguous.
//
// Layout.  B and Y are column-major at the boundary (R's NumericMatrix).  The kernels read B and write Y ROW-major,
// so the k values of one row sit next to each other: a stored entry (row r, value a) then costs one gather of
// k*8 contiguous bytes of B instead of k gathers of 8 bytes.  spmm_transpose_kernel converts between the two layouts
// (32x32 tiles through shared memory); the conversion is part of every call.
//
// Work decomposition.  The merge-path tiles of the gather plan (d_plan_g, GATHER_TILE items per tile, sweep.cu): a
// tile holds up to GATHER_TILE entries and column ends, whatever the column-length distribution.  A group of W lanes
// owns one tile; lane jl of the group owns right-hand-side column j = slab*W + jl.  W is the slab width, a template
// argument: 2, 4, 8, 16 for k <= W (32/W tiles per warp, so small k leaves no lane idle), 32 above that, where the
// group walks the tile once per slab of 32 columns (the tile's i and x come back from L2 for the later slabs: 12 B
// against the 256 B gather per entry).
//
//   A^T B (spmm_gather_kernel): per lane one FP64 accumulator for the column in progress, fed in entry order.  A
//     column that ends inside the tile is stored straight from the registers: no cross-lane reduction.  The column
//     left open at the tile's end leaves a k-wide carry in scratch; spmm_fold_kernel adds the carries of a column in
//     tile order, then the share of the tile in which it ends.  No atomics: bit-stable run to run.
//   A B on the CSC arrays (spmm_scatter_kernel): the same walk; lane jl holds B[c, j] of the column in progress and
//     sends red.global.add.f64 to the contiguous slots Y[r, j0 .. j0+W) of a zeroed row-major result.
//   A B on the row-ordered copy (a resident mirror's transposed copy, capi.cu): the gather kernel on the copy,
//     A B = (A^T)^T B, so gather-only and deterministic there too.
//
// Sizes are 64-bit inside the kernels: nrow * k may pass 2^31.
//
// launch_spmm_rm stops before the final transpose and leaves Y row-major: the sharded A B (sharded.cu) sums the
// blocks' row-major partials across devices and turns the sum column-major in the same pass.
#include <cuda_runtime.h>
#include <limits.h>
#include <stdint.h>

#include "common.cuh"
#include "ptx.cuh"

namespace sb200 {

constexpr int SPMM_THREADS = 256;
constexpr int SPMM_UNROLL = 4;  // entries whose loads are in flight together per lane

struct SpmmParams {
  const int32_t* i;
  const int32_t* p;
  const double* x;
  const int32_t* plan;  // gather plan: plan[t] = column ends before item t * GATHER_TILE
  int64_t n_tiles;
  int64_t ncol;
  int64_t nnz;
  int64_t k;
  const double* b;     // row-major operand: b[r * k + j]
  double* y;           // row-major result:  y[c * k + j]
  double* carry;       // gather only: [n_tiles * k], the open column's share of each tile
  int32_t* carry_col;  // gather only: [n_tiles], that column, -1 when the tile leaves none
};

struct TileSpan {
  int64_t c0, c1;  // columns c0 .. c1-1 end inside the tile; column c1 is open at its end
  int64_t k0, k1;  // entries [k0, k1)
};

__device__ __forceinline__ TileSpan tile_span(const SpmmParams& prm, int64_t t) {
  TileSpan s;
  s.c0 = __ldg(prm.plan + t);
  s.c1 = __ldg(prm.plan + t + 1);
  const int64_t total = prm.ncol + prm.nnz;
  const int64_t d0 = t * GATHER_TILE;
  int64_t d1 = d0 + GATHER_TILE;
  if (d1 > total) d1 = total;
  s.k0 = d0 - s.c0;
  s.k1 = d1 - s.c1;
  return s;
}

template <int W>
__global__ void __launch_bounds__(SPMM_THREADS) spmm_gather_kernel(const SpmmParams prm) {
  constexpr int GROUPS = 32 / W;  // tiles a warp walks side by side
  constexpr int U = SPMM_UNROLL;
  const int lane = threadIdx.x & 31;
  const int jl = lane % W;
  const int64_t n_groups = static_cast<int64_t>(gridDim.x) * (SPMM_THREADS / 32) * GROUPS;
  const int64_t first = (static_cast<int64_t>(blockIdx.x) * (SPMM_THREADS / 32) + (threadIdx.x >> 5)) * GROUPS + lane / W;
  const int64_t K = prm.k;
  const int64_t n_slabs = (K + W - 1) / W;
  for (int64_t t = first; t < prm.n_tiles; t += n_groups) {
    const TileSpan s = tile_span(prm, t);
    const bool open = s.c1 < prm.ncol && s.k1 > __ldg(prm.p + s.c1);
    if (jl == 0) prm.carry_col[t] = open ? static_cast<int32_t>(s.c1) : -1;
    for (int64_t slab = 0; slab < n_slabs; ++slab) {
      const int64_t j = slab * W + jl;
      const bool on = j < K;  // lanes past the last column load nothing and store nothing
      const double* __restrict__ bj = prm.b + j;
      double* __restrict__ yj = prm.y + j;
      int64_t c = s.c0;
      int64_t e = (c < prm.ncol) ? __ldg(prm.p + c + 1) : LLONG_MAX;  // end of column c
      double acc = 0.0;
      for (int64_t kb = s.k0; kb < s.k1; kb += U) {
        int32_t r[U];
        double a[U], g[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const bool in = kb + u < s.k1;
          r[u] = in ? __ldg(prm.i + kb + u) : 0;
          a[u] = in ? __ldg(prm.x + kb + u) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) g[u] = (on && kb + u < s.k1) ? __ldg(bj + static_cast<int64_t>(r[u]) * K) : 0.0;
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int64_t kk = kb + u;
          if (kk < s.k1) {
            while (kk >= e) {  // column c ended before entry kk (empty columns in between store 0)
              if (on) yj[c * K] = acc;
              acc = 0.0;
              ++c;
              e = __ldg(prm.p + c + 1);  // c <= column of entry kk < ncol
            }
            acc = __fma_rn(a[u], g[u], acc);
          }
        }
      }
      for (; c < s.c1; ++c) {  // columns ending after the tile's last entry
        if (on) yj[c * K] = acc;
        acc = 0.0;
      }
      if (open && on) prm.carry[t * K + j] = acc;
    }
  }
}

// One warp per tile that starts a run of carries into the same column: carries in tile order, then the share the
// column's last tile stored.  Lanes stride over the k right-hand sides.
__global__ void __launch_bounds__(SPMM_THREADS) spmm_fold_kernel(const double* __restrict__ carry,
                                                                 const int32_t* __restrict__ carry_col, int64_t n_tiles,
                                                                 int64_t K, double* __restrict__ y) {
  const int lane = threadIdx.x & 31;
  const int64_t n_warps = static_cast<int64_t>(gridDim.x) * (SPMM_THREADS / 32);
  for (int64_t t = static_cast<int64_t>(blockIdx.x) * (SPMM_THREADS / 32) + (threadIdx.x >> 5); t < n_tiles; t += n_warps) {
    const int32_t c = carry_col[t];
    if (c < 0 || (t > 0 && carry_col[t - 1] == c)) continue;
    int64_t h_end = t + 1;
    while (h_end < n_tiles && carry_col[h_end] == c) ++h_end;
    for (int64_t j = lane; j < K; j += 32) {
      double tot = 0.0;
      for (int64_t h = t; h < h_end; ++h) tot = __dadd_rn(tot, carry[h * K + j]);
      y[c * K + j] = __dadd_rn(tot, y[c * K + j]);
    }
  }
}

template <int W>
__global__ void __launch_bounds__(SPMM_THREADS) spmm_scatter_kernel(const SpmmParams prm) {
  constexpr int GROUPS = 32 / W;
  constexpr int U = SPMM_UNROLL;
  const int lane = threadIdx.x & 31;
  const int jl = lane % W;
  const int64_t n_groups = static_cast<int64_t>(gridDim.x) * (SPMM_THREADS / 32) * GROUPS;
  const int64_t first = (static_cast<int64_t>(blockIdx.x) * (SPMM_THREADS / 32) + (threadIdx.x >> 5)) * GROUPS + lane / W;
  const int64_t K = prm.k;
  const int64_t n_slabs = (K + W - 1) / W;
  for (int64_t t = first; t < prm.n_tiles; t += n_groups) {
    const TileSpan s = tile_span(prm, t);
    if (s.k1 <= s.k0) continue;  // only column ends: nothing to scatter
    for (int64_t slab = 0; slab < n_slabs; ++slab) {
      const int64_t j = slab * W + jl;
      const bool on = j < K;
      double* __restrict__ yj = prm.y + j;
      int64_t c = s.c0;
      int64_t e = __ldg(prm.p + c + 1);  // the tile has an entry, so c0 < ncol
      double vc = on ? __ldg(prm.b + c * K + j) : 0.0;  // B[c, j] of the column in progress
      for (int64_t kb = s.k0; kb < s.k1; kb += U) {
        int32_t r[U];
        double a[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const bool in = kb + u < s.k1;
          r[u] = in ? __ldg(prm.i + kb + u) : 0;
          a[u] = in ? __ldg(prm.x + kb + u) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int64_t kk = kb + u;
          if (kk < s.k1) {
            if (kk >= e) {  // column c ended before entry kk: skip to the column of kk
              do {
                ++c;
                e = __ldg(prm.p + c + 1);
              } while (kk >= e);
              vc = on ? __ldg(prm.b + c * K + j) : 0.0;
            }
            if (on) ptx::red_add_f64(yj + static_cast<int64_t>(r[u]) * K, __dmul_rn(a[u], vc));
          }
        }
      }
    }
  }
}

// dst (C x R, row-major) = transpose of src (R x C, row-major); a column-major R x C matrix is a row-major C x R one.
__global__ void __launch_bounds__(256) spmm_transpose_kernel(const double* __restrict__ src, int64_t R, int64_t C,
                                                             double* __restrict__ dst) {
  __shared__ double tile[32][33];
  const int tx = threadIdx.x, ty = threadIdx.y;  // 32 x 8
  const int64_t tr = (R + 31) / 32, tc = (C + 31) / 32;
  for (int64_t blk = blockIdx.x; blk < tr * tc; blk += gridDim.x) {
    const int64_t r0 = (blk / tc) * 32, c0 = (blk % tc) * 32;
    for (int q = ty; q < 32; q += 8) {
      const int64_t r = r0 + q, c = c0 + tx;
      if (r < R && c < C) tile[q][tx] = src[r * C + c];
    }
    __syncthreads();
    for (int q = ty; q < 32; q += 8) {
      const int64_t c = c0 + q, r = r0 + tx;
      if (r < R && c < C) dst[c * R + r] = tile[tx][q];
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static int launch_transpose(cudaStream_t st, const double* src, int64_t R, int64_t C, double* dst) {
  const int64_t tiles = ((R + 31) / 32) * ((C + 31) / 32);
  int64_t grid = tiles < 148 * 16 ? tiles : 148 * 16;
  if (grid < 1) return SB200_OK;
  spmm_transpose_kernel<<<static_cast<unsigned>(grid), dim3(32, 8), 0, st>>>(src, R, C, dst);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return SB200_OK;
}

template <typename Kern>
static int launch_tiles(Kern kern, const sb200_matrix* a, const SpmmParams& prm, int w, cudaStream_t st) {
  int per_sm = 0;
  SB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, SPMM_THREADS, 0));
  if (per_sm < 1) per_sm = 1;
  int64_t grid = static_cast<int64_t>(a->sm_count) * per_sm;
  const int64_t groups_per_block = (SPMM_THREADS / 32) * (32 / w);
  const int64_t need = (prm.n_tiles + groups_per_block - 1) / groups_per_block;  // no block without a tile
  if (grid > need) grid = need;
  if (grid < 1) return SB200_OK;
  kern<<<static_cast<unsigned>(grid), SPMM_THREADS, 0, st>>>(prm);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return SB200_OK;
}

static int slab_width(int64_t k) { return k <= 2 ? 2 : k <= 4 ? 4 : k <= 8 ? 8 : k <= 16 ? 16 : 32; }

template <template <int> class Sel>
static int launch_by_width(const sb200_matrix* a, const SpmmParams& prm, cudaStream_t st) {
  switch (slab_width(prm.k)) {
    case 2: return launch_tiles(Sel<2>::kern(), a, prm, 2, st);
    case 4: return launch_tiles(Sel<4>::kern(), a, prm, 4, st);
    case 8: return launch_tiles(Sel<8>::kern(), a, prm, 8, st);
    case 16: return launch_tiles(Sel<16>::kern(), a, prm, 16, st);
    default: return launch_tiles(Sel<32>::kern(), a, prm, 32, st);
  }
}
template <int W>
struct GatherSel {
  static auto kern() { return spmm_gather_kernel<W>; }
};
template <int W>
struct ScatterSel {
  static auto kern() { return spmm_scatter_kernel<W>; }
};

static SpmmParams params_of(const sb200_matrix* a, const double* b_rm, int64_t k, double* y_rm) {
  SpmmParams prm;
  prm.i = a->d_i;
  prm.p = a->d_p;
  prm.x = a->d_x;
  prm.plan = a->d_plan_g;
  prm.n_tiles = a->n_tiles_g;
  prm.ncol = a->ncol;
  prm.nnz = a->nnz;
  prm.k = k;
  prm.b = b_rm;
  prm.y = y_rm;
  prm.carry = nullptr;
  prm.carry_col = nullptr;
  return prm;
}

// y_rm[a->ncol x k] = a^T b_rm[a->nrow x k], deterministic; scratch for the carries from the pool
static int gather_rm(const sb200_matrix* a, const double* b_rm, int64_t k, double* y_rm, cudaStream_t st) {
  SpmmParams prm = params_of(a, b_rm, k, y_rm);
  if (prm.n_tiles == 0) return SB200_OK;
  const size_t carry_bytes = sizeof(double) * static_cast<size_t>(prm.n_tiles) * static_cast<size_t>(k);
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&prm.carry), carry_bytes, st));
  int rc = pool_alloc(reinterpret_cast<void**>(&prm.carry_col), sizeof(int32_t) * static_cast<size_t>(prm.n_tiles), st);
  if (rc == SB200_OK) rc = launch_by_width<GatherSel>(a, prm, st);
  if (rc == SB200_OK) {
    int64_t grid = (prm.n_tiles + SPMM_THREADS / 32 - 1) / (SPMM_THREADS / 32);
    if (grid > 148 * 16) grid = 148 * 16;
    spmm_fold_kernel<<<static_cast<unsigned>(grid), SPMM_THREADS, 0, st>>>(prm.carry, prm.carry_col, prm.n_tiles, k, y_rm);
    count_launch();
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) rc = cuda_fail(e, "spmm_fold_kernel", __FILE__, __LINE__);
  }
  pool_free(prm.carry, st);
  pool_free(prm.carry_col, st);
  return rc;
}

static bool bytes_of(int64_t rows, int64_t k, size_t* out) {
  if (rows > 0 && k > static_cast<int64_t>(SIZE_MAX / 16) / rows) return false;
  *out = sizeof(double) * static_cast<size_t>(rows) * static_cast<size_t>(k);
  return true;
}

// d_Yrm (y_rows x k, ROW-major) = A d_B or A^T d_B (d_B column-major): everything launch_spmm does before its final
// transpose.  The sharded A B (sharded.cu) sums these row-major partials across devices and transposes while it sums.
int launch_spmm_rm(sb200_matrix* m, bool transposed, const double* d_B, int64_t k, double* d_Yrm) {
  const int64_t b_rows = transposed ? m->nrow : m->ncol;
  const int64_t y_rows = transposed ? m->ncol : m->nrow;
  if (k == 0 || y_rows == 0) return SB200_OK;
  if (k == 1) return launch_sweep(m, transposed ? SWEEP_SPMV_T : SWEEP_SPMV, d_B, 0.0, d_Yrm);  // n x 1: both layouts
  cudaStream_t st = m->stream;
  size_t b_bytes = 0, y_bytes = 0;
  if (!bytes_of(b_rows, k, &b_bytes) || !bytes_of(y_rows, k, &y_bytes))
    return fail(SB200_E_NOMEM, "spmm: the dense operand or result does not fit in device memory");
  if (m->nnz == 0 || b_rows == 0) {  // no stored entry: the zero matrix, as k calls of spmv give
    SB_CUDA(cudaMemsetAsync(d_Yrm, 0, y_bytes, st));
    return SB200_OK;
  }
  // A B on a resident mirror: same ski-rental rule as A v (launch_sweep) — a k-wide call counts once
  if (!transposed && m->rows_state == 0 && m->owns_arrays) {
    const int after = row_companion_after();
    if (after > 0 && ++m->row_sum_calls > after) build_row_companion(m);
  }
  const bool on_rows = !transposed && m->rows_state == 1;
  if (on_rows) m->rows->stream = st;
  double* b_rm = nullptr;
  int rc = pool_alloc(reinterpret_cast<void**>(&b_rm), b_bytes, st);
  if (rc == SB200_OK) rc = launch_transpose(st, d_B, k, b_rows, b_rm);  // column-major b_rows x k -> row-major
  if (rc == SB200_OK) {
    if (transposed)
      rc = gather_rm(m, b_rm, k, d_Yrm, st);
    else if (on_rows)
      rc = gather_rm(m->rows, b_rm, k, d_Yrm, st);  // A B = (A^T)^T B on the row-ordered copy
    else {
      const cudaError_t e = cudaMemsetAsync(d_Yrm, 0, y_bytes, st);
      rc = e == cudaSuccess ? launch_by_width<ScatterSel>(m, params_of(m, b_rm, k, d_Yrm), st)
                            : cuda_fail(e, "cudaMemsetAsync", __FILE__, __LINE__);
    }
  }
  pool_free(b_rm, st);
  if (rc == SB200_E_NOMEM) cudaGetLastError();  // a refused allocation leaves the stream usable
  return rc;
}

int launch_spmm(sb200_matrix* m, bool transposed, const double* d_B, int64_t k, double* d_Y) {
  const int64_t b_rows = transposed ? m->nrow : m->ncol;
  const int64_t y_rows = transposed ? m->ncol : m->nrow;
  // k <= 1 or no stored entry: the row-major result is the column-major one (n x 1, or all zeros)
  if (k <= 1 || y_rows == 0 || m->nnz == 0 || b_rows == 0) return launch_spmm_rm(m, transposed, d_B, k, d_Y);
  cudaStream_t st = m->stream;
  size_t y_bytes = 0;
  if (!bytes_of(y_rows, k, &y_bytes)) return fail(SB200_E_NOMEM, "spmm: the dense operand or result does not fit in device memory");
  double* y_rm = nullptr;
  int rc = pool_alloc(reinterpret_cast<void**>(&y_rm), y_bytes, st);
  if (rc == SB200_OK) rc = launch_spmm_rm(m, transposed, d_B, k, y_rm);
  if (rc == SB200_OK) rc = launch_transpose(st, y_rm, y_rows, k, d_Y);  // row-major y_rows x k -> column-major
  pool_free(y_rm, st);
  if (rc == SB200_E_NOMEM) cudaGetLastError();  // a refused allocation leaves the stream usable
  return rc;
}

}  // namespace sb200
