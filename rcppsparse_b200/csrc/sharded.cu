// One process, several GPUs: the column-sharding layer behind the C ABI (SURVEY.md 8e, 8b).
//
// The reference is one R process (zdebruine/RcppSparse; every method of RcppSparse::Matrix, RcppSparse.h:131-156,
// runs on the calling thread), so a drop-in that wants more than one GPU cannot ask for one process per device.
// sb200_sharded_create cuts the dgCMatrix into nnz-balanced contiguous column blocks (binary search in p; a block
// is itself a dgCMatrix with the full row count and p rebased to 0), uploads block k to devices[k] as an ordinary
// mirror (worker thread per device: each device has its own PCIe link), and gives every device a window of
// peer-mapped memory.  The ops then run as the same kernels as on one GPU:
//   column-indexed results (colSums, colMeans, A^T v)  disjoint slices: every device sweeps its block and its slice
//                                                      goes straight to its place in the caller's host vector;
//   row-indexed results (rowSums, rowMeans, A v)       full-length partials in the windows, summed in rank order by
//                                                      the library's own P2P reduction kernel (exchange.cu) running
//                                                      on every device at once; the mean's division by the GLOBAL
//                                                      ncol rides in that kernel (RcppSparse.h:154).
// All launches come from the calling thread, device after device, nothing blocks until the final synchronisation.
//
// The k-wide products (sb200_sharded_spmm / _t) follow the same split:
//   A^T B   every device gets the whole B, runs the one-GPU block product on its block, and its rows of Y (a strided
//           piece of the caller's column-major Y) go straight home;
//   A B     device w gets its rows of B (a strided slice), leaves its full-height partial A_w B_w ROW-major in a buffer
//           of plain cudaMalloc memory (pool memory is not peer-readable), and device q sums rows
//           [q nrow / W, (q+1) nrow / W) of all partials over peer memory, in rank order, turning the sum column-major
//           in the same pass (sharded_sum_transpose_kernel); then every device copies its rows home.
//           Ordering across devices is CUDA events only (no in-kernel barrier), so blocks that share a device are fine.
// Host copies run from one thread per device (a copy from pageable memory blocks the thread that issues it).
// The variances (sb200_sharded_col_vars / _row_vars): colVars is column-indexed like colMeans; rowVars takes the global row
// means as rowMeans does, then reduces every block's sums of squared deviations and entry counts in rank order over peer
// memory (sharded_row_var_kernel, ordered by events like the A B reduce) and applies the formula on every device.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <limits>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"
#include "pushrows.cuh"

struct sb200_sharded {
  uint32_t magic;
  int world;
  int32_t nrow, ncol;
  int64_t nnz;
  std::vector<int> devices;
  std::vector<int64_t> bounds;  // [world + 1] first column of every block
  std::vector<sb200_matrix*> blocks;
  std::vector<sb200_exchange*> windows;
  int64_t partial_off, result_off;  // byte offsets of the row partial / the row result inside every window
  // per block a partial its peers read (cudaMalloc: pool memory is not peer-readable), grown on demand, kept between
  // calls: A B's row-major nrow x k partial, rowVars' sums and counts
  std::vector<double*> peer_partial;
  std::vector<size_t> peer_partial_bytes;
  std::vector<cudaEvent_t> ev_partial;  // per block: its partial is complete
  std::vector<cudaEvent_t> ev_reduced;  // per block: its reduce has read every partial
};

namespace sb200 {
namespace {

constexpr uint32_t SHARDED_MAGIC = 0x5B2005A4u;

int check_sharded(const sb200_sharded* s) {
  if (!s || s->magic != SHARDED_MAGIC) return fail(SB200_E_INVALID, "not a live sb200_sharded handle");
  return SB200_OK;
}

// Waits for every block's stream, whatever happened on another; the first error
cudaError_t sync_blocks(const sb200_sharded* s) {
  cudaError_t first = cudaSuccess;
  for (int w = 0; w < s->world; ++w) {
    DeviceGuard g(s->blocks[w]->device);
    const cudaError_t e = cudaStreamSynchronize(s->blocks[w]->stream);
    if (first == cudaSuccess) first = e;
  }
  return first;
}

// fn(w) on one host thread per block, on the block's device; the first failure, with its message, is returned
template <typename F>
int on_every_block(const sb200_sharded* s, const char* what, F fn) {
  std::vector<int> rcs(s->world, SB200_OK);
  std::vector<std::string> errs(s->world);
  std::vector<std::thread> workers;
  for (int w = 0; w < s->world; ++w)
    workers.emplace_back([&, w] {
      if (cudaSetDevice(s->devices[w]) != cudaSuccess) {
        rcs[w] = SB200_E_CUDA;
        errs[w] = "cudaSetDevice failed";
        return;
      }
      rcs[w] = fn(w);
      if (rcs[w] != SB200_OK) errs[w] = sb200_last_error();
    });
  for (auto& t : workers) t.join();
  for (int w = 0; w < s->world; ++w)
    if (rcs[w] != SB200_OK)
      return fail(rcs[w], std::string(what) + ", column block " + std::to_string(w) + " (device " + std::to_string(s->devices[w]) +
                              "): " + errs[w]);
  return SB200_OK;
}

// Contiguous ranges of [0, len) with about total / n entries each: out[0] = 0, out[n] = len, and out[k] the first index
// whose offset off[index] reaches k * total / n.  off is a prefix array of len + 1 entries (p of a CSC matrix).
template <typename B>
void nnz_balanced_bounds(const int32_t* off, int64_t len, int64_t total, int n, B* out) {
  out[0] = 0;
  for (int k = 1; k < n; ++k) {
    const int64_t target = (total * k) / n;
    int64_t lo = out[k - 1], hi = len;
    while (lo < hi) {
      const int64_t mid = lo + ((hi - lo) >> 1);
      if (off[mid] < target)
        lo = mid + 1;
      else
        hi = mid;
    }
    out[k] = static_cast<B>(lo);
  }
  out[n] = static_cast<B>(len);
}

// SB200_TRACE=1: CUDA-event time of a call's device part on every block's stream, from start() to stop(); report()
// prints its max and per-device times (tools/sharded_*_bench.py read "device part <ms> ms")
struct DevicePartTimer {
  const sb200_sharded* s;
  bool on;
  std::vector<cudaEvent_t> t0, t1;
  DevicePartTimer(const sb200_sharded* sh, bool trace) : s(sh), on(trace), t0(sh->world, nullptr), t1(sh->world, nullptr) {}
  ~DevicePartTimer() {
    for (int w = 0; w < s->world; ++w) {
      DeviceGuard g(s->blocks[w]->device);
      if (t0[w]) cudaEventDestroy(t0[w]);
      if (t1[w]) cudaEventDestroy(t1[w]);
    }
  }
  int record(std::vector<cudaEvent_t>& ev) {
    for (int w = 0; w < s->world && on; ++w) {
      DeviceGuard g(s->blocks[w]->device);
      if (!ev[w]) SB_CUDA(cudaEventCreate(&ev[w]));
      SB_CUDA(cudaEventRecord(ev[w], s->blocks[w]->stream));
    }
    return SB200_OK;
  }
  int start() { return record(t0); }
  int stop() { return record(t1); }
  void report(const char* title) {  // every stream has passed stop()
    if (!on) return;
    std::string per;
    float worst = 0.0f;
    for (int w = 0; w < s->world; ++w) {
      DeviceGuard g(s->blocks[w]->device);
      float ms = 0.0f;
      cudaEventElapsedTime(&ms, t0[w], t1[w]);
      worst = std::max(worst, ms);
      per += (w ? " " : "") + std::to_string(ms);
    }
    fprintf(stderr, "[sb200 trace] %s: device part %.4f ms (max over devices; per device: %s)\n", title, worst, per.c_str());
  }
};

void destroy_sharded(sb200_sharded* s) {
  if (!s) return;
  WallTrace tr("sharded destroy");
  for (cudaEvent_t e : s->ev_reduced)  // no reader still has a partial in flight (every call also ends synchronised)
    if (e) cudaEventSynchronize(e);
  for (size_t k = 0; k < s->peer_partial.size(); ++k) {
    DeviceGuard g(s->devices[k]);
    if (s->peer_partial[k]) cudaFree(s->peer_partial[k]);
  }
  for (size_t k = 0; k < s->ev_partial.size(); ++k) {
    DeviceGuard g(s->devices[k]);
    if (s->ev_partial[k]) cudaEventDestroy(s->ev_partial[k]);
    if (s->ev_reduced[k]) cudaEventDestroy(s->ev_reduced[k]);
  }
  cudaGetLastError();
  for (sb200_matrix* m : s->blocks)
    if (m) sb200_matrix_destroy(m);
  tr.phase("blocks");
  for (sb200_exchange* x : s->windows)
    if (x) sb200_exchange_destroy(x);
  tr.phase("windows");
  s->magic = 0;
  delete s;
}

// column-indexed op: out[bounds[k] .. bounds[k+1]) from device k
int run_columns(sb200_sharded* s, SweepMode mode, const double* v_host, double divisor, double* out) {
  if (s->ncol > 0 && !out) return fail(SB200_E_INVALID, "output buffer is NULL");
  DeviceGuard restore(s->blocks[0]->device);  // the caller's current device is put back on return
  int rc = SB200_OK;
  for (int k = 0; k < s->world && rc == SB200_OK; ++k) {
    sb200_matrix* m = s->blocks[k];
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(SB200_E_CUDA, "cudaSetDevice failed");
    if (mode == SWEEP_SPMV_T && s->nrow > 0)
      SB_CUDA(cudaMemcpyAsync(m->d_stage_in, v_host, sizeof(double) * static_cast<size_t>(s->nrow), cudaMemcpyHostToDevice, m->stream));
    rc = launch_sweep(m, mode, m->d_stage_in, divisor, m->d_stage_out);
    if (rc == SB200_OK && m->ncol > 0)
      SB_CUDA(cudaMemcpyAsync(out + s->bounds[k], m->d_stage_out, sizeof(double) * static_cast<size_t>(m->ncol), cudaMemcpyDeviceToHost,
                              m->stream));
  }
  const cudaError_t e = sync_blocks(s);
  if (e != cudaSuccess && rc == SB200_OK) rc = cuda_fail(e, "sharded column sweep", __FILE__, __LINE__);
  return rc;
}

// row-indexed op up to its result: partials in the windows, rank-ordered P2P reduction on every device.  The result
// (divided by divisor when it is not 0) is at byte offset *off of every window, in each block's stream order.
int rows_into_windows(sb200_sharded* s, SweepMode mode, const double* v_host, double divisor, int64_t* off) {
  *off = s->world > 1 ? s->result_off : s->partial_off;
  int rc = SB200_OK;
  for (int k = 0; k < s->world && rc == SB200_OK; ++k) {
    sb200_matrix* m = s->blocks[k];
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(SB200_E_CUDA, "cudaSetDevice failed");
    double* partial = reinterpret_cast<double*>(exchange_window_base(s->windows[k]) + s->partial_off);
    if (mode == SWEEP_SPMV && m->ncol > 0)
      SB_CUDA(cudaMemcpyAsync(m->d_stage_in, v_host + s->bounds[k], sizeof(double) * static_cast<size_t>(m->ncol), cudaMemcpyHostToDevice,
                              m->stream));
    rc = launch_sweep(m, mode, m->d_stage_in, 0.0, partial);
  }
  if (rc == SB200_OK) {
    if (s->world > 1) {
      for (int k = 0; k < s->world && rc == SB200_OK; ++k)
        rc = sb200_exchange_reduce(s->windows[k], s->blocks[k]->stream, s->partial_off, s->result_off, s->nrow, divisor);
    } else if (divisor != 0.0 && s->nrow > 0) {
      DeviceGuard guard(s->blocks[0]->device);
      rc = launch_vec_div(s->blocks[0]->stream, reinterpret_cast<double*>(exchange_window_base(s->windows[0]) + s->partial_off), s->nrow,
                          divisor);
    }
  }
  return rc;
}

// row-indexed op: rows_into_windows, result read from device 0
int run_rows(sb200_sharded* s, SweepMode mode, const double* v_host, double divisor, double* out) {
  if (s->nrow > 0 && !out) return fail(SB200_E_INVALID, "output buffer is NULL");
  DeviceGuard restore(s->blocks[0]->device);  // the exchange entry points switch devices; put the caller's back on return
  int64_t off = 0;
  int rc = rows_into_windows(s, mode, v_host, divisor, &off);
  if (rc == SB200_OK && s->nrow > 0) {
    DeviceGuard guard(s->blocks[0]->device);
    SB_CUDA(cudaMemcpyAsync(out, exchange_window_base(s->windows[0]) + off, sizeof(double) * static_cast<size_t>(s->nrow),
                            cudaMemcpyDeviceToHost, s->blocks[0]->stream));
  }
  const cudaError_t e = sync_blocks(s);
  if (e != cudaSuccess && rc == SB200_OK) rc = cuda_fail(e, "sharded row sweep", __FILE__, __LINE__);
  return rc;
}


// ---- sharded transpose (SURVEY.md 8e): local transposes, row segments pushed to the devices that own the rows -------
struct TpPtrs {
  const int32_t* p[PUSH_MAX_RANKS];  // row pointers of the devices' local transposes (peer-readable)
};
struct PtrDest {
  int32_t* c[PUSH_MAX_RANKS];
  double* v[PUSH_MAX_RANKS];
  __device__ __forceinline__ int32_t* cols(int q) const { return c[q]; }
  __device__ __forceinline__ double* vals(int q) const { return v[q]; }
};

// cnt[r] = entries of row r over all column blocks
__global__ void shard_row_counts_kernel(const TpPtrs tp, int world, int32_t nrow, uint32_t* __restrict__ cnt) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < nrow; r += stride) {
    uint32_t n = 0;
    for (int k = 0; k < world; ++k) n += static_cast<uint32_t>(tp.p[k][r + 1] - tp.p[k][r]);
    cnt[r] = n;
  }
}

struct RowBounds {
  int32_t rb[PUSH_MAX_RANKS + 1];
};

// dst[k * nrow + r] = where block k's piece of row r starts inside the arrays of the row's owner: the row's place in
// the result (P[r], relative to the owner's first row) plus the pieces of the blocks before k — block order = column order
__global__ void shard_row_dst_kernel(const TpPtrs tp, int world, int32_t nrow, const int32_t* __restrict__ P, const RowBounds b,
                                     int64_t* __restrict__ dst) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < nrow; r += stride) {
    int q = 0;
    while (q + 1 < world && b.rb[q + 1] <= r) ++q;
    int64_t run = static_cast<int64_t>(P[r]) - P[b.rb[q]];
    for (int k = 0; k < world; ++k) {
      dst[static_cast<int64_t>(k) * nrow + r] = run;
      run += tp.p[k][r + 1] - tp.p[k][r];
    }
  }
}

__global__ void __launch_bounds__(256) push_rows_local_kernel(const PushRowsSrc a, int world, const PtrDest d) {
  push_rows_body(a, world, d);
}

// Whole rows from the blocks' row-ordered copies, shared by the sharded transpose (rows dealt to owners) and the sharded
// crossprod (every row to every device).  T[k] is block k's row-ordered copy on its device (local column ids), or null
// for a block without entries.  count(): row counts over the blocks, scanned into the whole matrix's row pointer P on
// device 0 and copied to the host.  offsets(rb): where every block's piece of every row starts in the arrays of the
// row's owner (rows [rb[q], rb[q+1]) belong to owner q, relative to the owner's first row), on the block's device.
// push(rb, d): every block pushes its pieces into the owners' arrays d over peer memory, asynchronously on its stream;
// block order is column order inside a row, so the rows come out as the one-GPU transpose has them.
struct RowExchange {
  sb200_sharded* s;
  std::vector<const sb200_matrix*> T;
  TpPtrs tp{};
  int32_t* tpc = nullptr;  // device 0: copies of every block's row pointer
  uint32_t* cnt = nullptr;
  int32_t* P = nullptr;
  void* ws = nullptr;
  int64_t* dst = nullptr;
  std::vector<int64_t*> dstk;  // device k: its slice of dst
  RowExchange(sb200_sharded* sh, std::vector<const sb200_matrix*> t) : s(sh), T(std::move(t)), dstk(sh->world, nullptr) {}
  ~RowExchange() {  // released on every way out, once nothing reads it any more
    sync_blocks(s);
    for (int k = s->world - 1; k > 0; --k) {
      DeviceGuard g(s->blocks[k]->device);
      pool_free(dstk[k], s->blocks[k]->stream);
    }
    cudaStream_t st0 = s->blocks[0]->stream;
    DeviceGuard g(s->blocks[0]->device);
    pool_free(tpc, st0);
    pool_free(cnt, st0);
    pool_free(P, st0);
    pool_free(ws, st0);
    pool_free(dst, st0);
    cudaGetLastError();
  }
  unsigned grid() const { return static_cast<unsigned>(std::min<int64_t>((static_cast<int64_t>(s->nrow) + 255) / 256, 4096)); }

  int count(int32_t* p_host) {
    const int W = s->world;
    const int32_t nrow = s->nrow;
    sb200_matrix* m0 = s->blocks[0];
    cudaStream_t st0 = m0->stream;
    DeviceGuard g(m0->device);
    // the library's arrays are pool memory, which peers cannot address: bring the (small) row pointers to device 0
    const size_t pb = sizeof(int32_t) * (static_cast<size_t>(nrow) + 1);
    SB_TRY(pool_alloc(reinterpret_cast<void**>(&tpc), pb * W, st0));
    for (int k = 0; k < PUSH_MAX_RANKS; ++k) tp.p[k] = k < W ? tpc + static_cast<size_t>(k) * (nrow + 1) : nullptr;
    for (int k = 0; k < W; ++k) {
      int32_t* to = tpc + static_cast<size_t>(k) * (nrow + 1);
      if (T[k])
        SB_CUDA(cudaMemcpyPeerAsync(to, m0->device, T[k]->d_p, s->blocks[k]->device, pb, st0));
      else
        SB_CUDA(cudaMemsetAsync(to, 0, pb, st0));
    }
    const size_t ws_bytes = scan_workspace_bytes(nrow);
    SB_TRY(pool_alloc(reinterpret_cast<void**>(&cnt), sizeof(uint32_t) * static_cast<size_t>(nrow), st0));
    SB_TRY(pool_alloc(reinterpret_cast<void**>(&P), sizeof(int32_t) * (static_cast<size_t>(nrow) + 1), st0));
    SB_TRY(pool_alloc(&ws, ws_bytes, st0));
    shard_row_counts_kernel<<<grid(), 256, 0, st0>>>(tp, W, nrow, cnt);
    count_launch();
    SB_CUDA(cudaGetLastError());
    SB_TRY(exclusive_scan_u32(st0, cnt, P, nrow, nullptr, ws, ws_bytes));
    SB_CUDA(cudaMemcpyAsync(p_host, P, sizeof(int32_t) * (static_cast<size_t>(nrow) + 1), cudaMemcpyDeviceToHost, st0));
    SB_CUDA(cudaStreamSynchronize(st0));
    if (p_host[nrow] != s->nnz) return fail(SB200_E_CUDA, "sharded rows: the blocks' row counts do not add up to nnz");
    return SB200_OK;
  }

  int offsets(const RowBounds& rb) {
    const int W = s->world;
    const int32_t nrow = s->nrow;
    sb200_matrix* m0 = s->blocks[0];
    {
      DeviceGuard g(m0->device);
      SB_TRY(pool_alloc(reinterpret_cast<void**>(&dst), sizeof(int64_t) * static_cast<size_t>(W) * nrow, m0->stream));
      shard_row_dst_kernel<<<grid(), 256, 0, m0->stream>>>(tp, W, nrow, P, rb, dst);
      count_launch();
      SB_CUDA(cudaGetLastError());
      SB_CUDA(cudaStreamSynchronize(m0->stream));
    }
    dstk[0] = dst;
    for (int k = 1; k < W; ++k) {
      DeviceGuard gk(s->blocks[k]->device);
      SB_TRY(pool_alloc(reinterpret_cast<void**>(&dstk[k]), sizeof(int64_t) * static_cast<size_t>(nrow), s->blocks[k]->stream));
      SB_CUDA(cudaMemcpyPeerAsync(dstk[k], s->blocks[k]->device, dst + static_cast<int64_t>(k) * nrow, m0->device,
                                  sizeof(int64_t) * static_cast<size_t>(nrow), s->blocks[k]->stream));
    }
    return SB200_OK;
  }

  int push(const RowBounds& rb, const PtrDest& pd) {
    for (int k = 0; k < s->world; ++k) {
      if (!T[k]) continue;
      DeviceGuard gk(s->blocks[k]->device);
      PushRowsSrc a;
      a.p_loc = T[k]->d_p;
      a.cols = T[k]->d_i;
      a.vals = T[k]->d_x;
      a.dst_off = dstk[k];
      a.nrow = s->nrow;
      a.col_offset = static_cast<int32_t>(s->bounds[k]);
      for (int q = 0; q <= PUSH_MAX_RANKS; ++q) a.rb[q] = rb.rb[q];
      int64_t blocks = ((static_cast<int64_t>(s->nrow) + 31) / 32 + 7) / 8;
      if (blocks > 592) blocks = 592;
      push_rows_local_kernel<<<static_cast<unsigned>(blocks), 256, 0, s->blocks[k]->stream>>>(a, s->world, pd);
      count_launch();
      SB_CUDA(cudaGetLastError());
    }
    return SB200_OK;
  }
};

// ---- k-wide products: the rank-ordered reduce of the row-major partials ------------------------------------------------
struct PartialPtrs {
  const double* p[PUSH_MAX_RANKS];  // the blocks' row-major nrow x k partials (peer-readable)
};

constexpr int SUMT_THREADS = 256;
constexpr int SUMT_TILE = 1024;                       // outputs per tile
constexpr int SUMT_U = SUMT_TILE / SUMT_THREADS;      // outputs per thread: their loads are in flight together
constexpr int SUMT_SMEM = 2016;                       // max of tr * (w | 1): the folded last slab, tr = 32, w = 63

// Tile geometry: tc = min(k, 32) columns, tr = the largest multiple of 32 rows with tr * tc <= SUMT_TILE.  For small k a
// tile is many rows of few columns, so every lane has an output whatever k is.  Above 32 the columns go in slabs of 32
// and the last slab takes the k mod 32 left over (33 .. 63 columns): no slab is so narrow that its peer loads, one
// run of w values per row at a row stride of 8k bytes, stop being coalesced.
void sumt_geometry(int64_t k, int* tr, int* tc) {
  *tc = static_cast<int>(k < 32 ? k : 32);
  *tr = (SUMT_TILE / *tc) / 32 * 32;
}

// out (nq x k, column-major) = rows [r0, r0 + nq) of P_0 + P_1 + ... + P_{world-1} (row-major nrow x k), added in rank
// order with __dadd_rn like xg_reduce_kernel: the same bits on every device and every run.  A tile's rows are runs of
// w contiguous values in every partial (one contiguous run of rows * k values when w = k): loaded in order, summed in
// registers, staged in shared memory at an odd pitch, and stored column by column with consecutive lanes on
// consecutive rows.
__global__ void __launch_bounds__(SUMT_THREADS) sharded_sum_transpose_kernel(const __grid_constant__ PartialPtrs P, int world, int64_t k, int64_t r0,
                                                                           int64_t nq, int tr, int tc, double* __restrict__ out) {
  __shared__ double tile[SUMT_SMEM];
  const int64_t row_tiles = (nq + tr - 1) / tr;
  const int64_t slabs = k / tc;  // >= 1; the last one also takes the k mod tc columns left over
  for (int64_t t = blockIdx.x; t < row_tiles * slabs; t += gridDim.x) {
    const int64_t rt = (t / slabs) * tr;  // first row of the tile, relative to r0
    const int64_t c0 = (t % slabs) * tc;  // first column
    const int w = static_cast<int>(t % slabs == slabs - 1 ? k - c0 : tc);
    const int rows = static_cast<int>(nq - rt < tr ? nq - rt : tr);
    const int pitch = w | 1;  // odd: the column-wise reads below hit 32 different banks
    const int n = rows * w;
    const int64_t base = (r0 + rt) * k + c0;
    for (int e0 = threadIdx.x; e0 < n; e0 += SUMT_THREADS * SUMT_U) {
      int64_t off[SUMT_U];
      double acc[SUMT_U];
#pragma unroll
      for (int u = 0; u < SUMT_U; ++u) {
        const int e = e0 + u * SUMT_THREADS;
        off[u] = e < n ? base + static_cast<int64_t>(e / w) * k + e % w : 0;
        acc[u] = e < n ? P.p[0][off[u]] : 0.0;
      }
      for (int q = 1; q < world; ++q) {
        const double* __restrict__ pq = P.p[q];
        double v[SUMT_U];
#pragma unroll
        for (int u = 0; u < SUMT_U; ++u) v[u] = e0 + u * SUMT_THREADS < n ? pq[off[u]] : 0.0;
#pragma unroll
        for (int u = 0; u < SUMT_U; ++u) acc[u] = __dadd_rn(acc[u], v[u]);
      }
#pragma unroll
      for (int u = 0; u < SUMT_U; ++u) {
        const int e = e0 + u * SUMT_THREADS;
        if (e < n) tile[(e / w) * pitch + e % w] = acc[u];
      }
    }
    __syncthreads();
    for (int e = threadIdx.x; e < n; e += SUMT_THREADS) {
      const int c = e / rows, r = e % rows;
      out[(c0 + c) * nq + rt + r] = tile[r * pitch + c];
    }
    __syncthreads();
  }
}

int launch_sum_transpose(cudaStream_t st, int sm_count, const PartialPtrs& P, int world, int64_t k, int64_t r0, int64_t nq,
                         double* out) {
  if (nq == 0 || k == 0) return SB200_OK;
  int tr = 0, tc = 0;
  sumt_geometry(k, &tr, &tc);
  const int64_t tiles = ((nq + tr - 1) / tr) * (k / tc);
  const int64_t grid = std::min<int64_t>(tiles, static_cast<int64_t>(sm_count) * 8);
  sharded_sum_transpose_kernel<<<static_cast<unsigned>(grid), SUMT_THREADS, 0, st>>>(P, world, k, r0, nq, tr, tc, out);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return SB200_OK;
}

int ensure_peer_partials(sb200_sharded* s) {
  if (!s->ev_partial.empty()) return SB200_OK;
  s->peer_partial.assign(s->world, nullptr);
  s->peer_partial_bytes.assign(s->world, 0);
  s->ev_partial.assign(s->world, nullptr);
  s->ev_reduced.assign(s->world, nullptr);
  for (int w = 0; w < s->world; ++w) {
    DeviceGuard g(s->devices[w]);
    SB_CUDA(cudaEventCreateWithFlags(&s->ev_partial[w], cudaEventDisableTiming));
    SB_CUDA(cudaEventCreateWithFlags(&s->ev_reduced[w], cudaEventDisableTiming));
  }
  return SB200_OK;
}

// block w's partial holds at least `bytes`; the current device is block w's.  `what` names the partial in the error.
int ensure_partial(sb200_sharded* s, int w, size_t bytes, const char* what) {
  if (s->peer_partial_bytes[w] >= bytes) return SB200_OK;
  for (cudaEvent_t e : s->ev_reduced) SB_CUDA(cudaEventSynchronize(e));  // no reader still has the old one in flight
  if (s->peer_partial[w]) cudaFree(s->peer_partial[w]);
  s->peer_partial[w] = nullptr;
  s->peer_partial_bytes[w] = 0;
  if (cudaMalloc(reinterpret_cast<void**>(&s->peer_partial[w]), bytes) != cudaSuccess) {
    cudaGetLastError();
    s->peer_partial[w] = nullptr;
    return fail(SB200_E_NOMEM, std::string(what) + " does not fit on device " + std::to_string(s->devices[w]));
  }
  s->peer_partial_bytes[w] = bytes;
  return SB200_OK;
}

int sharded_spmm_args(const sb200_sharded* s, bool transposed, const double* B, int64_t k, const double* Y) {
  if (k < 0) return fail(SB200_E_INVALID, "spmm: k must not be negative");
  const int64_t b_rows = transposed ? s->nrow : s->ncol, y_rows = transposed ? s->ncol : s->nrow;
  if (k > 0 && ((b_rows > 0 && !B) || (y_rows > 0 && !Y))) return fail(SB200_E_INVALID, "spmm: NULL operand or result");
  return SB200_OK;
}

// Y = A B (transposed = false) or A^T B, host buffers, column-major.  Four phases: operands up (a thread per block,
// blocking), launches (this thread, device after device, ordered by events), results home (a thread per block), and a
// synchronisation of every stream whatever happened before.
int run_block_product(sb200_sharded* s, bool transposed, const double* B, int64_t k, double* Y) {
  const int W = s->world;
  const int64_t nrow = s->nrow, ncol = s->ncol;
  const int64_t b_rows = transposed ? nrow : ncol, y_rows = transposed ? ncol : nrow;
  if (k == 0 || y_rows == 0) return SB200_OK;
  if ((b_rows > 0 && k > INT64_MAX / 8 / b_rows) || k > INT64_MAX / 8 / y_rows)
    return fail(SB200_E_NOMEM, "spmm: the dense operand or result does not fit in device memory");
  WallTrace tr(transposed ? "sharded spmm_t" : "sharded spmm");
  DeviceGuard restore(s->blocks[0]->device);
  SB_TRY(ensure_peer_partials(s));
  // rows of the operand block w reads and of the result piece it brings home
  auto b_lo = [&](int w) { return transposed ? int64_t{0} : s->bounds[w]; };
  auto b_n = [&](int w) { return transposed ? nrow : s->bounds[w + 1] - s->bounds[w]; };
  auto y_lo = [&](int w) { return transposed ? s->bounds[w] : nrow * w / W; };
  auto y_n = [&](int w) { return transposed ? s->bounds[w + 1] - s->bounds[w] : nrow * (w + 1) / W - nrow * w / W; };
  std::vector<double*> dB(W, nullptr), dY(W, nullptr);
  int rc = SB200_OK;
  for (int w = 0; w < W && rc == SB200_OK; ++w) {
    sb200_matrix* m = s->blocks[w];
    DeviceGuard g(m->device);
    const double partial = transposed ? 0.0 : 8.0 * static_cast<double>(k) * static_cast<double>(nrow);
    const double need = 8.0 * static_cast<double>(k) * static_cast<double>(b_n(w) + y_n(w)) +
                        std::max(0.0, partial - static_cast<double>(s->peer_partial_bytes[w]));
    if (need > static_cast<double>(device_free_bytes())) {
      rc = fail(SB200_E_NOMEM, "sharded spmm: the operand, result and partial of block " + std::to_string(w) +
                                   " do not fit on device " + std::to_string(m->device));
      break;
    }
    rc = pool_alloc(reinterpret_cast<void**>(&dB[w]), std::max<size_t>(16, sizeof(double) * static_cast<size_t>(b_n(w) * k)), m->stream);
    if (rc == SB200_OK)
      rc = pool_alloc(reinterpret_cast<void**>(&dY[w]), std::max<size_t>(16, sizeof(double) * static_cast<size_t>(y_n(w) * k)), m->stream);
    if (rc == SB200_OK && !transposed) rc = ensure_partial(s, w, sizeof(double) * static_cast<size_t>(nrow * k), "sharded spmm: the row-major partial (8 nrow k bytes)");
  }
  tr.phase("scratch");
  // block w's piece of B or Y: n rows of each of the k columns of the host matrix (`rows` rows), blocking
  auto copy_piece = [&](int w, cudaMemcpyKind kind, double* host, int64_t rows, double* dev, int64_t n) {
    sb200_matrix* m = s->blocks[w];
    const size_t width = sizeof(double) * static_cast<size_t>(n);
    SB_TRY(host_copies(m->device, m->stream, kind, {{host, dev, width, static_cast<size_t>(k), sizeof(double) * static_cast<size_t>(rows), width}}));
    SB_CUDA(cudaStreamSynchronize(m->stream));
    return SB200_OK;
  };
  // 1. operands up: block w's rows of B, a strided slice (A B) or all of it (A^T B)
  if (rc == SB200_OK)
    rc = on_every_block(s, "sharded spmm: operand upload", [&](int w) {
      return copy_piece(w, cudaMemcpyHostToDevice, const_cast<double*>(B) + b_lo(w), b_rows, dB[w], b_n(w));
    });
  tr.phase("operands up");
  // 2. the device part, from every operand resident to every result piece complete
  DevicePartTimer dp(s, tr.on);
  if (rc == SB200_OK) rc = dp.start();
  if (rc == SB200_OK && transposed) {
    for (int w = 0; w < W && rc == SB200_OK; ++w) {
      DeviceGuard g(s->blocks[w]->device);
      rc = launch_spmm(s->blocks[w], true, dB[w], k, dY[w]);
    }
  } else if (rc == SB200_OK) {
    PartialPtrs P{};
    for (int w = 0; w < W && rc == SB200_OK; ++w) {
      sb200_matrix* m = s->blocks[w];
      DeviceGuard g(m->device);
      P.p[w] = s->peer_partial[w];
      rc = launch_spmm_rm(m, false, dB[w], k, s->peer_partial[w]);
      if (rc == SB200_OK && cudaEventRecord(s->ev_partial[w], m->stream) != cudaSuccess) rc = fail(SB200_E_CUDA, "cudaEventRecord");
    }
    for (int q = 0; q < W && rc == SB200_OK; ++q) {
      sb200_matrix* m = s->blocks[q];
      DeviceGuard g(m->device);
      for (int w = 0; w < W && rc == SB200_OK; ++w)
        if (cudaStreamWaitEvent(m->stream, s->ev_partial[w], 0) != cudaSuccess) rc = fail(SB200_E_CUDA, "cudaStreamWaitEvent");
      if (rc == SB200_OK) rc = launch_sum_transpose(m->stream, m->sm_count, P, W, k, y_lo(q), y_n(q), dY[q]);
      if (rc == SB200_OK && cudaEventRecord(s->ev_reduced[q], m->stream) != cudaSuccess) rc = fail(SB200_E_CUDA, "cudaEventRecord");
    }
  }
  if (rc == SB200_OK) rc = dp.stop();
  tr.phase("launched");
  // 3. results home: block w's piece of Y, `y_n(w)` rows of every column
  if (rc == SB200_OK)
    rc = on_every_block(s, "sharded spmm: result download",
                        [&](int w) { return copy_piece(w, cudaMemcpyDeviceToHost, Y + y_lo(w), y_rows, dY[w], y_n(w)); });
  tr.phase("results home");
  // 4. every stream is waited for (no partial is rewritten or freed while a reader may still run), scratch released
  const cudaError_t e = sync_blocks(s);
  if (e != cudaSuccess && rc == SB200_OK) rc = cuda_fail(e, "sharded spmm", __FILE__, __LINE__);
  for (int w = 0; w < W; ++w) {
    sb200_matrix* m = s->blocks[w];
    DeviceGuard g(m->device);
    pool_free(dB[w], m->stream);
    pool_free(dY[w], m->stream);
  }
  if (rc == SB200_OK) dp.report(tr.title);
  if (rc == SB200_E_NOMEM) cudaGetLastError();  // a refused allocation leaves the streams usable
  return rc;
}

// ---- rowVars: the rank-ordered reduce of the blocks' sums of squares and counts ---------------------------------------
// Rows [r0, r1): S and cnt are the blocks' partials (P.p[w][r] and P.p[w][nrow + r]) added in block order with __dadd_rn,
// like xg_reduce_kernel, and out[r] = var_from_sums(S, cnt, mean[r], n).  The same bits on every device and every run.
__global__ void __launch_bounds__(256) sharded_row_var_kernel(const __grid_constant__ PartialPtrs P, int world, int64_t nrow, int64_t r0,
                                                              int64_t r1, const double* __restrict__ mean, double n,
                                                              double* __restrict__ out) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = r0 + static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < r1; r += stride) {
    double S = P.p[0][r], c = P.p[0][nrow + r];
    for (int q = 1; q < world; ++q) {
      S = __dadd_rn(S, P.p[q][r]);
      c = __dadd_rn(c, P.p[q][nrow + r]);
    }
    out[r] = var_from_sums(S, c, mean[r], n);
  }
}

// rowVars on every device: (1) the global row means as sb200_sharded_row_means computes them, in every window; (2) every
// block's S and counts over its own columns into its peer-readable partial (16 nrow bytes, kept between calls); (3)
// device q reduces rows [q nrow / W, (q+1) nrow / W) of all partials and copies them home.  Steps 2 and 3 are ordered
// by CUDA events only, so blocks may share a device.
int run_row_vars(sb200_sharded* s, double* out) {
  const int W = s->world;
  const int64_t nrow = s->nrow;
  DeviceGuard restore(s->blocks[0]->device);
  SB_TRY(ensure_peer_partials(s));
  int64_t mean_off = 0;
  int rc = rows_into_windows(s, SWEEP_ROWSUM, nullptr, static_cast<double>(s->ncol), &mean_off);
  PartialPtrs P{};
  for (int w = 0; w < W && rc == SB200_OK; ++w) {
    sb200_matrix* m = s->blocks[w];
    DeviceGuard g(m->device);
    rc = ensure_partial(s, w, 2 * sizeof(double) * static_cast<size_t>(nrow), "sharded rowVars: the sums and counts (16 nrow bytes)");
    if (rc != SB200_OK) break;
    P.p[w] = s->peer_partial[w];
    const double* mean = reinterpret_cast<const double*>(exchange_window_base(s->windows[w]) + mean_off);
    rc = launch_row_var_sums(m, mean, s->peer_partial[w], s->peer_partial[w] + nrow);
    if (rc == SB200_OK && cudaEventRecord(s->ev_partial[w], m->stream) != cudaSuccess) rc = fail(SB200_E_CUDA, "cudaEventRecord");
  }
  for (int q = 0; q < W && rc == SB200_OK; ++q) {
    sb200_matrix* m = s->blocks[q];
    DeviceGuard g(m->device);
    for (int w = 0; w < W && rc == SB200_OK; ++w)
      if (cudaStreamWaitEvent(m->stream, s->ev_partial[w], 0) != cudaSuccess) rc = fail(SB200_E_CUDA, "cudaStreamWaitEvent");
    const int64_t r0 = nrow * q / W, r1 = nrow * (q + 1) / W;
    if (rc != SB200_OK || r1 == r0) continue;
    const double* mean = reinterpret_cast<const double*>(exchange_window_base(s->windows[q]) + mean_off);
    int64_t blocks = (r1 - r0 + 255) / 256;
    if (blocks > static_cast<int64_t>(m->sm_count) * 8) blocks = static_cast<int64_t>(m->sm_count) * 8;
    sharded_row_var_kernel<<<static_cast<unsigned>(blocks), 256, 0, m->stream>>>(P, W, nrow, r0, r1, mean, static_cast<double>(s->ncol),
                                                                               m->d_stage_out);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaEventRecord(s->ev_reduced[q], m->stream);
    if (e == cudaSuccess)
      e = cudaMemcpyAsync(out + r0, m->d_stage_out + r0, sizeof(double) * static_cast<size_t>(r1 - r0), cudaMemcpyDeviceToHost, m->stream);
    if (e != cudaSuccess) rc = cuda_fail(e, "sharded rowVars: reduce", __FILE__, __LINE__);
  }
  const cudaError_t e = sync_blocks(s);
  if (e != cudaSuccess && rc == SB200_OK) rc = cuda_fail(e, "sharded rowVars", __FILE__, __LINE__);
  if (rc == SB200_E_NOMEM) cudaGetLastError();
  return rc;
}

}  // namespace
}  // namespace sb200

using namespace sb200;

extern "C" {

int sb200_sharded_create(const int32_t* i, const int32_t* p, const double* x, int32_t nrow, int32_t ncol, int64_t nnz, int n_gpus,
                         const int* devices, unsigned flags, sb200_sharded** out) {
  if (!out) return fail(SB200_E_INVALID, "out is NULL");
  *out = nullptr;
  if (!p || (nnz > 0 && (!i || !x))) return fail(SB200_E_INVALID, "NULL slot array");
  if (nrow < 0 || ncol < 0 || nnz < 0) return fail(SB200_E_INVALID, "negative dimension");
  if (n_gpus < 1 || n_gpus > 16) return fail(SB200_E_INVALID, "n_gpus must be 1..16 (the GPUs of one node)");
  int have = 0;
  if (cudaGetDeviceCount(&have) != cudaSuccess || have <= 0) {
    cudaGetLastError();
    return fail(SB200_E_NODEVICE, "no CUDA device available: libsparse_b200 has no CPU fallback");
  }
  // the host arrays are validated on the device block by block; the split itself needs p[0] = 0, p monotone, p[ncol] = nnz
  if (p[0] != 0 || p[ncol] != nnz) return fail(SB200_E_STRUCTURE, "p[0] must be 0 and p[ncol] must be nnz");
  sb200_sharded* s = new (std::nothrow) sb200_sharded();
  if (!s) return fail(SB200_E_NOMEM, "host allocation failed");
  s->magic = SHARDED_MAGIC;
  s->world = n_gpus;
  s->nrow = nrow;
  s->ncol = ncol;
  s->nnz = nnz;
  s->devices.resize(n_gpus);
  for (int k = 0; k < n_gpus; ++k) {
    s->devices[k] = devices ? devices[k] : k;
    if (s->devices[k] < 0 || s->devices[k] >= have) {
      destroy_sharded(s);
      return fail(SB200_E_NODEVICE, "requested CUDA device " + std::to_string(devices ? devices[k] : k) + " not present");
    }
  }
  // nnz-balanced contiguous column blocks (SURVEY.md 8e)
  s->bounds.resize(n_gpus + 1);
  nnz_balanced_bounds(p, ncol, nnz, n_gpus, s->bounds.data());
  s->blocks.assign(n_gpus, nullptr);
  s->windows.assign(n_gpus, nullptr);
  // upload the blocks concurrently: one worker per device
  WallTrace tr("sharded create");
  int rc = on_every_block(s, "sharded create", [&](int k) {
    const int64_t c0 = s->bounds[k], c1 = s->bounds[k + 1];
    const int64_t k0 = p[c0], k1 = p[c1];
    std::vector<int32_t> pk(static_cast<size_t>(c1 - c0) + 1);
    for (int64_t c = c0; c <= c1; ++c) {
      pk[c - c0] = static_cast<int32_t>(p[c] - k0);
      if (c > c0 && p[c] < p[c - 1]) return fail(SB200_E_STRUCTURE, "p is not monotone");
    }
    return sb200_matrix_create(i + k0, pk.data(), x + k0, nrow, static_cast<int32_t>(c1 - c0), k1 - k0, s->devices[k], flags & ~SB200_LAZY_ROWS,
                               &s->blocks[k]);
  });
  tr.phase("blocks uploaded");
  // windows: [row partial | row result], 256-byte aligned, behind the exchange header
  const int64_t vec = ((static_cast<int64_t>(nrow > 0 ? nrow : 1) * 8 + 255) / 256) * 256;
  int prev = 0;
  cudaGetDevice(&prev);
  for (int k = 0; k < n_gpus && rc == SB200_OK; ++k) {
    unsigned char handle[64];
    rc = sb200_exchange_create(s->devices[k], 2 * vec, &s->windows[k], handle);
  }
  tr.phase("windows allocated");
  if (rc == SB200_OK) rc = exchange_connect_local(s->windows.data(), n_gpus);
  cudaSetDevice(prev);
  tr.phase("peers connected");
  if (rc != SB200_OK) {
    const std::string msg = sb200_last_error();
    destroy_sharded(s);
    return fail(rc, msg);
  }
  void* base = nullptr;
  int64_t data_off = 0, bytes = 0;
  sb200_exchange_window(s->windows[0], &base, &data_off, &bytes);
  s->partial_off = data_off;
  s->result_off = data_off + vec;
  *out = s;
  return SB200_OK;
}

int sb200_sharded_destroy(sb200_sharded* s) {
  if (!s) return SB200_OK;
  SB_TRY(check_sharded(s));
  int prev = 0;
  cudaGetDevice(&prev);
  destroy_sharded(s);
  cudaSetDevice(prev);
  return SB200_OK;
}

int sb200_sharded_info(const sb200_sharded* s, int* n_gpus, int64_t* bounds) {
  SB_TRY(check_sharded(s));
  if (n_gpus) *n_gpus = s->world;
  if (bounds)
    for (int k = 0; k <= s->world; ++k) bounds[k] = s->bounds[k];
  return SB200_OK;
}

int sb200_sharded_block(const sb200_sharded* s, int k, sb200_matrix** block) {
  SB_TRY(check_sharded(s));
  if (k < 0 || k >= s->world || !block) return fail(SB200_E_INVALID, "sb200_sharded_block: bad block index");
  *block = s->blocks[k];
  return SB200_OK;
}

int sb200_sharded_col_sums(sb200_sharded* s, double* out) {
  SB_TRY(check_sharded(s));
  return run_columns(s, SWEEP_COLSUM, nullptr, 0.0, out);
}
int sb200_sharded_col_means(sb200_sharded* s, double* out) {
  SB_TRY(check_sharded(s));
  if (s->nrow == 0) {  // RcppSparse.h:148: sums / Dim[0]; 0/0 = NaN there and here
    for (int32_t c = 0; c < s->ncol; ++c) out[c] = 0.0 / static_cast<double>(s->nrow);
    return SB200_OK;
  }
  return run_columns(s, SWEEP_COLSUM, nullptr, static_cast<double>(s->nrow), out);
}
int sb200_sharded_spmv_t(sb200_sharded* s, const double* v, double* y) {
  SB_TRY(check_sharded(s));
  if (s->nrow > 0 && !v) return fail(SB200_E_INVALID, "operand vector is NULL");
  return run_columns(s, SWEEP_SPMV_T, v, 0.0, y);
}
int sb200_sharded_row_sums(sb200_sharded* s, double* out) {
  SB_TRY(check_sharded(s));
  return run_rows(s, SWEEP_ROWSUM, nullptr, 0.0, out);
}
int sb200_sharded_row_means(sb200_sharded* s, double* out) {
  SB_TRY(check_sharded(s));
  if (s->ncol == 0) {
    for (int32_t r = 0; r < s->nrow; ++r) out[r] = 0.0 / static_cast<double>(s->ncol);
    return SB200_OK;
  }
  return run_rows(s, SWEEP_ROWSUM, nullptr, static_cast<double>(s->ncol), out);
}
int sb200_sharded_col_vars(sb200_sharded* s, double* out) {
  SB_TRY(check_sharded(s));
  return run_columns(s, SWEEP_COLVAR, nullptr, 0.0, out);
}
int sb200_sharded_row_vars(sb200_sharded* s, double* out) {
  SB_TRY(check_sharded(s));
  if (s->nrow == 0) return SB200_OK;
  if (!out) return fail(SB200_E_INVALID, "output buffer is NULL");
  if (s->ncol < 2) {  // no variance of fewer than two values (R: NA)
    for (int32_t r = 0; r < s->nrow; ++r) out[r] = std::numeric_limits<double>::quiet_NaN();
    return SB200_OK;
  }
  return run_row_vars(s, out);
}
int sb200_sharded_spmv(sb200_sharded* s, const double* v, double* y) {
  SB_TRY(check_sharded(s));
  if (s->ncol > 0 && !v) return fail(SB200_E_INVALID, "operand vector is NULL");
  return run_rows(s, SWEEP_SPMV, v, 0.0, y);
}
int sb200_sharded_spmm(sb200_sharded* s, const double* B, int64_t k, double* Y) {
  SB_TRY(check_sharded(s));
  SB_TRY(sharded_spmm_args(s, false, B, k, Y));
  return run_block_product(s, false, B, k, Y);
}
int sb200_sharded_spmm_t(sb200_sharded* s, const double* B, int64_t k, double* Y) {
  SB_TRY(check_sharded(s));
  SB_TRY(sharded_spmm_args(s, true, B, k, Y));
  return run_block_product(s, true, B, k, Y);
}


// CSC(A^T) of the whole matrix into host arrays (RcppSparse.h:375-385): every device transposes its column block, the
// row counts are summed and scanned on device 0 (p_out), rows are dealt to the devices in nnz-balanced contiguous
// ranges, every device pushes its piece of every row straight to its place in the owner's arrays over peer memory
// (block order = column order inside a row: bit-exact), and every owner copies its range of i_out / x_out to the host
// over its own PCIe link.
int sb200_sharded_transpose(sb200_sharded* s, int32_t* p_out, int32_t* i_out, double* x_out) {
  SB_TRY(check_sharded(s));
  if (!p_out || (s->nnz > 0 && (!i_out || !x_out))) return fail(SB200_E_INVALID, "NULL output array");
  const int W = s->world;
  const int32_t nrow = s->nrow;
  if (s->nnz == 0 || nrow == 0) {
    for (int64_t r = 0; r <= nrow; ++r) p_out[r] = 0;
    return SB200_OK;
  }
  DeviceGuard restore(s->blocks[0]->device);
  WallTrace tr("sharded transpose");
  std::vector<sb200_matrix*> T(W, nullptr);
  struct Scratch {  // the local transposes and the owners' arrays are released on every way out
    std::vector<sb200_matrix*>& T;
    sb200_sharded* s;
    std::vector<int32_t*> oc;  // the owners' arrays: plain cudaMalloc, visible to the peers (pool memory is not)
    std::vector<double*> ov;
    ~Scratch() {
      sync_blocks(s);
      for (int k = 0; k < s->world; ++k) {
        DeviceGuard g(s->blocks[k]->device);
        if (k < static_cast<int>(oc.size()) && oc[k]) cudaFree(oc[k]);
        if (k < static_cast<int>(ov.size()) && ov[k]) cudaFree(ov[k]);
        if (T[k]) sb200_matrix_destroy(T[k]);
      }
      cudaGetLastError();
    }
  } sc{T, s};
  // 1. local transposes, concurrently (the entry point blocks)
  int rc = on_every_block(s, "sharded transpose", [&](int k) { return sb200_transpose_dev(s->blocks[k], &T[k]); });
  tr.phase("local transposes");
  SB_TRY(rc);
  // 2. row counts over the blocks -> p_out
  RowExchange rx(s, std::vector<const sb200_matrix*>(T.begin(), T.end()));
  SB_TRY(rx.count(p_out));
  tr.phase("row counts, scan, p_out");
  // 3. rows dealt to the devices: nnz-balanced contiguous ranges
  RowBounds rb;
  nnz_balanced_bounds(p_out, nrow, s->nnz, W, rb.rb);
  for (int q = W + 1; q <= PUSH_MAX_RANKS; ++q) rb.rb[q] = nrow;
  SB_TRY(rx.offsets(rb));
  // 4. the owners' arrays
  sc.oc.assign(W, nullptr);
  sc.ov.assign(W, nullptr);
  for (int q = 0; q < W; ++q) {
    DeviceGuard gq(s->blocks[q]->device);
    const size_t n = static_cast<size_t>(p_out[rb.rb[q + 1]] - p_out[rb.rb[q]]);
    SB_CUDA(cudaMalloc(reinterpret_cast<void**>(&sc.oc[q]), padded_bytes(sizeof(int32_t) * (n + 1))));
    SB_CUDA(cudaMalloc(reinterpret_cast<void**>(&sc.ov[q]), padded_bytes(sizeof(double) * (n + 1))));
  }
  // 5. every device pushes its pieces
  PtrDest pd;
  for (int q = 0; q < PUSH_MAX_RANKS; ++q) {
    pd.c[q] = q < W ? sc.oc[q] : nullptr;
    pd.v[q] = q < W ? sc.ov[q] : nullptr;
  }
  SB_TRY(rx.push(rb, pd));
  SB_CUDA(sync_blocks(s));
  tr.phase("push");
  // 6. every owner brings its range home over its own link
  rc = on_every_block(s, "sharded transpose: copy to the host", [&](int q) {
    sb200_matrix* m = s->blocks[q];
    const int64_t o = p_out[rb.rb[q]];
    const size_t n = static_cast<size_t>(p_out[rb.rb[q + 1]] - o);
    SB_TRY(host_copies(m->device, m->stream, cudaMemcpyDeviceToHost,
                       {{i_out + o, sc.oc[q], sizeof(int32_t) * n}, {x_out + o, sc.ov[q], sizeof(double) * n}}));
    SB_CUDA(cudaStreamSynchronize(m->stream));
    return SB200_OK;
  });
  tr.phase("copies to the host");
  return rc;
}

// Matrix::crossprod() (RcppSparse.h:158-194): block w computes the full-height slab A^T A_w, result columns
// [bounds[w], bounds[w+1]), which is one contiguous range of the column-major `out`.  Its columns need every whole row that
// has an entry in them, so every block first gets the row-ordered copy of the whole matrix: the blocks' own row-ordered
// copies, their pieces of every row pushed over peer memory into every block's copy (plain cudaMalloc: peers write it).
// The ordered sweep (crossprod.cu, crossprod_slab_kernel) adds every entry in ascending row order, so the result is the
// reference's bit for bit, exactly symmetric, and the same for every split and placement.  Slabs go home from one
// thread per block.
int sb200_sharded_crossprod(sb200_sharded* s, double* out) {
  SB_TRY(check_sharded(s));
  const int W = s->world;
  const int64_t nrow = s->nrow, ncol = s->ncol, nnz = s->nnz;
  if (ncol == 0) return SB200_OK;
  if (!out) return fail(SB200_E_INVALID, "output buffer is NULL");
  if (nnz == 0 || nrow == 0) {  // no products at all: the zero matrix
    for (int64_t c = 0; c < ncol; ++c) memset(out + c * ncol, 0, sizeof(double) * static_cast<size_t>(ncol));
    return SB200_OK;
  }
  WallTrace tr("sharded crossprod");
  DeviceGuard restore(s->blocks[0]->device);
  auto ncol_w = [&](int w) { return s->bounds[w + 1] - s->bounds[w]; };
  // 0. every device must hold the slabs and whole-matrix copies of the blocks it carries
  {
    std::vector<int> seen;
    for (int w = 0; w < W; ++w) {
      const int dev = s->blocks[w]->device;
      if (std::find(seen.begin(), seen.end(), dev) != seen.end()) continue;
      seen.push_back(dev);
      double need = 0.0;
      for (int v = 0; v < W; ++v)
        if (s->blocks[v]->device == dev && ncol_w(v) > 0)
          need += 8.0 * static_cast<double>(ncol) * static_cast<double>(ncol_w(v)) + 12.0 * static_cast<double>(nnz) +
                  4.0 * static_cast<double>(nrow + 1) + 4096.0;
      DeviceGuard g(dev);
      if (need > static_cast<double>(device_free_bytes()))
        return fail(SB200_E_NOMEM, "sharded crossprod: the result slabs (8 ncol ncol_w bytes) and row-ordered copies of the blocks on device " +
                                       std::to_string(dev) + " do not fit");
    }
  }
  struct Scratch {  // released on every way out, after every stream is done with it
    sb200_sharded* s;
    std::vector<sb200_matrix*> tmp;  // temporary row-ordered copies (blocks that keep none)
    std::vector<int32_t*> rp, rc;    // every block's copy of the whole matrix's rows
    std::vector<double*> rv, slab;
    ~Scratch() {
      sync_blocks(s);
      for (int w = 0; w < s->world; ++w) {
        sb200_matrix* m = s->blocks[w];
        DeviceGuard g(m->device);
        if (rc[w]) cudaFree(rc[w]);
        if (rv[w]) cudaFree(rv[w]);
        pool_free(rp[w], m->stream);
        pool_free(slab[w], m->stream);
        if (tmp[w]) sb200_matrix_destroy(tmp[w]);
      }
      cudaGetLastError();
    }
  } sc{s, std::vector<sb200_matrix*>(W, nullptr), std::vector<int32_t*>(W, nullptr), std::vector<int32_t*>(W, nullptr),
       std::vector<double*>(W, nullptr), std::vector<double*>(W, nullptr)};
  // 1. the blocks' row-ordered copies: the one a block keeps (built now where it fits, as sb200_crossprod does), else
  //    a temporary transpose
  std::vector<const sb200_matrix*> T(W, nullptr);
  SB_TRY(on_every_block(s, "sharded crossprod: row-ordered copy", [&](int w) {
    sb200_matrix* m = s->blocks[w];
    if (m->nnz == 0) return SB200_OK;
    if ((T[w] = crossprod_row_copy(m))) return SB200_OK;
    SB_TRY(sb200_transpose_dev(m, &sc.tmp[w]));
    T[w] = sc.tmp[w];
    return SB200_OK;
  }));
  tr.phase("row-ordered copies");
  // 2. the whole matrix's row pointer, and where every block's piece of every row starts in it
  RowExchange rx(s, T);
  std::vector<int32_t> P(static_cast<size_t>(nrow) + 1);
  SB_TRY(rx.count(P.data()));
  RowBounds all;  // one owner of every row: each block's copy holds them all
  all.rb[0] = 0;
  for (int q = 1; q <= PUSH_MAX_RANKS; ++q) all.rb[q] = static_cast<int32_t>(nrow);
  SB_TRY(rx.offsets(all));
  // 3. every block's copy and slab
  int rc = SB200_OK;
  for (int w = 0; w < W && rc == SB200_OK; ++w) {
    if (ncol_w(w) == 0) continue;
    sb200_matrix* m = s->blocks[w];
    DeviceGuard g(m->device);
    if (cudaMalloc(reinterpret_cast<void**>(&sc.rc[w]), padded_bytes(sizeof(int32_t) * static_cast<size_t>(nnz))) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&sc.rv[w]), padded_bytes(sizeof(double) * static_cast<size_t>(nnz))) != cudaSuccess) {
      cudaGetLastError();
      rc = fail(SB200_E_NOMEM, "sharded crossprod: the row-ordered copy does not fit on device " + std::to_string(m->device));
      break;
    }
    rc = pool_alloc(reinterpret_cast<void**>(&sc.rp[w]), sizeof(int32_t) * static_cast<size_t>(nrow + 1), m->stream);
    if (rc == SB200_OK)
      rc = pool_alloc(reinterpret_cast<void**>(&sc.slab[w]), sizeof(double) * static_cast<size_t>(ncol) * static_cast<size_t>(ncol_w(w)),
                      m->stream);
    if (rc != SB200_OK) {
      cudaGetLastError();
      rc = fail(SB200_E_NOMEM, "sharded crossprod: the result slab of block " + std::to_string(w) + " does not fit on device " +
                                   std::to_string(m->device));
    }
  }
  if (rc != SB200_OK) return rc;
  tr.phase("scratch");
  // 4. the device part: the gather, then the ordered sweep
  DevicePartTimer dp(s, tr.on);
  SB_TRY(dp.start());
  for (int w = 0; w < W; ++w) {
    if (ncol_w(w) == 0) continue;
    sb200_matrix* m0 = s->blocks[0];
    DeviceGuard g(s->blocks[w]->device);
    SB_CUDA(cudaMemcpyPeerAsync(sc.rp[w], s->blocks[w]->device, rx.P, m0->device, sizeof(int32_t) * static_cast<size_t>(nrow + 1),
                                s->blocks[w]->stream));
    PtrDest pd{};
    pd.c[0] = sc.rc[w];
    pd.v[0] = sc.rv[w];
    SB_TRY(rx.push(all, pd));
  }
  SB_CUDA(sync_blocks(s));  // every piece has landed in every copy
  tr.phase("rows gathered");
  for (int w = 0; w < W; ++w) {
    DeviceGuard g(s->blocks[w]->device);
    SB_TRY(launch_crossprod_slab(s->blocks[w], sc.rp[w], sc.rc[w], sc.rv[w], ncol, sc.slab[w]));
  }
  SB_TRY(dp.stop());
  tr.phase("launched");
  // 5. every slab home over its block's own link
  SB_TRY(on_every_block(s, "sharded crossprod: result download", [&](int w) {
    sb200_matrix* m = s->blocks[w];
    const size_t bytes = sizeof(double) * static_cast<size_t>(ncol) * static_cast<size_t>(ncol_w(w));
    SB_TRY(host_copies(m->device, m->stream, cudaMemcpyDeviceToHost, {{out + s->bounds[w] * ncol, sc.slab[w], bytes}}));
    SB_CUDA(cudaStreamSynchronize(m->stream));
    return SB200_OK;
  }));
  tr.phase("results home");
  dp.report(tr.title);
  return SB200_OK;
}

}  // extern "C"
