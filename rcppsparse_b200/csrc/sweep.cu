// The column sweep on B200: merge-path balanced, TMA-staged, persistent.
//
// Replaces the serial loops of the reference (zdebruine/RcppSparse):
//   colSums / columnSums   RcppSparse.h:131-137, src/example.cpp:26-32      -> SWEEP_COLSUM
//   colMeans               RcppSparse.h:145-150                             -> SWEEP_COLSUM, divisor = nrow
//   A^T v (iterator idiom, gather shape of :133-135)                        -> SWEEP_SPMV_T
//   A v   (iterator idiom, scatter shape of :140-142)                       -> SWEEP_SPMV
//   rowSums / rowMeans     RcppSparse.h:138-144,151-156                     -> rowsum_stream_kernel
//   colVars (second pass: sum of (x - mean)^2 per column, formula at the store) -> SWEEP_COLVAR (vars.cu)
//
// Work decomposition.  The sweep is a merge of two sorted lists: the column end offsets
// A[c] = p[c+1] and the entry indices B[k] = k.  One merge "item" is either "consume entry
// k" or "column c ends"; there are ncol + nnz items whatever the column-length distribution,
// so cutting the merge path into equal tiles balances power-law columns, empty columns and
// one-dense-column matrices alike.  plan[t] (built once per matrix, cached in the handle)
// holds the column coordinate of the path at diagonal t*TILE.
//
// One persistent CTA per SM slot owns a CONTIGUOUS range of tiles.  Thread 0 drives a
// STAGES-deep ring: for each upcoming tile it issues 1-D bulk async copies (cp.async.bulk ->
// SASS UBLKCP, the TMA engine) of the tile's x segment, its column-end window of p and (for
// the gather) its i segment into shared memory, completion counted on an mbarrier.  All
// threads then walk IPT items each out of shared memory (IPT odd => conflict-free 8-byte
// reads), a warp-shuffle segmented scan stitches the per-thread partial sums, and completed
// columns are stored directly.  Contiguous tile ranges mean the running partial of a column
// that spans tiles stays in a register; only G-1 cross-CTA carries exist, and the last CTA
// to finish (ticket) folds them in a fixed order => results are bit-stable run to run.
//
// Roofline: HBM.  Algorithmic bytes 8N+4(n+1)+8n (COLSUM), 12N+4(n+1)+8m+8n (SPMV_T, SPMV),
// 12N+8m (rowsum).  No tensor cores: nothing here is a dense contraction.
#include <cuda_runtime.h>
#include <limits.h>
#include <stdint.h>
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"
#include "ptx.cuh"

namespace sb200 {

// Number of column-end items that precede diagonal d of the merge path.  Ends win ties:
// a column whose end offset equals k has ended before entry k is consumed.
__host__ __device__ __forceinline__ int64_t merge_path_cols(const int32_t* __restrict__ p, int64_t ncol, int64_t nnz,
                                                            int64_t d) {
  int64_t lo = d > nnz ? d - nnz : 0;
  int64_t hi = d < ncol ? d : ncol;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (static_cast<int64_t>(p[mid + 1]) <= d - mid - 1)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

__global__ void sweep_plan_kernel(const int32_t* __restrict__ p, int64_t ncol, int64_t nnz, int64_t n_tiles,
                                  int tile, int32_t* __restrict__ plan) {
  const int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t > n_tiles) return;
  const int64_t total = ncol + nnz;
  int64_t d = t * tile;
  if (d > total) d = total;
  plan[t] = static_cast<int32_t>(merge_path_cols(p, ncol, nnz, d));
}

struct SweepParams {
  const int32_t* i;
  const int32_t* p;
  const double* x;
  const int32_t* plan;
  int64_t n_tiles;
  int32_t ncol;
  int32_t nnz;
  const double* v;
  double* out;
  int32_t* carry_col;  // [grid]
  double* carry_val;   // [grid]
  unsigned int* ticket;
  int mask;  // SPMV_T only: v is an indicator — entries whose v[row] is 0 are SKIPPED (x * 0 would turn Inf into NaN)
  double var_n;  // COLVAR only (v = the column means): the column length n of var_from_sums; 0 = store the raw sums
};

struct StageMeta {
  int32_t c0;     // first column of the tile (the one in progress at its start)
  int32_t nc;     // column ends inside the tile
  int32_t k0;     // first entry of the tile
  int32_t nk;     // entries inside the tile
  int32_t a_off;  // where p[c0+1] sits in the staged window
  int32_t x_off;  // where x[k0] sits
  int32_t i_off;  // where i[k0] sits
  int32_t pad;
};

template <int IPT_>
struct SweepGeom {
  static constexpr int TILE = SWEEP_THREADS * IPT_;
  static constexpr int X_ELEMS = TILE + 2;   // +1 align-down slack, +1 round-up
  static constexpr int A_ELEMS = TILE + 8;   // nc+1 values, +3 align-down, +3 round-up, +1 spare
  static constexpr int I_ELEMS = TILE + 8;
  static constexpr size_t X_BYTES = ((X_ELEMS * 8 + 15) / 16) * 16;
  static constexpr size_t A_BYTES = ((A_ELEMS * 4 + 15) / 16) * 16;
  static constexpr size_t I_BYTES = ((I_ELEMS * 4 + 15) / 16) * 16;
  static constexpr size_t stage_bytes(bool with_i) { return X_BYTES + A_BYTES + (with_i ? I_BYTES : 0); }
};

constexpr int SWEEP_BLOCK = SWEEP_THREADS + 32;  // 8 consumer warps + 1 producer warp

// tiles with this many column ends are summed a column per lane group (sweep_kernel)
constexpr int SEG_LANES = 8;
constexpr int SEG_MIN_ENDS = 2;
constexpr int SEG_MAX_ENDS = 512;

// consumer-only barrier (the producer warp never joins it)
__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, %0;" ::"n"(SWEEP_THREADS) : "memory"); }

template <int MODE, int STAGES>
__global__ void __launch_bounds__(SWEEP_BLOCK) sweep_kernel(const SweepParams prm) {
  constexpr bool VAR = (MODE == SWEEP_COLVAR);
  constexpr int IPT = (MODE == SWEEP_COLSUM || VAR) ? SWEEP_IPT : GATHER_IPT;
  using G = SweepGeom<IPT>;
  constexpr int THREADS = SWEEP_THREADS;
  constexpr int TILE = G::TILE;
  constexpr bool WITH_I = (MODE == SWEEP_SPMV_T || MODE == SWEEP_SPMV);
  constexpr bool REDUCES = (MODE == SWEEP_COLSUM || MODE == SWEEP_SPMV_T || VAR);
  constexpr int WARPS = THREADS / 32;
  static_assert(WARPS <= 32, "warp fold uses one lane per warp");

  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ uint64_t full_bar[STAGES];   // producer -> consumers: the stage's bytes have landed
  __shared__ uint64_t empty_bar[STAGES];  // consumers -> producer: every consumer warp is done with the stage
  __shared__ StageMeta meta[STAGES];
  __shared__ double warp_sum[2][WARPS];   // double-buffered by tile parity: one barrier per tile
  __shared__ int warp_flag[2][WARPS];
  __shared__ double seg_carry[2];         // segment-parallel tiles: sum of the column left open by the tile
  __shared__ int cta_info[4];

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;

  // contiguous tile range of this CTA
  const int64_t t_begin = (prm.n_tiles * blockIdx.x) / gridDim.x;
  const int64_t t_end = (prm.n_tiles * (blockIdx.x + 1)) / gridDim.x;
  const int n_local = static_cast<int>(t_end - t_begin);
  const int64_t total_items = static_cast<int64_t>(prm.ncol) + prm.nnz;

  auto stage_x = [&](int s) { return reinterpret_cast<double*>(smem_raw + s * G::stage_bytes(WITH_I)); };
  auto stage_a = [&](int s) {
    return reinterpret_cast<int32_t*>(smem_raw + s * G::stage_bytes(WITH_I) + G::X_BYTES);
  };
  auto stage_i = [&](int s) {
    return reinterpret_cast<int32_t*>(smem_raw + s * G::stage_bytes(WITH_I) + G::X_BYTES + G::A_BYTES);
  };

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], WARPS);
    }
    ptx::fence_mbar_init();
  }
  __syncthreads();

  if (warp == WARPS) {
    // =========================== producer warp: one lane drives the TMA ring ===========================
    if (lane == 0 && n_local > 0) {
      int32_t pl_lo = __ldg(prm.plan + t_begin);      // plan[t], plan[t + 1] of the tile being issued
      int32_t pl_hi = __ldg(prm.plan + t_begin + 1);
      for (int j = 0; j < n_local; ++j) {
        const int s = j % STAGES;
        const int64_t t = t_begin + j;
        // fetch the next plan entry before (possibly) blocking on the stage
        int32_t pl_next = 0;
        if (j + 1 < n_local) pl_next = __ldg(prm.plan + t + 2);
        if (j >= STAGES) ptx::mbar_wait(&empty_bar[s], static_cast<uint32_t>(j / STAGES - 1) & 1u);
        const int64_t d0 = t * TILE;
        int64_t d1 = d0 + TILE;
        if (d1 > total_items) d1 = total_items;
        const int32_t c0 = pl_lo, c1 = pl_hi;
        const int32_t k0 = static_cast<int32_t>(d0 - c0), k1 = static_cast<int32_t>(d1 - c1);
        StageMeta mt;
        mt.c0 = c0;
        mt.nc = c1 - c0;
        mt.k0 = k0;
        mt.nk = k1 - k0;
        // column-end window: p[c0+1 .. min(c1+1, ncol)]
        const int32_t a_first = c0 + 1;
        const int32_t a_last = (c1 + 1 <= prm.ncol) ? c1 + 1 : prm.ncol;
        const int32_t a_al = a_first & ~3;
        const int32_t a_cnt = (a_last >= a_first) ? (((a_last - a_al + 1) + 3) & ~3) : 0;
        mt.a_off = a_first - a_al;
        const int32_t x_al = k0 & ~1;
        const int32_t x_cnt = (mt.nk > 0) ? (((k1 - x_al) + 1) & ~1) : 0;
        mt.x_off = k0 - x_al;
        const int32_t i_al = k0 & ~3;
        const int32_t i_cnt = (WITH_I && mt.nk > 0) ? (((k1 - i_al) + 3) & ~3) : 0;
        mt.i_off = k0 - i_al;
        mt.pad = 0;
        meta[s] = mt;
        const uint32_t bytes = static_cast<uint32_t>(a_cnt) * 4u + static_cast<uint32_t>(x_cnt) * 8u +
                               static_cast<uint32_t>(i_cnt) * 4u;
        ptx::mbar_arrive_expect_tx(&full_bar[s], bytes);
        if (a_cnt > 0) ptx::bulk_g2s(stage_a(s), prm.p + a_al, static_cast<uint32_t>(a_cnt) * 4u, &full_bar[s]);
        if (x_cnt > 0) ptx::bulk_g2s(stage_x(s), prm.x + x_al, static_cast<uint32_t>(x_cnt) * 8u, &full_bar[s]);
        if (i_cnt > 0) ptx::bulk_g2s(stage_i(s), prm.i + i_al, static_cast<uint32_t>(i_cnt) * 4u, &full_bar[s]);
        pl_lo = pl_hi;
        pl_hi = pl_next;
      }
    }
    return;
  }

  // ======================================= consumer warps ================================================
  double cta_carry = 0.0;  // partial sum of the column in progress, carried across this CTA's tiles
  int32_t last_c1 = 0, last_k1 = 0;

  // COLVAR: every item adds (x - m)^2 with m = its column's mean, and a column's store applies var_from_sums.  The one
  // exception is the column earlier CTAs carry into (it began before this CTA's first item): its store here is only
  // this CTA's share, and the last CTA applies the formula when it folds the carries in.  Every other mode compiles
  // these helpers down to the plain sum and store.
  int32_t in_col = -1;
  if constexpr (VAR) {
    if (n_local > 0) {
      const int32_t c = __ldg(prm.plan + t_begin);
      if (c < prm.ncol && t_begin * TILE - c > __ldg(prm.p + c)) in_col = c;
    }
  }
  auto mean_of = [&](int64_t c) -> double {
    if constexpr (VAR)
      return c < prm.ncol ? __ldg(prm.v + c) : 0.0;
    else
      return 0.0;
  };
  auto term = [&](double xv, double mu) -> double {
    if constexpr (VAR) {
      const double d = __dsub_rn(xv, mu);
      return __dmul_rn(d, d);
    } else {
      return xv;
    }
  };
  auto finish = [&](int32_t c, double s) -> double {
    if constexpr (VAR) {
      if (prm.var_n == 0.0) return s;
      return var_from_sums(s, static_cast<double>(__ldg(prm.p + c + 1) - __ldg(prm.p + c)), __ldg(prm.v + c), prm.var_n);
    } else {
      return s;
    }
  };
  auto store_col = [&](int32_t c, double s) {
    if constexpr (VAR)
      prm.out[c] = (c == in_col) ? s : finish(c, s);
    else
      prm.out[c] = s;
  };

  for (int j = 0; j < n_local; ++j) {
    const int s = j % STAGES;
    const int buf = j & 1;
    const uint32_t parity = static_cast<uint32_t>(j / STAGES) & 1u;
    ptx::mbar_wait(&full_bar[s], parity);
    const StageMeta mt = meta[s];
    const double* __restrict__ xs = stage_x(s) + mt.x_off;
    const int32_t* __restrict__ as = stage_a(s) + mt.a_off;
    const int32_t* __restrict__ is = stage_i(s) + mt.i_off;
    const int items = mt.nc + mt.nk;
    last_c1 = mt.c0 + mt.nc;
    last_k1 = mt.k0 + mt.nk;

    if (MODE == SWEEP_SPMV_T) {
      // pre-multiply the staged values by the gathered operand, striped (IPT independent
      // L2 gathers in flight per thread); the walk below then is the plain column sum.
      double* xw = stage_x(s) + mt.x_off;
      double g[IPT];
#pragma unroll
      for (int r = 0; r < IPT; ++r) {
        const int k = tid + r * THREADS;
        g[r] = (k < mt.nk) ? __ldg(prm.v + is[k]) : 0.0;
      }
#pragma unroll
      for (int r = 0; r < IPT; ++r) {
        const int k = tid + r * THREADS;
        if (k < mt.nk) xw[k] = prm.mask ? (g[r] != 0.0 ? xw[k] : 0.0) : __dmul_rn(xw[k], g[r]);
      }
      consumer_sync();
    }

    // ---- tiles in which many columns end: a group of SEG_LANES lanes per column ----------------------
    // (short columns, and the row-ordered copy of a wide matrix).  The tile holds nc + 1 segments of the
    // entry stream: columns c0 .. c0+nc-1 end here, the last segment stays open.  Each group strides over
    // one segment, folds with shuffles and stores — ~2 instructions per entry at 100 entries per column,
    // where the per-thread walk below spends ~40 on searches, branches and the segmented scan.
    // (A^T v is bound by its gathers; with few, long columns the walk's all-thread sum is the shorter tail)
    constexpr int SEG_MIN = (MODE == SWEEP_SPMV_T) ? WARPS : SEG_MIN_ENDS;
    const bool seg_tile = REDUCES && mt.nc >= SEG_MIN && mt.nc <= SEG_MAX_ENDS;
    if (seg_tile) {
      auto sum_segments = [&](auto lanes_c) {
        constexpr int L = decltype(lanes_c)::value;
        constexpr int GROUPS = THREADS / L;
        const int gidx = tid / L, gl = tid % L;
        const int nseg = mt.nc + 1;
        for (int base = 0; base < nseg; base += GROUPS) {  // trip count uniform over the CTA
          const int c = base + gidx;
          double sacc = 0.0;
          if (c < nseg) {
            const int beg = (c == 0) ? 0 : as[c - 1] - mt.k0;
            const int end = (c == mt.nc) ? mt.nk : as[c] - mt.k0;
            const double mu = mean_of(mt.c0 + c);
            double a0 = 0.0, a1 = 0.0;
            int k = beg + gl;
            for (; k + L < end; k += 2 * L) {
              a0 = __dadd_rn(a0, term(xs[k], mu));
              a1 = __dadd_rn(a1, term(xs[k + L], mu));
            }
            if (k < end) a0 = __dadd_rn(a0, term(xs[k], mu));
            sacc = __dadd_rn(a0, a1);
          }
#pragma unroll
          for (int off = L / 2; off > 0; off >>= 1) sacc = __dadd_rn(sacc, __shfl_xor_sync(0xffffffffu, sacc, off));
          if (gl == 0 && c < nseg) {
            if (c < mt.nc)
              store_col(mt.c0 + c, (c == 0) ? __dadd_rn(cta_carry, sacc) : sacc);  // earlier CTAs' shares: fix-up below
            else
              seg_carry[buf] = sacc;
          }
        }
      };
      if (mt.nc < WARPS)
        sum_segments(std::integral_constant<int, 32>{});  // a warp per column: at most one round
      else
        sum_segments(std::integral_constant<int, SEG_LANES>{});
      if (MODE == SWEEP_SPMV_T) ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&empty_bar[s]);
      consumer_sync();
      cta_carry = seg_carry[buf];
      continue;
    }

    // ---- per-thread merge-path walk ------------------------------------------------------------
    int d_lo = tid * IPT;
    if (d_lo > items) d_lo = items;
    int d_hi = d_lo + IPT;
    if (d_hi > items) d_hi = items;
    const int n_my = d_hi - d_lo;
    int lo = d_lo > mt.nk ? d_lo - mt.nk : 0;
    int hi = d_lo < mt.nc ? d_lo : mt.nc;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (as[mid] - mt.k0 <= d_lo - mid - 1)
        lo = mid + 1;
      else
        hi = mid;
    }
    int ci = lo;         // column ends consumed before my first item
    int ki = d_lo - ci;  // entries consumed before my first item
    int col_end = as[ci] - mt.k0;  // stale past the last column, but then no items remain
    double acc = 0.0, head = 0.0;
    int first_ci = -1;

    if (MODE == SWEEP_SPMV) {
      double vc = (mt.c0 + ci < prm.ncol) ? __ldg(prm.v + mt.c0 + ci) : 0.0;
#pragma unroll
      for (int it = 0; it < IPT; ++it) {
        if (it < n_my) {
          if (ki < col_end) {
            ptx::red_add_f64(prm.out + is[ki], __dmul_rn(xs[ki], vc));
            ++ki;
          } else {
            ++ci;
            col_end = as[ci] - mt.k0;
            vc = (mt.c0 + ci < prm.ncol) ? __ldg(prm.v + mt.c0 + ci) : 0.0;
          }
        }
      }
    } else if (n_my == IPT && ki + IPT <= col_end) {
      // common case (columns much longer than IPT): all my items are entries of one column
      const double mu = mean_of(mt.c0 + ci);
      double a0 = 0.0, a1 = 0.0;
#pragma unroll
      for (int it = 0; it + 1 < IPT; it += 2) {
        a0 = __dadd_rn(a0, term(xs[ki + it], mu));
        a1 = __dadd_rn(a1, term(xs[ki + it + 1], mu));
      }
      if (IPT & 1) a0 = __dadd_rn(a0, term(xs[ki + IPT - 1], mu));
      acc = __dadd_rn(a0, a1);
    } else {
      // a column ends among my items (short columns; the row-ordered copy of a wide matrix): straight-line
      // adds, the rare end handled in place — the rest of the warp waits for this path, so it is unrolled
      double mu = mean_of(mt.c0 + ci);
#pragma unroll
      for (int it = 0; it < IPT; ++it) {
        if (it < n_my) {
          if (ki < col_end) {
            acc = __dadd_rn(acc, term(xs[ki], mu));
            ++ki;
          } else {
            if (first_ci < 0) {
              first_ci = ci;
              head = acc;
            } else {
              store_col(mt.c0 + ci, acc);  // began and ended inside this thread
            }
            acc = 0.0;
            ++ci;
            col_end = as[ci] - mt.k0;
            mu = mean_of(mt.c0 + ci);
          }
        }
      }
    }

    // this warp no longer reads stage s: hand it back to the producer
    if (MODE == SWEEP_SPMV_T) ptx::fence_proxy_async_smem();  // my generic writes precede the async refill
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(&empty_bar[s]);

    if (REDUCES) {
      // ---- stitch partial sums across threads.  Segment heads are threads in which at least one
      //      column ended (their tail starts a new column).  A warp without any column end only
      //      needs its total; otherwise a segmented inclusive scan over the lanes. ----
      const int fl_mine = first_ci >= 0 ? 1 : 0;
      const unsigned ends_in_warp = __ballot_sync(0xffffffffu, fl_mine);
      double sc = acc;
      int fl = fl_mine;
      double prev_sc = 0.0;
      int prev_fl = 0;
      if (ends_in_warp == 0u) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) sc = __dadd_rn(sc, __shfl_xor_sync(0xffffffffu, sc, off));
        if (lane == 31) {
          warp_sum[buf][warp] = sc;
          warp_flag[buf][warp] = 0;
        }
      } else {
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
          const double up = __shfl_up_sync(0xffffffffu, sc, off);
          const int fu = __shfl_up_sync(0xffffffffu, fl, off);
          if (lane >= off) {
            if (!fl) sc = __dadd_rn(up, sc);
            fl |= fu;
          }
        }
        if (lane == 31) {
          warp_sum[buf][warp] = sc;
          warp_flag[buf][warp] = fl;
        }
        prev_sc = __shfl_up_sync(0xffffffffu, sc, 1);
        prev_fl = __shfl_up_sync(0xffffffffu, fl, 1);
      }
      consumer_sync();
      // fold the warp totals with one lane per warp (every warp does it redundantly: no extra barrier)
      double ws = (lane < WARPS) ? warp_sum[buf][lane] : 0.0;
      int wf = (lane < WARPS) ? warp_flag[buf][lane] : 0;
      if (lane == 0 && !wf) ws = __dadd_rn(cta_carry, ws);
#pragma unroll
      for (int off = 1; off < WARPS; off <<= 1) {
        const double up = __shfl_up_sync(0xffffffffu, ws, off);
        const int fu = __shfl_up_sync(0xffffffffu, wf, off);
        if (lane >= off) {
          if (!wf) ws = __dadd_rn(up, ws);
          wf |= fu;
        }
      }
      const int src = warp > 0 ? warp - 1 : 0;
      double pre = __shfl_sync(0xffffffffu, ws, src);
      if (warp == 0) pre = cta_carry;
      const double all = __shfl_sync(0xffffffffu, ws, WARPS - 1);
      if (first_ci >= 0) {
        double carry_in;
        if (lane == 0)
          carry_in = pre;
        else
          carry_in = prev_fl ? prev_sc : __dadd_rn(pre, prev_sc);
        // partial sums carried in by EARLIER CTAs (a column spanning CTA boundaries) are added
        // afterwards, in CTA order, by the last CTA to finish
        store_col(mt.c0 + first_ci, __dadd_rn(carry_in, head));
      }
      cta_carry = all;
    }
  }

  if (REDUCES) {
    // ---- publish this CTA's carry, last CTA folds all carries in CTA order ------------------------
    if (tid == 0) {
      int32_t col = -1;
      if (n_local > 0 && last_c1 < prm.ncol && last_k1 > __ldg(prm.p + last_c1)) col = last_c1;
      prm.carry_col[blockIdx.x] = col;
      prm.carry_val[blockIdx.x] = cta_carry;
    }
    __threadfence();  // every consumer's stores to out[] are visible before the ticket is taken
    consumer_sync();
    if (tid == 0) {
      __threadfence();
      const unsigned int t = atomicAdd(prm.ticket, 1u);
      cta_info[1] = (t == gridDim.x - 1) ? 1 : 0;
    }
    consumer_sync();
    if (cta_info[1]) {
      __threadfence();
      const int G_ = gridDim.x;
      for (int g = tid; g < G_; g += THREADS) {
        const int32_t col = __ldcg(prm.carry_col + g);
        if (col < 0) continue;
        if (g > 0 && __ldcg(prm.carry_col + g - 1) == col) continue;  // not the first CTA carrying into col
        double tot = 0.0;
        for (int h = g; h < G_ && __ldcg(prm.carry_col + h) == col; ++h) tot = __dadd_rn(tot, __ldcg(prm.carry_val + h));
        // the CTA in which `col` ends stored only its own share (its cta_carry started from 0)
        prm.out[col] = finish(col, __dadd_rn(tot, __ldcg(prm.out + col)));
      }
      if (tid == 0) *prm.ticket = 0u;  // ready for the next launch
    }
  }
}

// rowSums: no column bookkeeping at all — stream i and x with 128-bit loads and fire FP64
// reductions at L2 (REDG.E.ADD.F64).  The m-length result lives in L2 (8 MB at m = 1M).
template <int THREADS, int UNROLL>
__global__ void __launch_bounds__(THREADS) rowsum_stream_kernel(const int32_t* __restrict__ gi,
                                                                 const double* __restrict__ gx, int64_t nnz,
                                                                 double* __restrict__ out) {
  const int64_t n4 = nnz >> 2;  // groups of four entries
  const int64_t stride = static_cast<int64_t>(gridDim.x) * THREADS;
  const int4* __restrict__ i4 = reinterpret_cast<const int4*>(gi);
  const double2* __restrict__ x2 = reinterpret_cast<const double2*>(gx);
  int64_t g = static_cast<int64_t>(blockIdx.x) * THREADS + threadIdx.x;
  for (; g + (UNROLL - 1) * stride < n4; g += UNROLL * stride) {
    int4 r[UNROLL];
    double2 a[UNROLL], b[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      r[u] = ptx::ld_stream_v4s32(i4 + g + u * stride);
      a[u] = ptx::ld_stream_v2f64(x2 + 2 * (g + u * stride));
      b[u] = ptx::ld_stream_v2f64(x2 + 2 * (g + u * stride) + 1);
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      ptx::red_add_f64(out + r[u].x, a[u].x);
      ptx::red_add_f64(out + r[u].y, a[u].y);
      ptx::red_add_f64(out + r[u].z, b[u].x);
      ptx::red_add_f64(out + r[u].w, b[u].y);
    }
  }
  for (; g < n4; g += stride) {
    const int4 r = ptx::ld_stream_v4s32(i4 + g);
    const double2 a = ptx::ld_stream_v2f64(x2 + 2 * g);
    const double2 b = ptx::ld_stream_v2f64(x2 + 2 * g + 1);
    ptx::red_add_f64(out + r.x, a.x);
    ptx::red_add_f64(out + r.y, a.y);
    ptx::red_add_f64(out + r.z, b.x);
    ptx::red_add_f64(out + r.w, b.y);
  }
  // tail (nnz % 4 entries)
  const int64_t k = (n4 << 2) + static_cast<int64_t>(blockIdx.x) * THREADS + threadIdx.x;
  if (k < nnz) ptx::red_add_f64(out + gi[k], gx[k]);
}

__global__ void vec_div_kernel(double* __restrict__ d, int64_t n, double divisor) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; k < n; k += stride) d[k] = d[k] / divisor;
}

__global__ void fill_zero_kernel(double* __restrict__ d, int64_t n) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; k < n; k += stride) d[k] = 0.0;
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct SweepConfig {
  int threads;  // 256 or 512
  int stages;   // 2..4
  int ctas_per_sm;
};

static SweepConfig sweep_config(SweepMode mode) {
  // defaults chosen to keep >= 100 KB of bulk copies in flight per SM; SB200_SWEEP_CFG=threads,stages,ctas
  // overrides (tuning runs only).
  SweepConfig c;
  c.threads = SWEEP_THREADS;
  c.stages = 2;       // measured best for every mode: two stages per CTA ...
  c.ctas_per_sm = 3;  // ... and three CTAs per SM (24 consumer warps) rather than deeper rings
  (void)mode;
  if (const char* e = getenv("SB200_SWEEP_CFG")) {
    int t = 0, s = 0, k = 0;
    if (sscanf(e, "%d,%d,%d", &t, &s, &k) == 3 && t == SWEEP_THREADS && s >= 2 && s <= 4 && k >= 1 && k <= 8) {
      c.stages = s;
      c.ctas_per_sm = k;
    }
  }
  return c;
}

template <int MODE>
using GeomOf = SweepGeom<(MODE == SWEEP_COLSUM || MODE == SWEEP_COLVAR) ? SWEEP_IPT : GATHER_IPT>;

template <int MODE, int STAGES>
static int launch_sweep_t(sb200_matrix* m, const SweepParams& prm, int ctas_per_sm) {
  using G = GeomOf<MODE>;
  constexpr bool WITH_I = (MODE == SWEEP_SPMV_T || MODE == SWEEP_SPMV);
  const size_t smem = STAGES * G::stage_bytes(WITH_I);
  auto kern = sweep_kernel<MODE, STAGES>;
  SB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  int64_t grid = static_cast<int64_t>(m->sm_count) * ctas_per_sm;
  if (grid > prm.n_tiles) grid = prm.n_tiles;
  if (grid > 1024) grid = 1024;  // capacity of the cross-CTA carry arrays in the workspace
  if (grid < 1) return SB200_OK;
  kern<<<static_cast<unsigned>(grid), SWEEP_BLOCK, smem, m->stream>>>(prm);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return SB200_OK;
}

template <int MODE>
static int launch_sweep_m(sb200_matrix* m, const SweepParams& prm, const SweepConfig& cfg) {
  using G = GeomOf<MODE>;
  constexpr bool WITH_I = (MODE == SWEEP_SPMV_T || MODE == SWEEP_SPMV);
  int stages = cfg.stages, ctas = cfg.ctas_per_sm;
  while (ctas > 1 && static_cast<size_t>(stages) * G::stage_bytes(WITH_I) * ctas > 220 * 1024) --ctas;
  while (stages > 2 && static_cast<size_t>(stages) * G::stage_bytes(WITH_I) * ctas > 220 * 1024) --stages;
  switch (stages) {
    case 2: return launch_sweep_t<MODE, 2>(m, prm, ctas);
    case 3: return launch_sweep_t<MODE, 3>(m, prm, ctas);
    default: return launch_sweep_t<MODE, 4>(m, prm, ctas);
  }
}

static int build_one_plan(sb200_matrix* m, int tile, int32_t** d_plan, int64_t* n_tiles) {
  const int64_t total = static_cast<int64_t>(m->ncol) + m->nnz;
  *n_tiles = (total + tile - 1) / tile;
  SB_TRY(pool_alloc(reinterpret_cast<void**>(d_plan), sizeof(int32_t) * static_cast<size_t>(*n_tiles + 2), m->stream));
  const int threads = 256;
  const int64_t blocks = (*n_tiles + 1 + threads - 1) / threads;
  sweep_plan_kernel<<<static_cast<unsigned>(blocks), threads, 0, m->stream>>>(m->d_p, m->ncol, m->nnz, *n_tiles, tile,
                                                                            *d_plan);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return SB200_OK;
}

int build_sweep_plan(sb200_matrix* m) {
  SB_TRY(build_one_plan(m, SWEEP_TILE, &m->d_plan, &m->n_tiles));
  SB_TRY(build_one_plan(m, GATHER_TILE, &m->d_plan_g, &m->n_tiles_g));
  return SB200_OK;
}

int launch_vec_div(cudaStream_t s, double* d, int64_t n, double divisor) {
  if (n <= 0) return SB200_OK;
  int64_t blocks = (n + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  vec_div_kernel<<<static_cast<unsigned>(blocks), 256, 0, s>>>(d, n, divisor);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return SB200_OK;
}

static int launch_tile_sweep(sb200_matrix* m, SweepMode mode, const double* d_v, double* d_out, int mask, double var_n = 0.0) {
  if (m->n_tiles == 0) return SB200_OK;  // ncol == 0 and nnz == 0: nothing to produce
  const bool cols = (mode == SWEEP_COLSUM || mode == SWEEP_COLVAR);  // the column-sum geometry and plan
  SweepParams prm;
  prm.i = m->d_i;
  prm.p = m->d_p;
  prm.x = m->d_x;
  prm.plan = cols ? m->d_plan : m->d_plan_g;
  prm.n_tiles = cols ? m->n_tiles : m->n_tiles_g;
  prm.ncol = m->ncol;
  prm.nnz = static_cast<int32_t>(m->nnz);
  prm.v = d_v;
  prm.out = d_out;
  prm.mask = mask;
  prm.var_n = var_n;
  // workspace layout: [ticket u32 | pad to 16] [carry_col int32 x 1024] [carry_val f64 x 1024]
  unsigned char* ws = static_cast<unsigned char*>(m->d_ws);
  prm.ticket = reinterpret_cast<unsigned int*>(ws);
  prm.carry_col = reinterpret_cast<int32_t*>(ws + 16);
  prm.carry_val = reinterpret_cast<double*>(ws + 16 + 4 * 1024);
  const SweepConfig cfg = sweep_config(mode);
  switch (mode) {
    case SWEEP_COLSUM: return launch_sweep_m<SWEEP_COLSUM>(m, prm, cfg);
    case SWEEP_SPMV_T: return launch_sweep_m<SWEEP_SPMV_T>(m, prm, cfg);
    case SWEEP_SPMV: return launch_sweep_m<SWEEP_SPMV>(m, prm, cfg);
    case SWEEP_COLVAR: return launch_sweep_m<SWEEP_COLVAR>(m, prm, cfg);
    default: return fail(SB200_E_INVALID, "unknown sweep mode");
  }
}

int launch_sweep(sb200_matrix* m, SweepMode mode, const double* d_v, double divisor, double* d_out) {
  if (mode == SWEEP_COLVAR) return launch_col_vars(m, d_out);  // two passes (vars.cu)
  if (mode == SWEEP_ROWVAR) return launch_row_vars(m, d_out);
  if ((mode == SWEEP_ROWSUM || mode == SWEEP_SPMV) && m->nnz > 0 && m->nrow > 0) {
    // A mirror whose row-indexed sweeps keep being asked for gets a row-major copy of itself: from then on a
    // row sum is the same streaming segmented sweep as a column sum (8 B per entry, no atomics) and A v is the
    // gather sweep of the copy (A v = (A^T)^T v) instead of a scatter.  Same arithmetic every call — only the
    // layout is kept, like the band plan.
    if (m->rows_state == 0 && m->owns_arrays) {
      const int after = row_companion_after();
      if (after > 0 && ++m->row_sum_calls > after) build_row_companion(m);
    }
    if (m->rows_state == 1) {
      m->rows->stream = m->stream;
      if (mode == SWEEP_ROWSUM) return launch_sweep(m->rows, SWEEP_COLSUM, nullptr, divisor, d_out);
      return launch_sweep(m->rows, SWEEP_SPMV_T, d_v, 0.0, d_out);
    }
  }
  if (mode == SWEEP_SPMV_T && m->nnz > 0 && m->nrow > 0 && m->ncol > 0) {
    // A mirror that keeps being asked for A^T v gets a band-major companion (bmc.cu): the operand's slice of a row
    // band sits in shared memory while the band's entries stream past, instead of one L2 gather per entry.
    if (m->bmc_state == 0 && m->owns_arrays) {
      const int after = row_companion_after();
      if (after > 0 && ++m->spmv_t_calls > after) build_band_companion(m);
    }
    if (m->bmc_state == 1) return launch_bandsweep(m, d_v, d_out);
  }
  if (mode == SWEEP_SPMV_T && m->nnz > 0) {
    SB_TRY(decide_gather_path(m));
    if (m->gather_path == 1) {
      const int rc = launch_band_gather(m, d_v, d_out);
      if (rc == SB200_OK) return SB200_OK;
      if (rc != SB200_E_UNSUPPORTED && rc != SB200_E_NOMEM) return rc;
      cudaGetLastError();  // no plan for this shape: the L2-gather sweep serves every shape
      m->gather_path = 0;
    }
  }
  if (mode == SWEEP_ROWSUM || mode == SWEEP_SPMV) SB_TRY(decide_row_path(m));
  if ((mode == SWEEP_ROWSUM || mode == SWEEP_SPMV) && m->row_path == 1) {
    const int rc = launch_band_scatter(m, mode == SWEEP_SPMV ? d_v : nullptr, d_out);
    if (rc == SB200_OK) {
      if (mode == SWEEP_ROWSUM && divisor != 0.0) SB_TRY(launch_vec_div(m->stream, d_out, m->nrow, divisor));
      return SB200_OK;
    }
    // the band plan could not be built for this shape (memory, row budget): not an error for the caller —
    // the plan-free L2-atomic kernels below serve every shape.  A CUDA failure is still a failure.
    if (rc != SB200_E_UNSUPPORTED && rc != SB200_E_NOMEM) return rc;
    cudaGetLastError();
    m->row_path = 0;
  }
  if (mode == SWEEP_ROWSUM || mode == SWEEP_SPMV) {
    // scatter targets start from zero (the reference's zero-initialised NumericVector, RcppSparse.h:139)
    if (m->nrow > 0) SB_CUDA(cudaMemsetAsync(d_out, 0, sizeof(double) * static_cast<size_t>(m->nrow), m->stream));
  }
  if (mode == SWEEP_ROWSUM) {
    if (m->nnz > 0) {
      constexpr int T = 256, U = 4;
      int64_t blocks = ((m->nnz >> 2) + static_cast<int64_t>(T) * U - 1) / (static_cast<int64_t>(T) * U);
      const int64_t cap = static_cast<int64_t>(m->sm_count) * 8;
      if (blocks > cap) blocks = cap;
      if (blocks < 1) blocks = 1;
      rowsum_stream_kernel<T, U><<<static_cast<unsigned>(blocks), T, 0, m->stream>>>(m->d_i, m->d_x, m->nnz, d_out);
      count_launch();
      SB_CUDA(cudaGetLastError());
    }
    if (divisor != 0.0) SB_TRY(launch_vec_div(m->stream, d_out, m->nrow, divisor));
    return SB200_OK;
  }
  SB_TRY(launch_tile_sweep(m, mode, d_v, d_out, 0));
  // colMeans: sums[c] / Dim[0] as a second pass over the ncol outputs, exactly the reference's
  // structure (RcppSparse.h:146-148); 16 B per column next to 8 B per stored entry.
  if (mode == SWEEP_COLSUM && divisor != 0.0) SB_TRY(launch_vec_div(m->stream, d_out, m->ncol, divisor));
  return SB200_OK;
}

// Masked column sums (N4): out[c] = sum of the entries of column c whose row has d_mask[row] != 0 — the sweep a user
// writes with InnerIteratorInRange / InnerIteratorNotInRange (reference RcppSparse.h:238-321), all columns at once.
// Always the tile sweep on the CSC arrays: skipping an entry is not the same as multiplying it by 0.0.
int launch_masked_col_sums(sb200_matrix* m, const double* d_mask, double* d_out) { return launch_tile_sweep(m, SWEEP_SPMV_T, d_mask, d_out, 1); }

// Second pass of colVars: d_out[c] = var_from_sums(sum over column c's entries of (x - d_mean[c])^2, its entry count,
// d_mean[c], n), or the sum itself when n = 0.  Same tiles, walk and carry fold as the column sums.
int launch_col_var_sweep(sb200_matrix* m, const double* d_mean, double n, double* d_out) {
  return launch_tile_sweep(m, SWEEP_COLVAR, d_mean, d_out, 0, n);
}

}  // namespace sb200
