// Row-banded kernels: the CSC -> CSR transpose and the row-indexed sweeps (rowSums, rowMeans, A v).
//
// Replaces, from the reference (zdebruine/RcppSparse):
//   Matrix::transpose()   RcppSparse.h:375-385 (arithmetic = R's Matrix::t, a serial counting sort)
//   Matrix::rowSums()     RcppSparse.h:138-144   sums(i[j]) += x[j]
//   Matrix::rowMeans()    RcppSparse.h:151-156
//   A v (iterator idiom)  y[it.row()] += it.value() * v[col]   (shape of :140-142)
//
// Why bands.  A row-indexed result of 1e6 doubles does not fit shared memory, and one L2 atomic
// per stored entry tops out at ~160 G RED.F64/s on B200 (profiles/r01/microbench: 31% of the
// rowSums roofline).  But rows are SORTED inside every column, so the entries of a column that fall
// in a row band [rb[b], rb[b+1]) are one contiguous run.  A band plan (built once per matrix
// structure, cached in the handle) stores for each band b and column c where that run starts
// ("band pointers").  CTA (b, h) then owns band b for column split h: it streams only its runs,
// keeps the band's rows in shared memory — accumulators for the sums, append cursors for the
// transpose — and nobody else ever touches those rows.  Neighbouring bands read neighbouring runs of
// the same columns at about the same time, so partially used 32-byte sectors are served from L2.
//
// Plan (one pass each, HBM-bound):
//   P1  histogram of row indices per column split (stream i, 4 B/nnz; counts privatised in shared
//       memory when u32[nrow*S] fits) -> exclusive scan (scan.cu) -> p' and per-split offsets
//   P2  band boundaries: nb bands of ~equal nnz, bounded in rows (binary searches in p')
//   P3  band pointers over the merge-path tiles of the sweeps (stream i again, 4 B/nnz)
//
// Inner skeleton (both kernels): a warp takes 32 consecutive columns of a chunk, one run descriptor
// per lane, flattens the runs with a shuffle scan, and walks the concatenated entries 32 at a time,
// so consecutive lanes read consecutive entries of a run (coalesced).
//   * sums:      acc[row - rb[b]] += x (* v[col])  shared-memory FP64 atomic; at the end the band's
//                accumulators are added to the result with coalesced REDs (plain stores when S = 1)
//   * transpose: pass 1 counts entries per (warp, row); a per-row scan over the 16 warps gives every
//                warp its private, ordered slot range; pass 2 re-walks the entries, ranks equal rows
//                inside a 32-entry step with match.any in lane order (= source column order) and
//                stores column id and value.  Order inside an output row is source-column order by
//                construction => bit-exact canonical CSC of A^T, no sort, no global atomics.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <new>

#include "common.cuh"
#include "ptx.cuh"
#include "walk.cuh"
#include "bandplan.cuh"

namespace sb200 {

namespace {

// ================================================================================================
// P1: per-split row histogram
// ================================================================================================
constexpr int HIST_THREADS = 512;
constexpr int HIST_SMEM_MAX_WORDS = 48 * 1024;  // u32 counters, 192 KB

// cnt[r * S + h] += number of entries with row r in column split h.  CTA (h, g): slice g of split h.
template <bool PRIVATE>
__global__ void __launch_bounds__(HIST_THREADS)
    row_hist_kernel(const int32_t* __restrict__ gi, const int32_t* __restrict__ gp, const int32_t* __restrict__ cs,
                    int S, int ctas_per_split, int32_t nrow, uint32_t* __restrict__ cnt) {
  extern __shared__ uint32_t hsm[];
  const int h = blockIdx.x / ctas_per_split, g = blockIdx.x % ctas_per_split;
  if (PRIVATE) {
    for (int r = threadIdx.x; r < nrow; r += HIST_THREADS) hsm[r] = 0u;
    __syncthreads();
  }
  const int64_t k_lo = gp[cs[h]], k_hi = gp[cs[h + 1]];
  // slice boundaries on multiples of 4 entries inside [k_lo, k_hi) so the body can use 128-bit loads
  const int64_t a_lo = (k_lo + 3) & ~int64_t(3), a_hi = k_hi & ~int64_t(3);
  auto bump = [&](int32_t r) {
    if (PRIVATE)
      atomicAdd(&hsm[r], 1u);
    else
      ptx::red_add_u32(cnt + static_cast<int64_t>(r) * S + h, 1u);
  };
  if (a_lo < a_hi) {
    const int64_t n4 = (a_hi - a_lo) >> 2;
    const int64_t g_begin = (n4 * g) / ctas_per_split, g_end = (n4 * (g + 1)) / ctas_per_split;
    const int4* __restrict__ i4 = reinterpret_cast<const int4*>(gi + a_lo);
    for (int64_t q = g_begin + threadIdx.x; q < g_end; q += HIST_THREADS) {
      const int4 r = ptx::ld_stream_v4s32(i4 + q);
      bump(r.x);
      bump(r.y);
      bump(r.z);
      bump(r.w);
    }
    if (g == 0) {  // ragged head and tail of the split
      for (int64_t k = k_lo + threadIdx.x; k < a_lo && k < k_hi; k += HIST_THREADS) bump(gi[k]);
      for (int64_t k = a_hi + threadIdx.x; k < k_hi; k += HIST_THREADS) bump(gi[k]);
    }
  } else if (g == 0) {
    for (int64_t k = k_lo + threadIdx.x; k < k_hi; k += HIST_THREADS) bump(gi[k]);
  }
  if (PRIVATE) {
    __syncthreads();
    for (int r = threadIdx.x; r < nrow; r += HIST_THREADS) {
      const uint32_t c = hsm[r];
      if (c) ptx::red_add_u32(cnt + static_cast<int64_t>(r) * S + h, c);
    }
  }
}

// column split boundaries: cs[h] = first column whose start offset reaches h * nnz / S
__global__ void split_bounds_kernel(const int32_t* __restrict__ gp, int32_t ncol, int64_t nnz, int S,
                                    int32_t* __restrict__ cs) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h > S) return;
  if (h == 0) {
    cs[0] = 0;
    return;
  }
  if (h == S) {
    cs[S] = ncol;
    return;
  }
  const int64_t target = (nnz * h) / S;
  int32_t lo = 0, hi = ncol;
  while (lo < hi) {
    const int32_t mid = lo + ((hi - lo) >> 1);
    if (gp[mid] < target)
      lo = mid + 1;
    else
      hi = mid;
  }
  cs[h] = lo;
}

// rowptr[r] = scan[r * S] (the scan runs over (row, split) pairs, row-major)
__global__ void extract_rowptr_kernel(const int32_t* __restrict__ scan, int32_t nrow, int S, int32_t* __restrict__ rowptr) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r <= nrow; r += stride)
    rowptr[r] = scan[r * S];
}

// ================================================================================================
// P2: band boundaries.  key(r) = (1-eps) * p'[r]/nnz + eps * r/nrow is non-decreasing; band b starts
// at the first row whose key reaches b/nb.  eps > 0 bounds the rows of a band (shared memory).
// ================================================================================================
__global__ void band_bounds_kernel(const int32_t* __restrict__ rowptr, int32_t nrow, int64_t nnz, int nb, double eps,
                                   int32_t* __restrict__ rb) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b > nb) return;
  int32_t r;
  if (b == 0) {
    r = 0;
  } else if (b == nb) {
    r = nrow;
  } else {
    const double wa = (1.0 - eps) / static_cast<double>(nnz);
    const double wb = eps / static_cast<double>(nrow);
    const double target = static_cast<double>(b) / static_cast<double>(nb);
    int32_t lo = 0, hi = nrow;
    while (lo < hi) {
      const int32_t mid = lo + ((hi - lo) >> 1);
      const double key = static_cast<double>(rowptr[mid]) * wa + static_cast<double>(mid) * wb;
      if (key < target)
        lo = mid + 1;
      else
        hi = mid;
    }
    r = lo;
  }
  rb[b] = r;
}

__global__ void band_max_rows_kernel(const int32_t* __restrict__ rb, int nb, int32_t* __restrict__ max_rows) {
  int32_t mx = 0;
  for (int b = threadIdx.x; b < nb; b += blockDim.x) {
    const int32_t d = rb[b + 1] - rb[b];
    mx = d > mx ? d : mx;
  }
  atomicMax(max_rows, mx);
}

// ================================================================================================
// P3: band pointers over merge-path tiles (same plan as the sweeps: SWEEP_TILE items per tile)
// bpt[(b-1)*ncol + c] = first k in column c with i[k] >= rb[b], for b = 1..nb-1
// ================================================================================================
constexpr int BP_THREADS = 256;
constexpr int BP_IPT = SWEEP_TILE / BP_THREADS;
static_assert(BP_THREADS * BP_IPT == SWEEP_TILE, "band-pointer tiling must match the sweep plan");

__global__ void __launch_bounds__(BP_THREADS)
    band_ptr_kernel(const int32_t* __restrict__ gi, const int32_t* __restrict__ gp, const int32_t* __restrict__ plan,
                    int64_t n_tiles, int32_t ncol, int32_t nnz, const int32_t* __restrict__ rb, int nb,
                    int32_t* __restrict__ bpt) {
  extern __shared__ int32_t sm[];
  int32_t* as = sm;                      // as[j] = p[c0 + j], j = 0..nc+1   (SWEEP_TILE + 2)
  int32_t* is = sm + (SWEEP_TILE + 4);   // is[j] = i[k0 - 1 + j]            (SWEEP_TILE + 1)
  int32_t* rbs = is + (SWEEP_TILE + 4);  // rbs[b] = rb[b], b = 0..nb
  for (int b = threadIdx.x; b <= nb; b += BP_THREADS) rbs[b] = rb[b];
  const int64_t total_items = static_cast<int64_t>(ncol) + nnz;

  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    __syncthreads();  // previous tile fully consumed (also covers the rbs fill)
    const int32_t c0 = plan[t], c1 = plan[t + 1];
    const int64_t d0 = t * SWEEP_TILE;
    int64_t d1 = d0 + SWEEP_TILE;
    if (d1 > total_items) d1 = total_items;
    const int32_t k0 = static_cast<int32_t>(d0 - c0), k1 = static_cast<int32_t>(d1 - c1);
    const int nc = c1 - c0, nk = k1 - k0;
    const int a_last = (c1 + 1 <= ncol) ? c1 + 1 : ncol;  // p index
    for (int j = threadIdx.x; c0 + j <= a_last; j += BP_THREADS) as[j] = gp[c0 + j];
    for (int j = threadIdx.x; j <= nk; j += BP_THREADS) {
      const int32_t k = k0 - 1 + j;
      is[j] = (k >= 0 && k < nnz) ? ptx::ld_stream_s32(gi + k) : 0;
    }
    __syncthreads();

    const int items = nc + nk;
    int d_lo = threadIdx.x * BP_IPT;
    if (d_lo > items) d_lo = items;
    int d_hi = d_lo + BP_IPT;
    if (d_hi > items) d_hi = items;
    if (d_lo >= d_hi) continue;
    // column ends consumed before d_lo: end of column c0+j is as[j+1]
    int lo = d_lo > nk ? d_lo - nk : 0;
    int hi = d_lo < nc ? d_lo : nc;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (as[mid + 1] - k0 <= d_lo - mid - 1)
        lo = mid + 1;
      else
        hi = mid;
    }
    int ci = lo;
    int ki = d_lo - ci;             // relative to k0; entry k0+ki is is[ki+1]
    int col_end = as[ci + 1] - k0;  // relative end of column c0+ci (stale past the last column: no items remain)
    // band of the previous entry when I start inside a column
    int cur = 0;
    if (k0 + ki > as[ci]) {  // column c0+ci started before my first item
      const int32_t prev_row = is[ki];
      int blo = 0, bhi = nb;  // largest b with rbs[b] <= prev_row
      while (blo < bhi) {
        const int mid = (blo + bhi + 1) >> 1;
        if (rbs[mid] <= prev_row)
          blo = mid;
        else
          bhi = mid - 1;
      }
      cur = blo;
    }
    int32_t next_rb = rbs[cur + 1];  // cur <= nb-1 always (rows < nrow = rbs[nb])
    for (int it = d_lo; it < d_hi; ++it) {
      const int64_t c = c0 + ci;
      if (ki < col_end) {
        const int32_t row = is[ki + 1];
        while (row >= next_rb) {  // entering band cur+1 (possibly skipping empty bands)
          ++cur;
          bpt[static_cast<int64_t>(cur - 1) * ncol + c] = k0 + ki;
          next_rb = rbs[cur + 1];
        }
        ++ki;
      } else {
        const int32_t e = k0 + col_end;
        while (cur < nb - 1) {  // bands after the column's last entry start at its end
          ++cur;
          bpt[static_cast<int64_t>(cur - 1) * ncol + c] = e;
        }
        cur = 0;
        next_rb = rbs[1];
        ++ci;
        col_end = as[ci + 1] - k0;
      }
    }
  }
}

// ================================================================================================
// shared skeleton of the band kernels
// ================================================================================================
constexpr int BAND_THREADS = 512;
constexpr int BAND_WARPS = BAND_THREADS / 32;
constexpr int BAND_CH = BAND_THREADS;  // columns per chunk: 32 per warp, one run descriptor per lane

// ================================================================================================
// row-indexed sums: rowSums / rowMeans / A v
// ================================================================================================
constexpr int BAND_UNROLL = 4;

struct ScatterItem {
  int32_t r;
  double xv, w;
};

struct ScatterArgs {
  BandView bv;
  const double* v;  // [ncol] or null (rowSums)
  double* out;      // [nrow]; pre-zeroed when S > 1
  int max_rows;     // accumulator capacity (rows of the widest band)
  // Lockstep: the CTAs of one column split advance through the columns together (a soft barrier every
  // `lock_every` chunks), so the 32-byte sectors that neighbouring bands share are fetched from HBM
  // once and hit L2 for everyone else.  Needs all CTAs co-resident (cooperative launch); 0 = off.
  int lock_every;
  unsigned int* lock_counters;  // [S], zeroed before the launch
  int cluster;                  // CTAs per thread-block cluster (adjacent bands), 1 = no clusters
  const double* mean;           // rowVars' second pass: [nrow] row means (band_var_kernel), else null
  int mean_rows;                // rows of mean staged per band (the widest band), 0 without
};

constexpr int SC_CAPW = 512;       // flattened entries a warp stages per round
constexpr int SC_PRIVATE_ROWS = 256;  // bands this narrow get one accumulator copy PER WARP (32 KB)

static size_t scatter_smem_bytes(int max_rows, bool spmv, int mean_rows = 0) {
  size_t rows = static_cast<size_t>(max_rows > 0 ? max_rows : 1);
  if (rows < static_cast<size_t>(BAND_WARPS) * SC_PRIVATE_ROWS) rows = static_cast<size_t>(BAND_WARPS) * SC_PRIVATE_ROWS;
  return sizeof(double) * (rows + static_cast<size_t>(mean_rows)) + BAND_WARPS * SC_CAPW * sizeof(int32_t) +
         (spmv ? BAND_WARPS * SC_CAPW : 0) + 16;
}

// CTA (band b, column split h).  A warp takes 32 consecutive columns of the chunk, one run descriptor
// per lane.  Instead of searching the run of every entry, each lane EXPANDS its own run into the
// warp's flat list in shared memory (entry index per slot; ~1 store per entry), then the lanes walk
// the list 32 slots at a time, so consecutive lanes read consecutive entries of a run (coalesced),
// U loads in flight before the first shared-memory FP64 add.
// VAR (rowVars' second pass): the band's slice of the row means sits in shared memory after the accumulators, and an
// entry adds (x - mean[row])^2 instead of x.
// (tid = threadIdx.x, read in the kernel itself: there the compiler knows its range from the launch bounds)
template <bool SPMV, bool VAR>
__device__ __forceinline__ void band_scatter_body(const ScatterArgs& a, const int tid) {
  extern __shared__ __align__(16) unsigned char ssm[];
  const BandView& bv = a.bv;
  const int MR = a.max_rows;
  double* acc = reinterpret_cast<double*>(ssm);
  double* means = acc + MR;  // VAR only
  const int lane = tid & 31, warp = tid >> 5;
  double* const acc_end = acc + MR + (VAR ? a.mean_rows : 0);
  int32_t* flat = reinterpret_cast<int32_t*>(acc_end) + warp * SC_CAPW;
  uint8_t* flatl = reinterpret_cast<uint8_t*>(reinterpret_cast<int32_t*>(acc_end) + BAND_WARPS * SC_CAPW) + warp * SC_CAPW;
  constexpr int U = BAND_UNROLL;
  const int units = bv.nb * bv.S;
  for (int u = blockIdx.x; u < units; u += gridDim.x) {
    const int h = u / bv.nb, b = u % bv.nb;  // consecutive CTAs = consecutive bands of one split
    const int32_t row0 = bv.rb[b];
    const int32_t R = bv.rb[b + 1] - row0;  // an empty band still takes part in the split's barriers
    const int32_t c_lo = bv.cs[h], c_hi = bv.cs[h + 1];
    // A narrow band is a band of POPULAR rows (bands hold equal numbers of entries): every warp step
    // then carries several entries of the same row, and 32 warps hammering a handful of shared-memory
    // words with CAS loops serialise.  Such bands get one accumulator copy per warp; inside a step equal
    // rows are combined with match.any + shuffles and one lane per row does a plain add.  No atomics.
    const bool priv = R <= SC_PRIVATE_ROWS;
    double* wacc = acc + (priv ? warp * R : 0);
    const unsigned lt_mask = (1u << lane) - 1u;
    __syncthreads();
    for (int r = tid; r < (priv ? R * BAND_WARPS : R); r += BAND_THREADS) acc[r] = 0.0;
    if constexpr (VAR)
      for (int r = tid; r < R; r += BAND_THREADS) means[r] = __ldg(a.mean + row0 + r);
    __syncthreads();
    // software-pipelined descriptors: the next chunk's are fetched (and its runs prefetched to L2)
    // while the current chunk is walked
    int32_t ns = 0, ne = 0;
    double nv = 0.0;
    {
      const int64_t c = static_cast<int64_t>(c_lo) + tid;
      if (c < c_hi && R > 0) {
        ns = band_start(bv, b, c);
        ne = band_start(bv, b + 1, c);
        if (SPMV) nv = __ldg(a.v + c);
      }
    }
    int chunk_no = 0;
    for (int64_t cbase = c_lo; cbase < c_hi; cbase += BAND_CH, ++chunk_no) {
      if (a.cluster > 1) {
        // the CTAs of a cluster own ADJACENT bands of the same split: keep them on the same chunk
        // (hardware cluster barrier), so the sectors their neighbouring runs share are fetched once
        asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");
        asm volatile("barrier.cluster.wait.aligned;" ::: "memory");
      }
      if (a.lock_every > 0 && chunk_no % a.lock_every == 0) {
        // soft barrier across the bv.nb CTAs of split h (all resident: cooperative launch)
        __syncthreads();
        if (tid == 0) {
          const unsigned int target = static_cast<unsigned int>(bv.nb) * (chunk_no / a.lock_every + 1);
          atomicAdd(a.lock_counters + h, 1u);
          unsigned int seen;
          do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(a.lock_counters + h) : "memory");
            if (seen < target) __nanosleep(64);
          } while (seen < target);
        }
        __syncthreads();
      }
      const int32_t s = ns, len = ne - ns;
      const double vc = nv;
      ns = ne = 0;
      nv = 0.0;
      {
        const int64_t c = cbase + BAND_CH + tid;
        if (c < c_hi && R > 0) {
          ns = band_start(bv, b, c);
          ne = band_start(bv, b + 1, c);
          if (SPMV) nv = __ldg(a.v + c);
          if (a.lock_every == 0) {  // without lockstep, at least pull the next runs towards L2 early
            for (int32_t k = ns & ~31; k < ne; k += 32) ptx::prefetch_l2(bv.i + k);
            for (int32_t k = ns & ~15; k < ne; k += 16) ptx::prefetch_l2(bv.x + k);
          }
        }
      }
      int32_t incl = len;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const int32_t up = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += up;
      }
      const int32_t excl = incl - len;
      const int32_t total = __shfl_sync(0xffffffffu, incl, 31);
      for (int32_t base = 0; base < total; base += SC_CAPW) {  // one round unless the runs are long
        // owner expansion of the slots [base, base + SC_CAPW)
        int32_t j0 = base - excl;
        if (j0 < 0) j0 = 0;
        int32_t j1 = base + SC_CAPW - excl;
        if (j1 > len) j1 = len;
        for (int32_t j = j0; j < j1; ++j) {
          flat[excl + j - base] = s + j;
          if (SPMV) flatl[excl + j - base] = static_cast<uint8_t>(lane);
        }
        __syncwarp();
        int32_t n = total - base;
        if (n > SC_CAPW) n = SC_CAPW;
        for (int32_t q0 = 0; q0 < n; q0 += 32 * U) {
          int32_t rr[U];
          double xx[U];
#pragma unroll
          for (int t = 0; t < U; ++t) {
            const int32_t q = q0 + t * 32 + lane;
            rr[t] = -1;
            xx[t] = 0.0;
            if (q < n) {
              const int32_t k = flat[q];
              rr[t] = ptx::ld_stream_s32(bv.i + k) - row0;
              xx[t] = ptx::ld_stream_f64(bv.x + k);
            }
          }
          if (SPMV) {
#pragma unroll
            for (int t = 0; t < U; ++t) {
              const int32_t q = q0 + t * 32 + lane;
              const int l = (q < n) ? flatl[q] : 0;
              const double w = __shfl_sync(0xffffffffu, vc, l);
              xx[t] = __dmul_rn(xx[t], w);
            }
          }
          if constexpr (VAR) {
#pragma unroll
            for (int t = 0; t < U; ++t) {
              if (rr[t] >= 0) {
                const double d = __dsub_rn(xx[t], means[rr[t]]);
                xx[t] = __dmul_rn(d, d);
              }
            }
          }
          if (priv) {
#pragma unroll
            for (int t = 0; t < U; ++t) {
              if (q0 + t * 32 >= n) break;  // warp-uniform
              const unsigned same = __match_any_sync(0xffffffffu, rr[t] >= 0 ? rr[t] : -1 - lane);
              // the lowest lane of each group gathers the group's values (groups are small: a row appears
              // at most once per column)
              double sum = xx[t];
              unsigned rest = same & ~lt_mask & ~(1u << lane);  // members above me
              const bool leader = (same & lt_mask) == 0u;
              unsigned pending = __ballot_sync(0xffffffffu, leader && rest != 0u);
              while (pending) {  // warp-uniform loop: at most (largest group - 1) rounds
                const int src = rest ? (__ffs(rest) - 1) : lane;
                const double v = __shfl_sync(0xffffffffu, xx[t], src);
                if (leader && rest) {
                  sum = __dadd_rn(sum, v);
                  rest &= rest - 1;
                }
                pending = __ballot_sync(0xffffffffu, leader && rest != 0u);
              }
              if (leader && rr[t] >= 0) wacc[rr[t]] = __dadd_rn(wacc[rr[t]], sum);
              __syncwarp();
            }
          } else {
#pragma unroll
            for (int t = 0; t < U; ++t)
              if (rr[t] >= 0) atomicAdd(&acc[rr[t]], xx[t]);
          }
        }
        __syncwarp();
      }
    }
    __syncthreads();
    for (int r = tid; r < R; r += BAND_THREADS) {
      double v = acc[r];
      if (priv) {
#pragma unroll
        for (int w = 1; w < BAND_WARPS; ++w) v = __dadd_rn(v, acc[w * R + r]);  // fixed order
      }
      if (bv.S == 1)
        a.out[row0 + r] = v;
      else
        ptx::red_add_f64(a.out + row0 + r, v);
    }
  }
}

template <bool SPMV>
__global__ void __launch_bounds__(BAND_THREADS) band_scatter_kernel(const ScatterArgs a) {
  band_scatter_body<SPMV, false>(a, threadIdx.x);
}

__global__ void __launch_bounds__(BAND_THREADS) band_var_kernel(const ScatterArgs a) { band_scatter_body<false, true>(a, threadIdx.x); }

// ================================================================================================
// transpose: banded stable scatter
// ================================================================================================
struct PlaceItem {
  int32_t r, col;
  double xv;
};

struct TransposeArgs {
  BandView bv;
  const int32_t* off;  // [nrow*S (+1)] first output slot of (row r, split h): off[r*S + h]
  int32_t* i_out;
  double* x_out;
  int max_rows;  // R capacity of the shared-memory tables (even)
  int cluster;   // CTAs per thread-block cluster (adjacent bands of one split kept on the same chunk), 1 = none
};

constexpr int TR_CAPW = 384;  // flattened entries of a warp's 32 columns kept in shared memory between the passes

static size_t transpose_smem_bytes(int max_rows) {
  const size_t R = static_cast<size_t>(max_rows);
  return R * 4 * 2 /* cursor, rowpos */ + R * 2 * BAND_WARPS * 2 /* cnt, rel (u16) */ +
         static_cast<size_t>(BAND_WARPS) * TR_CAPW * (4 + 2 + 2) /* entry index, row, column-in-warp */ + 32;
}

__global__ void __launch_bounds__(BAND_THREADS) band_transpose_kernel(const TransposeArgs a) {
  extern __shared__ __align__(16) unsigned char tsm[];
  const BandView& bv = a.bv;
  const int MR = a.max_rows;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint32_t* cursor = reinterpret_cast<uint32_t*>(tsm);                      // [MR] next free slot of each row
  uint32_t* rowpos = cursor + MR;                                           // [MR] slot base of the row for this chunk
  uint32_t* cntw = rowpos + MR;                                             // [WARPS*MR/2] u16 pairs: entries of (warp, row)
  uint16_t* rel = reinterpret_cast<uint16_t*>(cntw + (BAND_WARPS * MR) / 2);  // [WARPS*MR] running offset of (warp, row)
  uint16_t* cnt16 = reinterpret_cast<uint16_t*>(cntw);
  int32_t* flatk_all = reinterpret_cast<int32_t*>(rel + static_cast<size_t>(BAND_WARPS) * MR);  // [WARPS][CAPW]
  uint16_t* flatr_all = reinterpret_cast<uint16_t*>(flatk_all + BAND_WARPS * TR_CAPW);
  uint16_t* flatl_all = flatr_all + BAND_WARPS * TR_CAPW;
  int32_t* flatk = flatk_all + warp * TR_CAPW;   // entry index of every flattened slot of my 32 columns
  uint16_t* flatr = flatr_all + warp * TR_CAPW;  // its row inside the band (filled by pass 1)
  uint16_t* flatl = flatl_all + warp * TR_CAPW;  // its column inside the warp's 32
  const unsigned lt_mask = (1u << lane) - 1u;
  const int units = bv.nb * bv.S;

  for (int u = blockIdx.x; u < units; u += gridDim.x) {
    const int h = u / bv.nb, b = u % bv.nb;
    const int32_t row0 = bv.rb[b];
    const int32_t R = bv.rb[b + 1] - row0;  // an empty band still walks the chunks (cluster barriers)
    const int32_t c_lo = bv.cs[h], c_hi = bv.cs[h + 1];
    __syncthreads();
    for (int r = tid; r < R; r += BAND_THREADS)
      cursor[r] = static_cast<uint32_t>(a.off[static_cast<int64_t>(row0 + r) * bv.S + h]);
    for (int e = tid; e < (BAND_WARPS * MR) / 2; e += BAND_THREADS) cntw[e] = 0u;
    __syncthreads();

    auto count = [&](int32_t r) {
      const int idx = warp * MR + r;
      atomicAdd(&cntw[idx >> 1], 1u << ((idx & 1) * 16));
    };
    // equal rows inside a 32-entry step are ranked in lane order = source column order
    auto place = [&](int32_t r, int32_t col, double xv) {
      const unsigned same = __match_any_sync(0xffffffffu, r >= 0 ? r : -1 - lane);
      if (r >= 0) {
        const int idx = warp * MR + r;
        const uint32_t my = rel[idx];
        const uint32_t pos = rowpos[r] + my + __popc(same & lt_mask);
        a.i_out[pos] = col;
        a.x_out[pos] = xv;
        if ((same >> lane) == 1u) rel[idx] = static_cast<uint16_t>(my + __popc(same));  // highest lane of the group
      }
      __syncwarp();
    };

    int32_t ns = 0, ne = 0;
    {
      const int64_t c = static_cast<int64_t>(c_lo) + tid;
      if (c < c_hi && R > 0) {
        ns = band_start(bv, b, c);
        ne = band_start(bv, b + 1, c);
      }
    }
    for (int64_t cbase = c_lo; cbase < c_hi; cbase += BAND_CH) {
      if (a.cluster > 1) {
        // adjacent bands read adjacent runs of the same columns: keep the cluster on the same chunk so
        // HBM sees one stream per column block instead of hundreds of unrelated 32-byte reads
        asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");
        asm volatile("barrier.cluster.wait.aligned;" ::: "memory");
      }
      const int32_t s = ns, e = ne;
      ns = ne = 0;
      {
        const int64_t c = cbase + BAND_CH + tid;
        if (c < c_hi && R > 0) {
          ns = band_start(bv, b, c);
          ne = band_start(bv, b + 1, c);
          for (int32_t k = ns & ~31; k < ne; k += 32) ptx::prefetch_l2(bv.i + k);
          for (int32_t k = ns & ~15; k < ne; k += 16) ptx::prefetch_l2(bv.x + k);
        }
      }
      const int32_t len = e - s;
      int32_t incl = len;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const int32_t up = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += up;
      }
      const int32_t excl = incl - len;
      const int32_t total = __shfl_sync(0xffffffffu, incl, 31);
      const bool cached = total <= TR_CAPW;  // warp-uniform: the common case
      const int32_t col0 = static_cast<int32_t>(cbase) + 32 * warp;

      // ---- pass 1: entries per (warp, row) of this chunk (order-free) -------------------------------
      if (cached) {
        // each lane expands its own run into the warp's flat list (one store per entry, no per-entry
        // search); then 32 consecutive slots per step = consecutive entries of a run (coalesced)
        for (int32_t j = 0; j < len; ++j) {
          flatk[excl + j] = s + j;
          flatl[excl + j] = static_cast<uint16_t>(lane);
        }
        __syncwarp();
        for (int32_t q0 = 0; q0 < total; q0 += 32 * BAND_UNROLL) {
          int32_t rr[BAND_UNROLL];
#pragma unroll
          for (int t = 0; t < BAND_UNROLL; ++t) {
            const int32_t q = q0 + t * 32 + lane;
            rr[t] = (q < total) ? __ldg(bv.i + flatk[q]) - row0 : -1;
          }
#pragma unroll
          for (int t = 0; t < BAND_UNROLL; ++t) {
            const int32_t q = q0 + t * 32 + lane;
            if (rr[t] >= 0) {
              flatr[q] = static_cast<uint16_t>(rr[t]);
              count(rr[t]);
            }
          }
        }
      } else {
        warp_walk_runs<BAND_UNROLL, int32_t>(
            s, len, lane, [&](int32_t k, int l, bool valid) { return valid ? __ldg(bv.i + k) - row0 : -1; },
            [&](const int32_t& r) {
              if (r >= 0) count(r);
            });
      }
      __syncthreads();
      // ---- per row: slot ranges of the 16 warps in warp (= column) order; advance the cursor ------------
      for (int r = tid; r < R; r += BAND_THREADS) {
        uint32_t run = 0;
#pragma unroll
        for (int w = 0; w < BAND_WARPS; ++w) {
          const uint32_t c = cnt16[w * MR + r];
          rel[w * MR + r] = static_cast<uint16_t>(run);
          cnt16[w * MR + r] = 0;
          run += c;
        }
        const uint32_t base = cursor[r];
        rowpos[r] = base;
        cursor[r] = base + run;
      }
      __syncthreads();
      // ---- pass 2: place --------------------------------------------------------------------------------
      if (cached) {
        for (int32_t q0 = 0; q0 < total; q0 += 32 * BAND_UNROLL) {
          int32_t rr[BAND_UNROLL], cc[BAND_UNROLL];
          double xx[BAND_UNROLL];
#pragma unroll
          for (int t = 0; t < BAND_UNROLL; ++t) {
            const int32_t q = q0 + t * 32 + lane;
            rr[t] = -1;
            cc[t] = 0;
            xx[t] = 0.0;
            if (q < total) {
              rr[t] = flatr[q];
              cc[t] = col0 + flatl[q];
              xx[t] = ptx::ld_stream_f64(bv.x + flatk[q]);
            }
          }
#pragma unroll
          for (int t = 0; t < BAND_UNROLL; ++t)
            if (q0 + t * 32 < total) place(rr[t], cc[t], xx[t]);  // warp-uniform guard
        }
        __syncwarp();
      } else {
        warp_walk_runs<BAND_UNROLL, PlaceItem>(
            s, len, lane,
            [&](int32_t k, int l, bool valid) {
              PlaceItem it;
              it.r = -1;
              it.col = col0 + l;
              it.xv = 0.0;
              if (valid) {
                it.r = __ldg(bv.i + k) - row0;
                it.xv = ptx::ld_stream_f64(bv.x + k);
              }
              return it;
            },
            [&](const PlaceItem& it) { place(it.r, it.col, it.xv); });
      }
    }
  }
}

}  // namespace

// ================================================================================================
// the plan
// ================================================================================================
void free_band_plan(BandPlan* bp, cudaStream_t s) {
  if (!bp) return;
  pool_free(bp->d_rb, s);
  pool_free(bp->d_cs, s);
  pool_free(bp->d_bpt, s);
  if (bp->d_off != bp->d_rowptr) pool_free(bp->d_off, s);
  pool_free(bp->d_rowptr, s);
  delete bp;
}

// rows_cap: most rows a band may hold (consumer's shared-memory budget); want_bands: preferred band
// count; S: column splits.  nnz > 0 and nrow > 0 required.
int build_band_plan(sb200_matrix* m, int rows_cap, int want_bands, int S, BandPlan** out) {
  cudaStream_t st = m->stream;
  const int32_t nrow = m->nrow, ncol = m->ncol;
  const int64_t nnz = m->nnz;
  BandPlan* bp = new (std::nothrow) BandPlan();
  if (!bp) return fail(SB200_E_NOMEM, "host allocation failed");
  struct Guard {
    BandPlan*& p;
    cudaStream_t s;
    bool armed = true;
    ~Guard() {
      if (armed) free_band_plan(p, s);
    }
  } guard{bp, st};
  PhaseTrace tr(st);
  tr.mark("start");

  // ---- geometry: enough bands that none exceeds rows_cap, not more than leaves ~3 entries per run ----
  const double cap = 0.9 * rows_cap;
  int nb = want_bands;
  const int64_t floor_rows = static_cast<int64_t>((nrow + cap - 1) / cap);
  const int64_t by_density = nnz / (static_cast<int64_t>(ncol > 0 ? ncol : 1) * 3);
  if (nb > by_density) nb = static_cast<int>(by_density);
  if (nb < floor_rows) nb = static_cast<int>(floor_rows);
  if (nb < 1) nb = 1;
  if (const char* e = getenv("SB200_BANDS")) {
    const int v = atoi(e);
    if (v >= floor_rows) nb = v;
  }
  double eps = static_cast<double>(nrow) / (static_cast<double>(nb) * cap);
  if (eps < 1e-3) eps = 1e-3;
  if (eps > 1.0) eps = 1.0;
  if (S < 1) S = 1;
  if (S > ncol) S = ncol > 0 ? ncol : 1;
  bp->nb = nb;
  bp->S = S;

  const int64_t scan_n = static_cast<int64_t>(nrow) * S;
  if (scan_n > 2000000000LL) return fail(SB200_E_UNSUPPORTED, "band plan: nrow * splits too large");
  uint32_t* d_cnt = nullptr;
  void* d_scan_ws = nullptr;
  int32_t* d_maxrows = nullptr;
  const size_t scan_ws = scan_workspace_bytes(scan_n);
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&d_cnt), sizeof(uint32_t) * static_cast<size_t>(scan_n), st));
  struct Tmp {
    void* p[3];
    cudaStream_t s;
    ~Tmp() {
      for (void* q : p) pool_free(q, s);
    }
  } tmp{{d_cnt, nullptr, nullptr}, st};
  SB_TRY(pool_alloc(&d_scan_ws, scan_ws, st));
  tmp.p[1] = d_scan_ws;
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&d_maxrows), sizeof(int32_t), st));
  tmp.p[2] = d_maxrows;
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&bp->d_cs), sizeof(int32_t) * (S + 1), st));
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&bp->d_rb), sizeof(int32_t) * (nb + 1), st));
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&bp->d_off), sizeof(int32_t) * static_cast<size_t>(scan_n + 1), st));
  if (S == 1) {
    bp->d_rowptr = bp->d_off;
  } else {
    SB_TRY(pool_alloc(reinterpret_cast<void**>(&bp->d_rowptr), sizeof(int32_t) * (static_cast<size_t>(nrow) + 1), st));
  }
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&bp->d_bpt),
                    sizeof(int32_t) * static_cast<size_t>(nb > 1 ? nb - 1 : 1) * static_cast<size_t>(ncol > 0 ? ncol : 1), st));

  // ---- P1 --------------------------------------------------------------------------------------------
  split_bounds_kernel<<<(S + 1 + 63) / 64, 64, 0, st>>>(m->d_p, ncol, nnz, S, bp->d_cs);
  count_launch();
  SB_CUDA(cudaGetLastError());
  SB_CUDA(cudaMemsetAsync(d_cnt, 0, sizeof(uint32_t) * static_cast<size_t>(scan_n), st));
  {
    int per_split = (m->sm_count + S - 1) / S;
    const int64_t by_work = (nnz / S) / (HIST_THREADS * 16) + 1;
    if (per_split > by_work) per_split = static_cast<int>(by_work);
    if (per_split < 1) per_split = 1;
    if (nrow <= HIST_SMEM_MAX_WORDS) {
      const size_t smem = sizeof(uint32_t) * static_cast<size_t>(nrow);
      SB_CUDA(cudaFuncSetAttribute(row_hist_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
      row_hist_kernel<true><<<S * per_split, HIST_THREADS, smem, st>>>(m->d_i, m->d_p, bp->d_cs, S, per_split, nrow, d_cnt);
    } else {
      per_split *= 4;
      row_hist_kernel<false><<<S * per_split, HIST_THREADS, 0, st>>>(m->d_i, m->d_p, bp->d_cs, S, per_split, nrow, d_cnt);
    }
    count_launch();
    SB_CUDA(cudaGetLastError());
  }
  tr.mark("hist");
  SB_TRY(exclusive_scan_u32(st, d_cnt, bp->d_off, scan_n, nullptr, d_scan_ws, scan_ws));
  if (S > 1) {
    int64_t blocks = (static_cast<int64_t>(nrow) + 1 + 255) / 256;
    if (blocks > 1184) blocks = 1184;
    extract_rowptr_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(bp->d_off, nrow, S, bp->d_rowptr);
    count_launch();
    SB_CUDA(cudaGetLastError());
  }
  bp->has_offsets = true;
  tr.mark("scan");
  // ---- P2 ---------------------------------------------------------------------------------------------
  band_bounds_kernel<<<(nb + 1 + 127) / 128, 128, 0, st>>>(bp->d_rowptr, nrow, nnz, nb, eps, bp->d_rb);
  count_launch();
  SB_CUDA(cudaGetLastError());
  SB_CUDA(cudaMemsetAsync(d_maxrows, 0, sizeof(int32_t), st));
  band_max_rows_kernel<<<1, 256, 0, st>>>(bp->d_rb, nb, d_maxrows);
  count_launch();
  SB_CUDA(cudaGetLastError());
  int32_t h_maxrows = 0;
  SB_CUDA(cudaMemcpyAsync(&h_maxrows, d_maxrows, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  tr.mark("bands");
  // ---- P3 ---------------------------------------------------------------------------------------------
  SB_TRY(launch_band_ptr(m, bp->d_rb, nb, bp->d_bpt));
  tr.mark("band ptrs");
  SB_CUDA(cudaStreamSynchronize(st));
  bp->max_rows = h_maxrows;
  tr.report("band plan nb=%d S=%d maxrows=%d:", bp->nb, bp->S, bp->max_rows);
  if (h_maxrows > rows_cap) return fail(SB200_E_UNSUPPORTED, "band plan: a row band exceeds its shared-memory budget");
  guard.armed = false;
  *out = bp;
  return SB200_OK;
}

// Band pointers for caller-given band bounds d_rb[0..nb] (rb[0] = 0, rb[nb] = nrow, non-decreasing), on the
// matrix's stream: d_bpt[(b-1)*ncol + c] = first k of column c with i[k] >= rb[b], b = 1..nb-1.  Used by the band
// plan above and by the band-major companion builder (bmc.cu).
int launch_band_ptr(sb200_matrix* m, const int32_t* d_rb, int nb, int32_t* d_bpt) {
  if (nb <= 1 || m->n_tiles == 0) return SB200_OK;
  const size_t smem = sizeof(int32_t) * (2 * (SWEEP_TILE + 4) + static_cast<size_t>(nb) + 1);
  if (smem > 220 * 1024) return fail(SB200_E_UNSUPPORTED, "band pointers: too many row bands for one pass");
  SB_CUDA(cudaFuncSetAttribute(band_ptr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  int64_t blocks = m->n_tiles;
  const int64_t capb = static_cast<int64_t>(m->sm_count) * 6;
  if (blocks > capb) blocks = capb;
  band_ptr_kernel<<<static_cast<unsigned>(blocks), BP_THREADS, smem, m->stream>>>(m->d_i, m->d_p, m->d_plan, m->n_tiles, m->ncol,
                                                                                  static_cast<int32_t>(m->nnz), d_rb, nb, d_bpt);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return SB200_OK;
}

BandView make_view(const sb200_matrix* m, const BandPlan* bp) {
  BandView v;
  v.i = m->d_i;
  v.p = m->d_p;
  v.x = m->d_x;
  v.ncol = m->ncol;
  v.nb = bp->nb;
  v.S = bp->S;
  v.rb = bp->d_rb;
  v.cs = bp->d_cs;
  v.bpt = bp->d_bpt;
  return v;
}

// ---- row-indexed sums ----------------------------------------------------------------------------------
constexpr int SCATTER_ROWS_CAP = 12288;  // 96 KB of FP64 accumulators: two CTAs per SM

namespace {
// columns (non-empty) whose length is below `thresh`: their band runs would be shorter than ~3 entries
__global__ void short_columns_kernel(const int32_t* __restrict__ gp, int32_t ncol, int32_t thresh,
                                     unsigned int* __restrict__ out /* [2]: short, non-empty */) {
  unsigned int n_short = 0, n_some = 0;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; c < ncol; c += stride) {
    const int32_t len = gp[c + 1] - gp[c];
    if (len > 0) {
      ++n_some;
      if (len < thresh) ++n_short;
    }
  }
  n_short = __reduce_add_sync(0xffffffffu, n_short);
  n_some = __reduce_add_sync(0xffffffffu, n_some);
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(out, n_short);
    atomicAdd(out + 1, n_some);
  }
}
}  // namespace

// Which kernel serves rowSums / rowMeans / A v for this matrix (decided once per handle):
//   banded (1) when popular rows would serialise the L2 atomics (small row range), or when columns
//   are long enough that a band's run per column is several entries; the plan-free L2-atomic path (0)
//   when many columns are short (skewed column lengths: runs of 1-2 entries waste sectors).
// Measured on B200: C2 (uniform, 1000/col) banded 0.50 vs 0.60 ms; C3 (30k rows) 22 vs 42 ms;
// C4 (power-law columns) 12.9 vs 11.6 ms.
int decide_row_path(sb200_matrix* m) {
  if (m->row_path >= 0) return SB200_OK;
  int path = 0;
  if (m->nnz > 0 && m->nrow > 0 && m->ncol > 0) {
    if (m->nrow <= 65536) {
      path = 1;
    } else {
      unsigned int* d_cnt = reinterpret_cast<unsigned int*>(static_cast<unsigned char*>(m->d_ws) + 16 + 4 * 1024 + 8 * 1024);
      SB_CUDA(cudaMemsetAsync(d_cnt, 0, 2 * sizeof(unsigned int), m->stream));
      int64_t blocks = (static_cast<int64_t>(m->ncol) + 255) / 256;
      if (blocks > m->sm_count * 8) blocks = m->sm_count * 8;
      short_columns_kernel<<<static_cast<unsigned>(blocks), 256, 0, m->stream>>>(m->d_p, m->ncol, 3 * m->sm_count, d_cnt);
      count_launch();
      SB_CUDA(cudaGetLastError());
      unsigned int h[2] = {0, 0};
      SB_CUDA(cudaMemcpyAsync(h, d_cnt, sizeof(h), cudaMemcpyDeviceToHost, m->stream));
      SB_CUDA(cudaStreamSynchronize(m->stream));
      SB_CUDA(cudaMemsetAsync(d_cnt, 0, 2 * sizeof(unsigned int), m->stream));
      path = (h[1] > 0 && 4ull * h[0] <= h[1]) ? 1 : 0;  // at most a quarter of the columns are short
    }
  }
  if (const char* e = getenv("SB200_ROW_PLAN")) path = (e[0] != '0') ? 1 : 0;
  if (m->nnz == 0 || m->nrow == 0 || m->ncol == 0) path = 0;
  m->row_path = path;
  return SB200_OK;
}

int ensure_scatter_plan(sb200_matrix* m) {
  if (m->plan_scatter) return SB200_OK;
  const int bands = m->sm_count;      // one band per SM ...
  int S = 4;                          // ... times four column splits = two waves of two CTAs per SM
  if (const char* e = getenv("SB200_SCATTER_SPLITS")) {
    const int v = atoi(e);
    if (v >= 1 && v <= 64) S = v;
  }
  return build_band_plan(m, SCATTER_ROWS_CAP, bands, S, &m->plan_scatter);
}

// d_mean set: rowVars' second pass (band_var_kernel), d_v is null then
static int launch_band_scatter_impl(sb200_matrix* m, const double* d_v, const double* d_mean, double* d_out) {
  SB_TRY(ensure_scatter_plan(m));
  const BandPlan* bp = m->plan_scatter;
  ScatterArgs a;
  a.bv = make_view(m, bp);
  a.v = d_v;
  a.out = d_out;
  a.mean = d_mean;
  a.mean_rows = d_mean ? (bp->max_rows > 0 ? bp->max_rows : 1) : 0;
  if (bp->S > 1) SB_CUDA(cudaMemsetAsync(d_out, 0, sizeof(double) * static_cast<size_t>(m->nrow), m->stream));
  a.max_rows = (bp->max_rows > 0 ? bp->max_rows : 1);
  if (a.max_rows < BAND_WARPS * SC_PRIVATE_ROWS) a.max_rows = BAND_WARPS * SC_PRIVATE_ROWS;  // room for the per-warp copies
  const size_t smem = scatter_smem_bytes(a.max_rows, d_v != nullptr, a.mean_rows);
  int ctas = static_cast<int>((200 * 1024) / (smem + 2048));
  if (ctas > 2) ctas = 2;
  if (ctas < 1) ctas = 1;
  int grid = m->sm_count * ctas;
  if (grid > bp->nb * bp->S) grid = bp->nb * bp->S;
  // lockstep every few chunks: the columns in flight (all resident splits) should stay well inside L2
  // measured (profiles/r01): barriers every 1/2/4/8 chunks cost more than the L2 hits they buy at C2
  // (0.73/0.63/0.57/0.54 ms vs 0.50 ms free-running with L2 prefetch), so lockstep is off by default
  int lock_every = 0;
  if (const char* e = getenv("SB200_LOCKSTEP")) lock_every = atoi(e);
  if (lock_every < 0) lock_every = 0;
  if (bp->S > 1024) lock_every = 0;
  a.lock_every = lock_every;
  a.lock_counters = reinterpret_cast<unsigned int*>(static_cast<unsigned char*>(m->d_ws) + 16 + 4 * 1024 + 8 * 1024);
  if (lock_every > 0 && static_cast<size_t>(bp->S) * 4 > m->ws_bytes - (16 + 4 * 1024 + 8 * 1024)) a.lock_every = 0;
  void (*const kern)(ScatterArgs) = d_mean ? band_var_kernel : d_v ? band_scatter_kernel<true> : band_scatter_kernel<false>;
  SB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(kern), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  if (a.lock_every > 0) {
    // a soft barrier between CTAs is only safe if they are all resident: ask the driver to guarantee it
    SB_CUDA(cudaMemsetAsync(a.lock_counters, 0, sizeof(unsigned int) * bp->S, m->stream));
    a.cluster = 1;
    void* params[] = {&a};
    cudaError_t e = cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(kern), dim3(grid), dim3(BAND_THREADS), params, smem, m->stream);
    if (e == cudaErrorCooperativeLaunchTooLarge || e == cudaErrorNotSupported || e == cudaErrorLaunchOutOfResources) {
      cudaGetLastError();
      a.lock_every = 0;  // fall back to free-running CTAs
    } else {
      SB_CUDA(e);
      count_launch();
      return SB200_OK;
    }
  }
  // clusters of adjacent bands: every CTA of a cluster must walk the same number of chunks, i.e. be in
  // the same split in every round => cluster size divides the band count and the grid
  // measured (profiles/r01): a cluster barrier per chunk does cut HBM traffic but costs far more than it
  // saves (C2 rowSums 0.52 ms free-running, 0.71 ms with clusters of 2, 1.17 ms with clusters of 4) => off
  int cluster = 1;
  if (const char* e = getenv("SB200_SCATTER_CLUSTER")) cluster = atoi(e);
  while (cluster > 1 && (bp->nb % cluster != 0 || grid % cluster != 0)) cluster >>= 1;
  if (cluster < 1) cluster = 1;
  a.cluster = cluster;
  if (cluster > 1) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(BAND_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = m->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cluster;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, a);
    if (e == cudaSuccess) {
      count_launch();
      return SB200_OK;
    }
    cudaGetLastError();  // cluster launch not possible with this footprint: free-running CTAs
    a.cluster = 1;
  }
  kern<<<grid, BAND_THREADS, smem, m->stream>>>(a);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return SB200_OK;
}

int launch_band_scatter(sb200_matrix* m, const double* d_v, double* d_out) { return launch_band_scatter_impl(m, d_v, nullptr, d_out); }

int launch_band_var(sb200_matrix* m, const double* d_mean, double* d_S, const int32_t** d_rowptr) {
  SB_TRY(launch_band_scatter_impl(m, nullptr, d_mean, d_S));
  *d_rowptr = m->plan_scatter->d_rowptr;  // kept with the plan: the row counts are its differences
  return SB200_OK;
}

// ================================================================================================
// A^T v with the operand in shared memory (banded gather)
// ================================================================================================
// sweep_kernel<SPMV_T> gathers v[i[k]] from L2, one 8-byte request per entry: its ceiling is the L2 request rate
// (245 G gathers/s measured = 0.41 ms per 1e8 entries), a third of what HBM would allow.  Here a CTA (row band,
// column split) keeps v's slice of its band in shared memory and walks the band's run of every column of its
// split: the gathers become LDS, HBM sees i and x once (plus band pointers) and 8 bytes per (column, band) of
// partial results (REDs at L2, or plain stores when one band covers all rows).
//   A warp takes 32 columns (one run descriptor per lane) and sums them G lanes per column, 32/G columns at a
//   time, G picked per 32 columns from their mean run length (2, 8 or 32): the lanes of a group stride over
//   the run (so a load instruction covers 32/G contiguous pieces), fold with shuffles, and the group's first
//   lane stores.  Two rounds of loads are in flight per warp.  Runs much longer than their group are summed by
//   the whole warp first.  No shared-memory atomics, no per-entry index lists.
constexpr int GA_THREADS = 768;
constexpr int GA_WARPS = GA_THREADS / 32;
constexpr int GA_U = 4;      // loads per lane and round
constexpr int GATHER_ROWS_CAP = (216 * 1024) / 8;  // 27648 rows of v per band

struct GatherArgs {
  BandView bv;
  const double* v;
  double* out;
  int max_rows;
};

template <int G>
__device__ __forceinline__ void gather_rounds(const BandView& bv, const double* __restrict__ vs, int32_t row0, int32_t s,
                                              int32_t len, double extra, bool any, int lane, int64_t cg, int64_t c_hi,
                                              double* __restrict__ out) {
  constexpr int CPR = 32 / G;  // columns per round
  const int sub = lane % G, grp = lane / G;
#pragma unroll 1
  for (int r = 0; r < G; r += 2) {  // two rounds per step: their loads are issued together
    int32_t ks[2], ke[2];
    double part[2] = {0.0, 0.0};
#pragma unroll
    for (int w = 0; w < 2; ++w) {
      const int col = (r + w) * CPR + grp;
      ks[w] = __shfl_sync(0xffffffffu, s, col & 31);
      ke[w] = ks[w] + __shfl_sync(0xffffffffu, len, col & 31);
      if (G == 1 || r + w >= G) ke[w] = ks[w];
    }
    int32_t k0[2] = {ks[0] + sub, ks[1] + sub};
    while (__any_sync(0xffffffffu, k0[0] < ke[0] || k0[1] < ke[1])) {
      int32_t rr[2][GA_U];
      double xx[2][GA_U];
#pragma unroll
      for (int w = 0; w < 2; ++w)
#pragma unroll
        for (int t = 0; t < GA_U; ++t) {
          const int32_t k = k0[w] + t * G;
          rr[w][t] = -1;
          xx[w][t] = 0.0;
          if (k < ke[w]) {
            rr[w][t] = ptx::ld_stream_s32(bv.i + k) - row0;
            xx[w][t] = ptx::ld_stream_f64(bv.x + k);
          }
        }
#pragma unroll
      for (int w = 0; w < 2; ++w)
#pragma unroll
        for (int t = 0; t < GA_U; ++t)
          if (rr[w][t] >= 0) part[w] = __dadd_rn(part[w], __dmul_rn(xx[w][t], vs[rr[w][t]]));  // idle lanes add nothing (no 0 * Inf)
      k0[0] += G * GA_U;
      k0[1] += G * GA_U;
    }
#pragma unroll
    for (int w = 0; w < 2; ++w) {
#pragma unroll
      for (int off = G / 2; off > 0; off >>= 1) part[w] = __dadd_rn(part[w], __shfl_xor_sync(0xffffffffu, part[w], off));
      const int col = ((r + w) * CPR + grp) & 31;
      const double total = __dadd_rn(part[w], __shfl_sync(0xffffffffu, extra, col));  // + the run the whole warp summed
      const bool some = __shfl_sync(0xffffffffu, any ? 1 : 0, col) != 0;
      const int64_t c = cg + (r + w) * CPR + grp;
      if (sub == 0 && r + w < G && c < c_hi) {
        if (bv.nb == 1)
          out[c] = total;  // one band holds every row: the only contribution to this column (0 for an empty one)
        else if (some)
          ptx::red_add_f64(out + c, total);
      }
    }
  }
}

__global__ void __launch_bounds__(GA_THREADS, 1) band_gather_kernel(const GatherArgs a) {
  extern __shared__ __align__(16) unsigned char gsm[];
  const BandView& bv = a.bv;
  double* vs = reinterpret_cast<double*>(gsm);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int units = bv.nb * bv.S;
  for (int u = blockIdx.x; u < units; u += gridDim.x) {
    const int h = u / bv.nb, b = u % bv.nb;
    const int32_t row0 = bv.rb[b];
    const int32_t R = bv.rb[b + 1] - row0;
    const int64_t c_lo = bv.cs[h], c_hi = bv.cs[h + 1];
    __syncthreads();  // the previous unit's readers are done with vs
    for (int r = tid; r < R; r += GA_THREADS) vs[r] = __ldg(a.v + row0 + r);
    __syncthreads();
    // descriptors one group ahead
    int32_t ns = 0, ne = 0;
    {
      const int64_t c = c_lo + warp * 32 + lane;
      if (c < c_hi && R > 0) {
        ns = band_start(bv, b, c);
        ne = band_start(bv, b + 1, c);
      }
    }
    for (int64_t cg = c_lo + warp * 32; cg < c_hi; cg += GA_WARPS * 32) {
      const int64_t c = cg + lane;
      const int32_t s = ns;
      int32_t len = ne - ns;
      ns = ne = 0;
      {
        const int64_t cn = c + GA_WARPS * 32;
        if (cn < c_hi && R > 0) {
          ns = band_start(bv, b, cn);
          ne = band_start(bv, b + 1, cn);
        }
      }
      int32_t total = len;
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) total += __shfl_xor_sync(0xffffffffu, total, off);
      if (total == 0) {
        if (bv.nb == 1 && c < c_hi) a.out[c] = 0.0;
        continue;
      }
      const bool any = len > 0;
      const int mean = total >> 5;
      const int32_t long_len = mean <= 6 ? 64 : (mean <= 48 ? 256 : 0x7fffffff);  // far beyond the group's reach
      // ---- runs much longer than the rest: the whole warp on one run ----
      double extra = 0.0;
      unsigned longmask = __ballot_sync(0xffffffffu, len >= long_len);
      while (longmask) {
        const int src = __ffs(longmask) - 1;
        longmask &= longmask - 1;
        const int32_t rs = __shfl_sync(0xffffffffu, s, src);
        const int32_t re = rs + __shfl_sync(0xffffffffu, len, src);
        double part = 0.0;
        for (int32_t k0 = rs; k0 < re; k0 += 32 * GA_U) {
          int32_t rr[GA_U];
          double xx[GA_U];
#pragma unroll
          for (int t = 0; t < GA_U; ++t) {
            const int32_t k = k0 + t * 32 + lane;
            rr[t] = -1;
            xx[t] = 0.0;
            if (k < re) {
              rr[t] = ptx::ld_stream_s32(bv.i + k) - row0;
              xx[t] = ptx::ld_stream_f64(bv.x + k);
            }
          }
#pragma unroll
          for (int t = 0; t < GA_U; ++t)
            if (rr[t] >= 0) part = __dadd_rn(part, __dmul_rn(xx[t], vs[rr[t]]));
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) part = __dadd_rn(part, __shfl_xor_sync(0xffffffffu, part, off));
        if (lane == src) {
          extra = part;
          len = 0;  // the rounds below skip it and add `extra` when they store the column
        }
      }
      __syncwarp();
      if (mean <= 6)
        gather_rounds<2>(bv, vs, row0, s, len, extra, any, lane, cg, c_hi, a.out);
      else if (mean <= 48)
        gather_rounds<8>(bv, vs, row0, s, len, extra, any, lane, cg, c_hi, a.out);
      else
        gather_rounds<32>(bv, vs, row0, s, len, extra, any, lane, cg, c_hi, a.out);
    }
  }
}

// Opt-in (SB200_GATHER_PLAN=1), parity-tested, NOT the default: measured on B200 against sweep_kernel<SPMV_T>
// (L2 gathers) it is 0.50 vs 0.495 ms at C2, 5.25 vs 5.03 ms at C3, 14.8 vs 9.5 ms at C4.  The gathers do become
// LDS and DRAM traffic is the algorithmic 1.25 GB at C2, but the runs are fetched with register loads — at most
// ~70 KB in flight per SM, and only in bursts — where the TMA-staged sweep keeps ~200 KB in flight; the kernel is
// latency-bound (ncu: long_scoreboard 8.6 warps per issue, issue-active 33 %).  The next step is to stage the
// runs with cp.async.bulk like the sweep does (profiles/r01/README.md).
int decide_gather_path(sb200_matrix* m) {
  if (m->gather_path >= 0) return SB200_OK;
  int path = 0;
  if (const char* e = getenv("SB200_GATHER_PLAN")) path = (e[0] != '0' && m->nnz > 0 && m->nrow > 0 && m->ncol > 0) ? 1 : 0;
  m->gather_path = path;
  return SB200_OK;
}

int launch_band_gather(sb200_matrix* m, const double* d_v, double* d_out) {
  if (!m->plan_gather) {
    int64_t nb = (static_cast<int64_t>(m->nrow) + static_cast<int64_t>(0.9 * GATHER_ROWS_CAP) - 1) /
                 static_cast<int64_t>(0.9 * GATHER_ROWS_CAP);
    if (nb < 1) nb = 1;
    if (nb > 4096) return fail(SB200_E_UNSUPPORTED, "banded gather: too many row bands");
    int S = static_cast<int>((2 * m->sm_count + nb - 1) / nb);  // two units per SM
    if (S < 1) S = 1;
    if (S > 1024) S = 1024;
    SB_TRY(build_band_plan(m, GATHER_ROWS_CAP, static_cast<int>(nb), S, &m->plan_gather));
  }
  const BandPlan* bp = m->plan_gather;
  GatherArgs a;
  a.bv = make_view(m, bp);
  a.v = d_v;
  a.out = d_out;
  a.max_rows = (bp->max_rows > 0 ? (bp->max_rows + 1) & ~1 : 2);
  if (bp->nb > 1) SB_CUDA(cudaMemsetAsync(d_out, 0, sizeof(double) * static_cast<size_t>(m->ncol), m->stream));
  const size_t smem = sizeof(double) * static_cast<size_t>(a.max_rows);
  int ctas = static_cast<int>((220 * 1024) / (smem + 1024));
  if (ctas > 2) ctas = 2;
  if (ctas < 1) ctas = 1;
  int grid = m->sm_count * ctas;
  if (grid > bp->nb * bp->S) grid = bp->nb * bp->S;
  SB_CUDA(cudaFuncSetAttribute(band_gather_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  band_gather_kernel<<<grid, GA_THREADS, smem, m->stream>>>(a);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return SB200_OK;
}

// ---- transpose: the banded two-pass placement kernel (the plan and the entry point live in transpose.cu) ---------
int launch_transpose_banded(sb200_matrix* m, const BandPlan* bp, int32_t* d_i_out, double* d_x_out) {
  cudaStream_t st = m->stream;
  TransposeArgs a;
  a.bv = make_view(m, bp);
  a.off = bp->d_off;
  a.i_out = d_i_out;
  a.x_out = d_x_out;
  a.max_rows = (bp->max_rows + 1) & ~1;
  const size_t smem = transpose_smem_bytes(a.max_rows);
  int ctas = smem <= 100 * 1024 ? 2 : 1;
  int grid = m->sm_count * ctas;
  if (grid > bp->nb * bp->S) grid = bp->nb * bp->S;
  SB_CUDA(cudaFuncSetAttribute(band_transpose_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  a.cluster = 1;  // clusters of adjacent bands in lockstep were measured (profiles/r01): no gain
  band_transpose_kernel<<<grid, BAND_THREADS, smem, st>>>(a);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return SB200_OK;
}

void free_matrix_plans(sb200_matrix* m, cudaStream_t s) {
  if (m->plan_scatter) {
    free_band_plan(m->plan_scatter, s);
    m->plan_scatter = nullptr;
  }
  if (m->plan_gather) {
    free_band_plan(m->plan_gather, s);
    m->plan_gather = nullptr;
  }
  if (m->plan_transpose) {
    free_band_plan(m->plan_transpose, s);
    m->plan_transpose = nullptr;
  }
  if (m->plan_split) {
    free_split_plan(m->plan_split, s);
    m->plan_split = nullptr;
  }
}

}  // namespace sb200
