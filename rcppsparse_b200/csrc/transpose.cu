// CSC -> CSR transpose: the entry point, the cached band plan, and the chunk-sorting placement kernel.
//
// Replaces Matrix::transpose() of the reference (zdebruine/RcppSparse, RcppSparse.h:375-385), whose arithmetic is
// R's Matrix::t — a serial counting sort by row.  Result: canonical CSC of A^T (p'[nrow+1], i' = source column ids
// ascending inside every new column, x' the same bits permuted).  No floating-point arithmetic.
//
// Plan (bands.cu, structure only, kept on the handle between calls): per-split row histogram -> look-back scan ->
// p' and per-(row, split) offsets; row bands of <= 384 rows holding ~equal numbers of entries; band pointers
// (where every column's run inside a band starts).
//
// Placement (transpose_place_kernel).  A CTA owns (row band, column split) units, handed out through an atomic
// counter, heaviest work first come first served.  Its output rows are its own, so the only ordering problem is
// inside the CTA: entries of one output row must appear in source-column order.  The CTA walks its columns in
// chunks; one chunk's runs, concatenated in column order, are placed at most E = 2048 entries at a time ("flat" order = final order
// inside every row).  Per chunk:
//   1. every lane expands its own runs into the flat list (entry index, column) — one shared-memory store per
//      entry, no per-entry search;
//   2. count: the flat list is cut into one contiguous piece per warp; 32 consecutive slots = consecutive entries
//      of a run, so the row loads coalesce; counts per (warp, row) in shared memory;
//   3. a per-row scan over the warps gives every warp its ordered slot range inside the row's chunk segment, a
//      block scan over the rows lays the segments out back to back in a shared-memory IMAGE of the chunk's output;
//   4. place: the same walk again; equal rows inside a 32-entry step are ranked with match.any in lane (= column)
//      order; column id and row go to the image with plain shared-memory stores, the value with an 8-byte
//      cp.async straight from global memory into its image slot (no register round trip, 16 in flight per thread);
//   5. flush: the image is copied out linearly — consecutive image slots of a row are consecutive global slots,
//      so a row's chunk segment leaves as full 32-byte sectors (round 1 stored 4 + 8 bytes per entry to global,
//      two partial-sector requests each; that was 19 of its 35 ms at C3).
// Bit-exact by construction for any band count, split count and chunk size (tests force many combinations).
//
// Roofline: HBM, 24N + 4(n+1) + 4(m+1) algorithmic bytes; the kernel also reads two band pointers per run.
// Tall matrices (mean run per column and 384-row band below ~2 entries) keep round 1's banded two-pass kernel
// with 2432-row bands (bands.cu) for now.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "bandplan.cuh"
#include "common.cuh"
#include "ptx.cuh"

namespace sb200 {

namespace {

constexpr int PL_ROWS_CAP = 384;  // rows per band
constexpr int PL_KMAX = 4;        // columns per thread and chunk, at most (counter / match.any kernel)
constexpr int PB_KMAX = 2;        // same, bitmap-rank kernel (its bitmap has THREADS * K bits per row)

struct PlaceArgs {
  BandView bv;
  const int32_t* off;  // [nrow*S (+1)] first output slot of (row r, split h): off[r*S + h]
  int32_t* i_out;
  double* x_out;
  int max_rows;  // capacity of the per-row tables (even, >= rows of the widest band)
  int kcols;     // columns per thread and chunk (1..PL_KMAX)
  unsigned int* unit_counter;  // zeroed before the launch
  int prefetch;  // pull the next chunk's runs towards L2 while this one is placed
  int carry;     // bitmap-rank kernel: only full rounds of E entries; what a window leaves over opens the next window
};

template <int THREADS, int E>
struct PlGeom {
  static constexpr int W = THREADS / 32;
  static size_t smem_bytes(int max_rows) {
    const size_t MR = static_cast<size_t>(max_rows);
    return static_cast<size_t>(E) * (8 + 4 + 4 + 2 + 2 + 2) + MR * 4 * 3 + 16 + static_cast<size_t>(W) * MR * 4 + 64;
  }
};

__device__ __forceinline__ void cp_async_8(void* dst_smem, const void* src_gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(ptx::smem_addr(dst_smem)), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

template <int THREADS, int E>
__global__ void __launch_bounds__(THREADS, (E <= 2048) ? 3 : 2) transpose_place_kernel(const PlaceArgs a) {
  constexpr int W = THREADS / 32;
  constexpr int U = 4;
  extern __shared__ __align__(16) unsigned char psm[];
  __shared__ uint32_t wsum[2][W];  // flat entries of each warp's columns, double-buffered by chunk parity
  __shared__ uint32_t wscan[W];    // row-scan partials
  __shared__ int s_unit;

  const BandView& bv = a.bv;
  const int MR = a.max_rows, K = a.kcols;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;

  double* img_x = reinterpret_cast<double*>(psm);                  // [E] the chunk's output image: values,
  int32_t* img_i = reinterpret_cast<int32_t*>(img_x + E);          // [E] column ids,
  int32_t* flat_k = img_i + E;                                     // [E] entry index of every flat slot
  uint32_t* cursor = reinterpret_cast<uint32_t*>(flat_k + E);      // [MR] next free global slot of each row
  uint32_t* imgbase = cursor + MR;                                 // [MR] where the row's segment starts in the image
  int32_t* delta = reinterpret_cast<int32_t*>(imgbase + MR);       // [MR] global slot - image slot
  uint32_t* cntw = reinterpret_cast<uint32_t*>(delta + MR) + 4;    // [W*MR/2] u16 pairs: entries of (warp, row)
  uint16_t* cnt16 = reinterpret_cast<uint16_t*>(cntw);
  uint16_t* rel = reinterpret_cast<uint16_t*>(cntw + (W * MR) / 2);  // [W*MR] running offset of (warp, row)
  uint16_t* img_r = rel + static_cast<size_t>(W) * MR;             // [E] and rows (to find a slot's global address)
  uint16_t* flat_c = img_r + E;                                    // [E] column inside the chunk
  uint16_t* flat_r = flat_c + E;                                   // [E] row inside the band (filled by the count pass)

  const int units = bv.nb * bv.S;
  const int CC = THREADS * K;        // columns per chunk
  const int IT = (MR + THREADS - 1) / THREADS;  // rows per thread in the row scan (contiguous)
  int chunk_no = 0;

  for (;;) {
    __syncthreads();  // the previous unit's last flush is done
    if (tid == 0) s_unit = static_cast<int>(atomicAdd(a.unit_counter, 1u));
    __syncthreads();
    const int u = s_unit;
    if (u >= units) break;
    const int h = u / bv.nb, b = u % bv.nb;  // consecutive units = neighbouring bands of one split: they read
    const int32_t row0 = bv.rb[b];           // neighbouring runs of the same columns at about the same time
    const int R = bv.rb[b + 1] - row0;
    const int32_t c_lo = bv.cs[h], c_hi = bv.cs[h + 1];
    if (R <= 0 || c_lo >= c_hi) continue;
    for (int r = tid; r < R; r += THREADS) cursor[r] = static_cast<uint32_t>(a.off[static_cast<int64_t>(row0 + r) * bv.S + h]);
    for (int e = tid; e < (W * MR) / 2; e += THREADS) cntw[e] = 0u;

    int32_t ns[PL_KMAX], ne[PL_KMAX];
#pragma unroll
    for (int kk = 0; kk < PL_KMAX; ++kk) {
      ns[kk] = ne[kk] = 0;
      const int64_t c = static_cast<int64_t>(c_lo) + (warp * K + kk) * 32 + lane;
      if (kk < K && c < c_hi) {
        ns[kk] = band_start(bv, b, c);
        ne[kk] = band_start(bv, b + 1, c);
      }
    }
    for (int64_t cbase = c_lo; cbase < c_hi; cbase += CC, ++chunk_no) {
      // ---- this chunk's runs; flat offsets inside the warp ---------------------------------------------------
      int32_t rs[PL_KMAX], rl[PL_KMAX];
      uint32_t ex[PL_KMAX];
      uint32_t wtot = 0;
#pragma unroll
      for (int kk = 0; kk < PL_KMAX; ++kk) {
        rs[kk] = ns[kk];
        rl[kk] = ne[kk] - ns[kk];
        uint32_t incl = static_cast<uint32_t>(rl[kk]);
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
          const uint32_t up = __shfl_up_sync(0xffffffffu, incl, off);
          if (lane >= off) incl += up;
        }
        ex[kk] = wtot + incl - static_cast<uint32_t>(rl[kk]);
        wtot += __shfl_sync(0xffffffffu, incl, 31);
      }
      // next chunk's descriptors, and its runs on their way to L2
#pragma unroll
      for (int kk = 0; kk < PL_KMAX; ++kk) {
        ns[kk] = ne[kk] = 0;
        const int64_t c = cbase + CC + (warp * K + kk) * 32 + lane;
        if (kk < K && c < c_hi) {
          ns[kk] = band_start(bv, b, c);
          ne[kk] = band_start(bv, b + 1, c);
          if (a.prefetch) {
            for (int32_t k = ns[kk] & ~31; k < ne[kk]; k += 32) ptx::prefetch_l2(bv.i + k);
            for (int32_t k = ns[kk] & ~15; k < ne[kk]; k += 16) ptx::prefetch_l2(bv.x + k);
          }
        }
      }
      const int par = chunk_no & 1;
      if (lane == 0) wsum[par][warp] = wtot;
      __syncthreads();
      uint32_t woff = 0, total = 0;
#pragma unroll
      for (int w = 0; w < W; ++w) {
        const uint32_t v = wsum[par][w];
        if (w < warp) woff += v;
        total += v;
      }
      const int32_t col0 = static_cast<int32_t>(cbase);
      for (uint32_t lo = 0; lo < total; lo += E) {  // one round unless the chunk holds more than E entries
        const uint32_t hi = (lo + E < total) ? lo + E : total;
        const uint32_t n = hi - lo;
        // ---- 1. owner expansion of the flat slots [lo, hi) --------------------------------------------------
#pragma unroll
        for (int kk = 0; kk < PL_KMAX; ++kk) {
          if (kk < K && rl[kk] > 0) {
            const uint32_t q0 = woff + ex[kk];
            const uint32_t q1 = q0 + static_cast<uint32_t>(rl[kk]);
            const uint32_t f0 = q0 > lo ? q0 : lo, f1 = q1 < hi ? q1 : hi;
            const uint16_t cc = static_cast<uint16_t>((warp * K + kk) * 32 + lane);
            for (uint32_t q = f0; q < f1; ++q) {
              flat_k[q - lo] = rs[kk] + static_cast<int32_t>(q - q0);
              flat_c[q - lo] = cc;
            }
          }
        }
        __syncthreads();
        // ---- 2. count entries per (warp, row); the warp's piece of the flat list ------------------------------
        const uint32_t per = (((n + W - 1) / W) + 31u) & ~31u;
        const uint32_t wlo = (warp * per < n) ? warp * per : n;
        const uint32_t whi = (wlo + per < n) ? wlo + per : n;
        for (uint32_t q0 = wlo; q0 < whi; q0 += 32 * U) {
          int32_t rr[U];
#pragma unroll
          for (int t = 0; t < U; ++t) {
            const uint32_t q = q0 + t * 32 + lane;
            rr[t] = (q < whi) ? ptx::ld_stream_s32(bv.i + flat_k[q]) - row0 : -1;
          }
#pragma unroll
          for (int t = 0; t < U; ++t) {
            const uint32_t q = q0 + t * 32 + lane;
            if (rr[t] >= 0) {
              flat_r[q] = static_cast<uint16_t>(rr[t]);
              const int idx = warp * MR + rr[t];
              atomicAdd(&cntw[idx >> 1], 1u << ((idx & 1) * 16));
            }
          }
        }
        __syncthreads();
        // ---- 3. per row: slot ranges of the warps in warp (= column) order; image layout; cursors ----------------
        uint32_t tot[2] = {0u, 0u};
        for (int it = 0; it < IT && it < 2; ++it) {
          const int r = tid * IT + it;
          if (r < R) {
            uint32_t run = 0;
#pragma unroll
            for (int w = 0; w < W; ++w) {
              const uint32_t c = cnt16[w * MR + r];
              rel[w * MR + r] = static_cast<uint16_t>(run);
              cnt16[w * MR + r] = 0;
              run += c;
            }
            tot[it] = run;
          }
        }
        const uint32_t tsum = tot[0] + tot[1];
        uint32_t incl = tsum;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
          const uint32_t up = __shfl_up_sync(0xffffffffu, incl, off);
          if (lane >= off) incl += up;
        }
        if (lane == 31) wscan[warp] = incl;
        __syncthreads();
        uint32_t base = incl - tsum;
#pragma unroll
        for (int w = 0; w < W; ++w)
          if (w < warp) base += wscan[w];
        for (int it = 0; it < IT && it < 2; ++it) {
          const int r = tid * IT + it;
          if (r < R) {
            imgbase[r] = base;
            const uint32_t cur = cursor[r];
            delta[r] = static_cast<int32_t>(cur - base);
            cursor[r] = cur + tot[it];
            base += tot[it];
          }
        }
        __syncthreads();
        // ---- 4. place into the image: equal rows inside a step ranked in lane (= column) order -------------------
        for (uint32_t q0 = wlo; q0 < whi; q0 += 32) {
          const uint32_t q = q0 + lane;
          const bool valid = q < whi;
          const int r = valid ? static_cast<int>(flat_r[q]) : -1 - lane;
          const unsigned same = __match_any_sync(0xffffffffu, r);
          if (valid) {
            const int idx = warp * MR + r;
            const uint32_t my = rel[idx];
            const uint32_t pos = imgbase[r] + my + __popc(same & lt_mask);
            img_i[pos] = col0 + flat_c[q];
            img_r[pos] = static_cast<uint16_t>(r);
            cp_async_8(img_x + pos, bv.x + flat_k[q]);
            if ((same >> lane) == 1u) rel[idx] = static_cast<uint16_t>(my + __popc(same));  // highest lane of the group
          }
          __syncwarp();
        }
        cp_async_wait_all();
        __syncthreads();
        // ---- 5. flush: consecutive image slots of a row are consecutive global slots ---------------------------
        for (uint32_t p = tid; p < n; p += THREADS) {
          const int r = img_r[p];
          const int64_t gp = static_cast<int64_t>(delta[r]) + p;
          a.i_out[gp] = img_i[p];
          a.x_out[gp] = img_x[p];
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// Placement with bitmap ranks (default).  Same chunks, same image, same flush — but the position of an entry inside
// its row's chunk segment comes from a row-major BITMAP of the chunk (one bit per (row, column of the chunk)):
//   count   thread per flat slot (consecutive threads = consecutive entries of a run: coalesced row loads); the
//           entry sets its bit with one shared-memory atomic OR; row, column and entry index stay in registers;
//   layout  per row: prefix popcounts of its bitmap words; block scan over the rows -> image layout, cursors;
//   place   rank = prefix[word] + popc(word & bits below my column): a (row, column) pair is unique in a dgCMatrix,
//           so the rank IS the number of the row's entries in earlier columns — no ordering between threads or
//           warps, no per-warp counters, no match.any.
// ncu on the counter/match version above (C3 at 0.1 scale): 171 thread instructions per entry, issue-bound at 28 %.
// ------------------------------------------------------------------------------------------------------------
template <int THREADS, int E>
struct PlGeomB {
  static size_t smem_bytes(int max_rows, int words) {
    const size_t MR = static_cast<size_t>(max_rows);
    return static_cast<size_t>(E) * (8 + 4 + 4 + 2 + 2) + MR * 4 * 3 + 16 + MR * static_cast<size_t>(words) * 6 + 64;
  }
};

// KC = columns per thread and window (1 or 2), a template argument so that the bitmap's row stride (WW words) and the
// per-column loops are compile-time (ncu: the index arithmetic around the bitmap was 22 of 240 thread instructions per entry)
template <int THREADS, int E, int KC>
__global__ void __launch_bounds__(THREADS, THREADS >= 512 ? 2 : (E <= 512 ? 6 : (E <= 1024 ? 4 : (E <= 2048 ? 3 : 2)))) transpose_bitrank_kernel(const PlaceArgs a) {
  constexpr int W = THREADS / 32;
  constexpr int EPT = E / THREADS;  // flat slots per thread and round
  static_assert(EPT * THREADS == E, "E must be a multiple of the block size");
  extern __shared__ __align__(16) unsigned char psm[];
  __shared__ uint32_t wsum[2][W];
  __shared__ uint32_t wscan[W];
  __shared__ int s_unit;
  __shared__ int64_t s_next_c[2];  // carry: first column of the next window (two copies, like wsum: a window without
  __shared__ int32_t s_next_k[2];  // entries has no barrier after these are read), and the first entry of that column's
                                   // run that is still to be placed (-1: the whole run)

  const BandView& bv = a.bv;
  const int MR = a.max_rows;
  constexpr int K = KC;
  constexpr int WW = (THREADS * K) / 32;  // bitmap words per row = columns per chunk / 32
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  double* img_x = reinterpret_cast<double*>(psm);                // [E] the chunk's output image: values,
  int32_t* img_i = reinterpret_cast<int32_t*>(img_x + E);        // [E] column ids,
  int32_t* flat_k = img_i + E;                                   // [E] entry index of every flat slot
  uint32_t* cursor = reinterpret_cast<uint32_t*>(flat_k + E);    // [MR] next free global slot of each row
  uint32_t* imgbase = cursor + MR;                               // [MR] where the row's segment starts in the image
  int32_t* delta = reinterpret_cast<int32_t*>(imgbase + MR);     // [MR] global slot - image slot
  uint32_t* bm = reinterpret_cast<uint32_t*>(delta + MR) + 4;    // [MR*WW] bit c of row r: the chunk holds entry (r, c)
  uint16_t* pre = reinterpret_cast<uint16_t*>(bm + static_cast<size_t>(MR) * WW);  // [MR*WW] entries of the row in earlier words
  uint16_t* img_r = pre + static_cast<size_t>(MR) * WW;          // [E] rows (to find a slot's global address)
  uint16_t* flat_c = img_r + E;                                  // [E] column inside the chunk

  const int units = bv.nb * bv.S;
  constexpr int CC = THREADS * K;
  const int IT = (MR + THREADS - 1) / THREADS;
  int chunk_no = 0;

  for (;;) {
    __syncthreads();
    if (tid == 0) s_unit = static_cast<int>(atomicAdd(a.unit_counter, 1u));
    __syncthreads();
    const int u = s_unit;
    if (u >= units) break;
    const int h = u / bv.nb, b = u % bv.nb;
    const int32_t row0 = bv.rb[b];
    const int R = bv.rb[b + 1] - row0;
    const int32_t c_lo = bv.cs[h], c_hi = bv.cs[h + 1];
    if (R <= 0 || c_lo >= c_hi) continue;
    for (int r = tid; r < R; r += THREADS) cursor[r] = static_cast<uint32_t>(a.off[static_cast<int64_t>(row0 + r) * bv.S + h]);

    int32_t ns[KC], ne[KC];
#pragma unroll
    for (int kk = 0; kk < KC; ++kk) {
      ns[kk] = ne[kk] = 0;
      const int64_t c = static_cast<int64_t>(c_lo) + (warp * K + kk) * 32 + lane;
      if (kk < K && c < c_hi) {
        ns[kk] = band_start(bv, b, c);
        ne[kk] = band_start(bv, b + 1, c);
      }
    }
    // A window is the next CC columns.  Without carry every window is placed whole, E entries a round, and the last
    // round of a window is as full as it happens to be (C3: 62 % on average, and a round costs the same whatever its
    // fill).  With carry a window that is not the unit's last one is placed in FULL rounds only: the columns it leaves
    // over — the first of them possibly from the middle of its run, rows are unique inside a column so a run may be cut
    // anywhere — open the next window.
    for (int64_t cbase = c_lo; cbase < c_hi; ++chunk_no) {
      int32_t rs[KC], rl[KC];
      uint32_t ex[KC];
      uint32_t wtot = 0;
#pragma unroll
      for (int kk = 0; kk < KC; ++kk) {
        rs[kk] = ns[kk];
        rl[kk] = ne[kk] - ns[kk];
        uint32_t incl = static_cast<uint32_t>(rl[kk]);
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
          const uint32_t up = __shfl_up_sync(0xffffffffu, incl, off);
          if (lane >= off) incl += up;
        }
        ex[kk] = wtot + incl - static_cast<uint32_t>(rl[kk]);
        wtot += __shfl_sync(0xffffffffu, incl, 31);
      }
      const int par = chunk_no & 1;
      if (lane == 0) wsum[par][warp] = wtot;
      if (tid == 0) {
        s_next_c[par] = cbase + CC;
        s_next_k[par] = -1;
      }
      __syncthreads();
      uint32_t woff = 0, total = 0;
#pragma unroll
      for (int w = 0; w < W; ++w) {
        const uint32_t v = wsum[par][w];
        if (w < warp) woff += v;
        total += v;
      }
      const bool last_window = cbase + CC >= c_hi;
      const uint32_t limit = (a.carry && !last_window && total >= static_cast<uint32_t>(E)) ? (total / E) * E : total;
      if (limit < total) {  // the run that holds flat slot `limit` opens the next window
#pragma unroll
        for (int kk = 0; kk < KC; ++kk) {
          const uint32_t q0 = woff + ex[kk];
          if (kk < K && rl[kk] > 0 && q0 <= limit && limit < q0 + static_cast<uint32_t>(rl[kk])) {
            s_next_c[par] = cbase + (warp * K + kk) * 32 + lane;
            s_next_k[par] = rs[kk] + static_cast<int32_t>(limit - q0);
          }
        }
      }
      __syncthreads();
      const int64_t next_c = s_next_c[par];
      const int32_t next_k = s_next_k[par];
#pragma unroll
      for (int kk = 0; kk < KC; ++kk) {  // next window's descriptors
        ns[kk] = ne[kk] = 0;
        const int ci = (warp * K + kk) * 32 + lane;
        const int64_t c = next_c + ci;
        if (kk < K && c < c_hi) {
          ns[kk] = (ci == 0 && next_k >= 0) ? next_k : band_start(bv, b, c);
          ne[kk] = band_start(bv, b + 1, c);
        }
      }
      const int32_t col0 = static_cast<int32_t>(cbase);
      cbase = next_c;
      for (uint32_t lo = 0; lo < limit; lo += E) {
        const uint32_t hi = (lo + E < limit) ? lo + E : limit;
        const uint32_t n = hi - lo;
        // ---- clear the bitmap of the rows in use; owner expansion of the flat slots [lo, hi) -----------------------
        for (int e = tid; e < R * WW; e += THREADS) bm[e] = 0u;
#pragma unroll
        for (int kk = 0; kk < KC; ++kk) {
          if (kk < K && rl[kk] > 0) {
            const uint32_t q0 = woff + ex[kk];
            const uint32_t q1 = q0 + static_cast<uint32_t>(rl[kk]);
            const uint32_t f0 = q0 > lo ? q0 : lo, f1 = q1 < hi ? q1 : hi;
            const uint16_t cc = static_cast<uint16_t>((warp * K + kk) * 32 + lane);
            for (uint32_t q = f0; q < f1; ++q) {
              flat_k[q - lo] = rs[kk] + static_cast<int32_t>(q - q0);
              flat_c[q - lo] = cc;
            }
          }
        }
        __syncthreads();
        // ---- count: a thread per flat slot, everything about the entry stays in registers ----------------------------
        int32_t ek[EPT], er[EPT];
        uint32_t ec[EPT];
#pragma unroll
        for (int j = 0; j < EPT; ++j) {
          const uint32_t q = tid + j * THREADS;
          ek[j] = -1;
          er[j] = 0;
          ec[j] = 0;
          if (q < n) {
            ek[j] = flat_k[q];
            ec[j] = flat_c[q];
          }
        }
        const int used = static_cast<int>((n + THREADS - 1) / THREADS);  // slots per thread that hold anything (uniform)
#pragma unroll
        for (int j = 0; j < EPT; ++j) {
          if (j >= used) break;
          if (ek[j] >= 0) er[j] = ptx::ld_stream_s32(bv.i + ek[j]) - row0;
        }
#pragma unroll
        for (int j = 0; j < EPT; ++j) {
          if (j >= used) break;
          if (ek[j] >= 0) atomicOr(&bm[er[j] * WW + (ec[j] >> 5)], 1u << (ec[j] & 31u));
        }
        __syncthreads();
        // ---- layout: prefix popcounts per row, block scan over the rows, cursors ---------------------------------
        uint32_t tot[2] = {0u, 0u};
        for (int it = 0; it < IT && it < 2; ++it) {
          const int r = tid * IT + it;
          if (r < R) {
            uint32_t run = 0;
#pragma unroll
            for (int w = 0; w < WW; ++w) {
              pre[r * WW + w] = static_cast<uint16_t>(run);
              run += __popc(bm[r * WW + w]);
            }
            tot[it] = run;
          }
        }
        const uint32_t tsum = tot[0] + tot[1];
        uint32_t incl = tsum;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
          const uint32_t up = __shfl_up_sync(0xffffffffu, incl, off);
          if (lane >= off) incl += up;
        }
        if (lane == 31) wscan[warp] = incl;
        __syncthreads();
        uint32_t base = incl - tsum;
#pragma unroll
        for (int w = 0; w < W; ++w)
          if (w < warp) base += wscan[w];
        for (int it = 0; it < IT && it < 2; ++it) {
          const int r = tid * IT + it;
          if (r < R) {
            imgbase[r] = base;
            const uint32_t cur = cursor[r];
            delta[r] = static_cast<int32_t>(cur - base);
            cursor[r] = cur + tot[it];
            base += tot[it];
          }
        }
        __syncthreads();
        // ---- place: rank = entries of my row in earlier columns of the chunk -----------------------------------------
#pragma unroll
        for (int j = 0; j < EPT; ++j) {
          if (j >= used) break;
          if (ek[j] >= 0) {
            const int wi = er[j] * WW + static_cast<int>(ec[j] >> 5);
            const uint32_t below = bm[wi] & ((1u << (ec[j] & 31u)) - 1u);
            const uint32_t pos = imgbase[er[j]] + pre[wi] + __popc(below);
            img_i[pos] = col0 + static_cast<int32_t>(ec[j]);
            img_r[pos] = static_cast<uint16_t>(er[j]);
            cp_async_8(img_x + pos, bv.x + ek[j]);
          }
        }
        cp_async_wait_all();
        __syncthreads();
        // ---- flush: consecutive image slots of a row are consecutive global slots ----------------------------------
        for (uint32_t p = tid; p < n; p += THREADS) {
          const int r = img_r[p];
          const int64_t gp = static_cast<int64_t>(delta[r]) + p;
          a.i_out[gp] = img_i[p];
          a.x_out[gp] = img_x[p];
        }
      }
    }
  }
}

__global__ void zero_i32_kernel(int32_t* d, int64_t n) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; k < n; k += stride) d[k] = 0;
}

template <int THREADS, int E>
int launch_place(sb200_matrix* m, const BandPlan* bp, int32_t* d_i_out, double* d_x_out) {
  PlaceArgs a;
  a.bv = make_view(m, bp);
  a.off = bp->d_off;
  a.i_out = d_i_out;
  a.x_out = d_x_out;
  a.max_rows = (bp->max_rows + 1) & ~1;
  if (a.max_rows < 2) a.max_rows = 2;
  if (a.max_rows > 2 * THREADS) return fail(SB200_E_UNSUPPORTED, "transpose: a row band exceeds the row scan's reach");
  const char* rank = getenv("SB200_TRANSPOSE_RANK");
  const bool bitmap = !(rank && !strcmp(rank, "match"));
  const double mean_run = static_cast<double>(m->nnz) / (static_cast<double>(m->ncol > 0 ? m->ncol : 1) * bp->nb);
  int K = static_cast<int>(0.65 * E / (THREADS * (mean_run > 0.05 ? mean_run : 0.05)) + 0.5);
  if (K < 1) K = 1;
  if (K > PL_KMAX) K = PL_KMAX;
  if (const char* e = getenv("SB200_TRANSPOSE_KCOLS")) {
    const int v = atoi(e);
    if (v >= 1 && v <= PL_KMAX) K = v;
  }
  if (bitmap && K > 2) K = 2;  // the bitmap has THREADS * K bits per row
  a.kcols = K;
  a.prefetch = getenv("SB200_TRANSPOSE_PF") ? 1 : 0;  // measured: the L2 prefetch of the next chunk's runs costs more than it hides
  {
    const char* e = getenv("SB200_TRANSPOSE_CARRY");
    a.carry = (e && atoi(e) == 0) ? 0 : 1;
  }
  // the unit counter lives in the handle's workspace, behind the lockstep counters
  a.unit_counter = reinterpret_cast<unsigned int*>(static_cast<unsigned char*>(m->d_ws) + 16 + 4 * 1024 + 8 * 1024 + 2048);
  SB_CUDA(cudaMemsetAsync(a.unit_counter, 0, sizeof(unsigned int), m->stream));
  const size_t smem = bitmap ? PlGeomB<THREADS, E>::smem_bytes(a.max_rows, (THREADS * K) / 32) : PlGeom<THREADS, E>::smem_bytes(a.max_rows);
  int per_sm = static_cast<int>((224 * 1024) / (smem + 1024));
  if (per_sm > 2048 / THREADS) per_sm = 2048 / THREADS;
  if (per_sm > 6) per_sm = 6;
  if (per_sm < 1) per_sm = 1;
  int grid = m->sm_count * per_sm;
  if (grid > bp->nb * bp->S) grid = bp->nb * bp->S;
  if (bitmap) {
    auto kern = K == 1 ? transpose_bitrank_kernel<THREADS, E, 1> : transpose_bitrank_kernel<THREADS, E, 2>;
    SB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    kern<<<grid, THREADS, smem, m->stream>>>(a);
  } else {
    auto kern = transpose_place_kernel<THREADS, E>;
    SB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    kern<<<grid, THREADS, smem, m->stream>>>(a);
  }
  count_launch();
  SB_CUDA(cudaGetLastError());
  return SB200_OK;
}

}  // namespace

// kind: 1 = banded two-pass kernel of bands.cu (2432-row bands), 2 = chunk-sort placement (384-row bands),
// 3 = two stable stream splits (transpose_split.cu).  Tall matrices — too few entries per (column, 384-row band) for the
// chunk sort — take 3 when its tables fit, else 1.
static int transpose_kind(const sb200_matrix* m, bool allow_split = true) {
  if (const char* e = getenv("SB200_TRANSPOSE_PATH")) {
    if (!strcmp(e, "banded") || !strcmp(e, "1")) return 1;
    if (!strcmp(e, "place") || !strcmp(e, "2")) return 2;
    if ((!strcmp(e, "split") || !strcmp(e, "3")) && allow_split && split_transpose_fits(m)) return 3;
  }
  // Mean run of a column inside a 384-row band decides (measured, profiles/r02/opbench_crossover.jsonl): with runs of a
  // dozen entries and more (C3) the chunk sort's single pass wins; below that the two-split path does — by 1.3x at ~7
  // entries a run, 3x at ~2 — unless the matrix is so small that two more launches and their ~1000-key tables are what it costs.
  const double bands384 = static_cast<double>(m->nrow) / (0.9 * PL_ROWS_CAP) + 1.0;
  const double mean_run = static_cast<double>(m->nnz) / (static_cast<double>(m->ncol > 0 ? m->ncol : 1) * bands384);
  if (mean_run >= 12.0 || (m->nnz < 8000000 && mean_run >= 2.0)) return 2;
  if (m->nnz >= 4000000 && allow_split && split_transpose_fits(m)) return 3;  // 1e6 entries over 1e6 rows: 1.2 ms split, 0.33 banded
  return mean_run >= 2.0 ? 2 : 1;
}

int transpose_device(sb200_matrix* m, int32_t* d_p_out, int32_t* d_i_out, double* d_x_out) {
  cudaStream_t st = m->stream;
  const int32_t nrow = m->nrow;
  const int64_t nnz = m->nnz;
  if (nnz == 0 || nrow == 0) {
    int64_t blocks = (static_cast<int64_t>(nrow) + 1 + 255) / 256;
    if (blocks > 1024) blocks = 1024;
    zero_i32_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(d_p_out, static_cast<int64_t>(nrow) + 1);
    count_launch();
    SB_CUDA(cudaGetLastError());
    return SB200_OK;
  }
  PhaseTrace tr(st);
  tr.mark("start");
  int kind = transpose_kind(m);
  if (kind == 3) {
    const int rc3 = transpose_split_device(m, d_p_out, d_i_out, d_x_out);
    if (rc3 != SB200_E_NOMEM) return rc3;
    cudaGetLastError();  // no room for the tables or the record stream after all: the single-pass kernels need neither
    kind = transpose_kind(m, false);
  }
  int env_bands = 0, env_splits = 0;
  if (const char* e = getenv("SB200_TRANSPOSE_SPLITS")) env_splits = atoi(e);
  if (const char* e = getenv("SB200_TRANSPOSE_BANDS")) env_bands = atoi(e);
  // The plan depends on the structure only (p, i): it is kept on the handle and reused by later calls (and by
  // the row-ordered copy's build); dropped with the handle.
  if (m->plan_transpose && (m->plan_transpose->kind != kind || m->plan_transpose->env_bands != env_bands ||
                            m->plan_transpose->env_splits != env_splits)) {
    free_band_plan(m->plan_transpose, st);
    m->plan_transpose = nullptr;
  }
  const bool cached = m->plan_transpose != nullptr;
  if (!cached) {
    // chunk sort: many column splits — the units of one split run side by side (they are handed out in (split, band)
    // order), so neighbouring bands read their neighbouring runs of the same columns while the shared 32-byte sectors are
    // still in L2 (C3: 28.4 ms with 4 splits, 25.6 / 24.4 / 24.2 with 16 / 64 / 256)
    int S = kind == 2 ? 64 : 2;
    int bands = kind == 2 ? 2 * m->sm_count : m->sm_count;
    if (env_splits >= 1 && env_splits <= 1024) S = env_splits;
    if (env_bands >= 1) bands = env_bands;
    BandPlan* bp = nullptr;
    SB_TRY(build_band_plan(m, kind == 2 ? PL_ROWS_CAP : 2432, bands, S, &bp));
    bp->kind = kind;
    bp->env_bands = env_bands;
    bp->env_splits = env_splits;
    m->plan_transpose = bp;
  }
  const BandPlan* bp = m->plan_transpose;
  tr.mark("phase1");
  SB_CUDA(cudaMemcpyAsync(d_p_out, bp->d_rowptr, sizeof(int32_t) * (static_cast<size_t>(nrow) + 1), cudaMemcpyDeviceToDevice, st));
  int rc;
  if (kind == 2) {
    const char* cfg = getenv("SB200_TRANSPOSE_CFG");
    if (cfg && !strcmp(cfg, "512x3072"))
      rc = launch_place<512, 3072>(m, bp, d_i_out, d_x_out);
    else if (cfg && !strcmp(cfg, "256x4096"))
      rc = launch_place<256, 4096>(m, bp, d_i_out, d_x_out);
    else if (cfg && !strcmp(cfg, "256x1024"))
      rc = launch_place<256, 1024>(m, bp, d_i_out, d_x_out);
    else if (cfg && !strcmp(cfg, "256x512"))
      rc = launch_place<256, 512>(m, bp, d_i_out, d_x_out);
    else if (cfg && !strcmp(cfg, "512x2048"))
      rc = launch_place<512, 2048>(m, bp, d_i_out, d_x_out);
    else if (cfg && !strcmp(cfg, "256x2048"))
      rc = launch_place<256, 2048>(m, bp, d_i_out, d_x_out);
    // measured at C3 (profiles/r02), match.any ranks: 256x2048 (3 CTAs/SM) 26.5-27.8 ms, 256x4096 (2) 28.3-29.1, 128x2048 (4)
    // 31.1, 512x3072 29.4; bitmap ranks with carried windows: 256x2048 23.4-23.5, 256x1024 (4 CTAs/SM) 22.0, 512x2048 (2 CTAs
    // of 16 warps) 27.3.  The kernel waits on its gathers (ncu: long_scoreboard 4.6 warps per issue, 24 warps per SM): a
    // fourth CTA per SM is worth more than longer rounds.  Small matrices keep the geometry their crossover was measured with.
    else if (!cfg && m->nnz >= 8000000)
      rc = launch_place<256, 1024>(m, bp, d_i_out, d_x_out);
    else
      rc = launch_place<256, 2048>(m, bp, d_i_out, d_x_out);
  } else {
    rc = launch_transpose_banded(m, bp, d_i_out, d_x_out);
  }
  tr.mark("phase2");
  tr.report("transpose (%s, %s) nb=%d S=%d maxrows=%d:", cached ? "cached plan" : "plan built",
            kind == 2 ? "chunk-sort placement" : "banded two-pass", bp->nb, bp->S, bp->max_rows);
  return rc;
}

}  // namespace sb200
