// CSC -> CSR transpose of TALL matrices: two stable stream splits (tools/transpose_two_level_spec.py is the
// executable specification of the intermediate arrays).
//
// Replaces Matrix::transpose() of the reference (zdebruine/RcppSparse, RcppSparse.h:375-385; arithmetic = R's
// Matrix::t, a serial counting sort by row) where the chunk-sorting kernel of transpose.cu has nothing to chew on: a
// 1M-row matrix of density 1e-3 leaves 0.4 entries per (column, 384-row band), so a single pass can coalesce either
// its reads or its writes, never both.  Two passes, both with contiguous reads and short contiguous runs on the way out:
//
//   pass 1  the entry stream in storage (column-major) order is cut into tiles of 4096 entries; every tile is split,
//           stably, by ROW BAND (band = row >> sh, ~sqrt(nrow) rows each) and appends its piece of each band to that
//           band's stream of 16-byte records (value, source column, row inside the band).  Where the piece goes is
//           structure only: first slot of (tile, band) = exclusive scan over (band major, tile minor) of the per-tile
//           band counts — kept on the handle.
//   pass 2  a band's stream is cut into segments of 4 chunks; a CTA takes a segment, walks it 8192 records at a time and
//           splits each chunk, stably, by row; a row's piece is appended at the row's cursor (shared memory).  Where the
//           cursors of a segment start is structure only too: p'[row] + the row's records in the band's earlier segments
//           (counted once, on the first call, from the record stream pass 1 has just written; kept on the handle).
//
// Both passes are the same kernel (split_kernel<PASS>).  The stable split of a chunk: warp w owns the w-th contiguous
// 256 records; every lane learns which lanes of its 32-record step hold the same key (run heads inside one column in
// pass 1; a per-warp claim table otherwise — see the kernel); a table of counts per (warp, key) in shared memory — u16,
// written by a group's lowest lane only — carries the rank across the steps of a warp; one scan per key over the warps
// and one block scan over the keys lay the chunk out key-major in a shared-memory IMAGE; the image leaves linearly, so
// the records of one key are consecutive global stores.  Order inside a key = storage order in both passes => inside an
// output row = source column order: the canonical CSC of A^T bit for bit, no sort, no global atomics.  No
// floating-point arithmetic.  Both passes run one chunk ahead (next chunk's records in the registers the placement has
// freed, its cursors fetched, the chunk after that on its way to L2) while the image is flushed.
//
// Roofline: HBM.  Algorithmic bytes 24N + 4(n+1) + 4(m+1) (SURVEY 8d); this path moves 12N + 16N + 16N + 12N plus
// 4 bytes per (tile, band), so its ceiling is 0.43 of that roofline.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <vector>

#include "common.cuh"
#include "ptx.cuh"

namespace sb200 {

struct SplitPlan {
  int sh = 0;           // rows per band = 1 << sh
  int nb = 0;           // bands
  int te = 0;           // entries per tile
  int64_t ntiles = 0;
  int32_t* d_rowptr = nullptr;   // [nrow+1] p' of the result
  int32_t* d_tb = nullptr;       // [ntiles*nb] tile-major: first slot, in the band-major record stream, of (tile, band)
  int32_t* d_bstart = nullptr;   // [nb+1] where every band's stream starts
  int32_t* d_tilecol = nullptr;  // [ntiles+1] column holding the first entry of tile t
  int seg_chunks = 0;
  int nseg = 0;                  // pass-2 units: pieces of <= SP_SEG_CHUNKS chunks of one band's stream
  int32_t* d_seg = nullptr;      // [3*nseg] band, first record, end of every segment
  int32_t* d_segfirst = nullptr; // [nb+1] first segment of every band
  uint32_t* d_segcur = nullptr;  // [nseg << sh] where every row's cursor starts in a segment (filled on the first call)
  bool segcur_ready = false;
  unsigned int* d_counters = nullptr;  // [2] tickets of the two passes
  size_t bytes = 0;
};

namespace {

constexpr int SP_THREADS = 512;
constexpr int SP_TE = 4096;
constexpr int SP_SEG_CHUNKS = 4;  // chunks per pass-2 unit (SB200_SPLIT_SEG)
constexpr int SP_MAX_KEYS = 3072;  // bands, and rows per band: the (warp, key) table is 16 x keys x 2 bytes of shared memory

// One record of the band-major stream: value, source column, row inside the band — 16 bytes, so that a tile's piece of
// a band is ONE contiguous run (three arrays meant three partial-sector pieces per (tile, band): 72 M at C2, and the
// memory system takes ~50 G of those a second whatever the kernel does).
struct __align__(16) Rec {
  double x;
  int32_t c;
  uint32_t r;
};
__device__ __forceinline__ Rec ld_stream_rec(const Rec* p) {
  uint32_t a, b, c, d;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "l"(p));
  Rec r;
  r.x = __hiloint2double(static_cast<int>(b), static_cast<int>(a));
  r.c = static_cast<int32_t>(c);
  r.r = d;
  return r;
}
__device__ __forceinline__ void st_rec(Rec* p, double x, int32_t c, uint32_t r) {
  asm volatile("st.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(static_cast<uint32_t>(__double2loint(x))),
               "r"(static_cast<uint32_t>(__double2hiint(x))), "r"(static_cast<uint32_t>(c)), "r"(r)
               : "memory");
}


// ---- plan kernels -----------------------------------------------------------------------------------------------
// Hc[b * ntiles + t] = entries of tile t in band b;  rowcnt[r] += 1 per entry
__global__ void __launch_bounds__(SP_THREADS)
    split_hist_kernel(const int32_t* __restrict__ gi, int64_t nnz, int sh, int nb, int te, int64_t ntiles,
                      uint32_t* __restrict__ hc, uint32_t* __restrict__ rowcnt) {
  extern __shared__ uint32_t hist[];
  for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    for (int b = threadIdx.x; b < nb; b += SP_THREADS) hist[b] = 0u;
    __syncthreads();
    const int64_t k0 = t * te;
    const int n = static_cast<int>((nnz - k0 < te) ? nnz - k0 : te);
    for (int q = threadIdx.x; q < n; q += SP_THREADS) {
      const int32_t r = ptx::ld_stream_s32(gi + k0 + q);
      atomicAdd(&hist[r >> sh], 1u);
      ptx::red_add_u32(rowcnt + r, 1u);
    }
    __syncthreads();
    for (int b = threadIdx.x; b < nb; b += SP_THREADS) hc[static_cast<int64_t>(b) * ntiles + t] = hist[b];
    __syncthreads();
  }
}

// tb[t * nb + b] = scan[b * ntiles + t] (32 x 32 tiles through shared memory); bstart[b] = scan[b * ntiles]
__global__ void __launch_bounds__(256)
    split_table_kernel(const int32_t* __restrict__ scan, int nb, int64_t ntiles, int32_t nnz, int32_t* __restrict__ tb,
                       int32_t* __restrict__ bstart) {
  __shared__ int32_t tile[32][33];
  const int64_t t0 = static_cast<int64_t>(blockIdx.x) * 32;
  const int b0 = blockIdx.y * 32;
  const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;  // 32 x 8
  for (int j = ly; j < 32; j += 8) {
    const int b = b0 + j;
    const int64_t t = t0 + lx;
    if (b < nb && t < ntiles) tile[j][lx] = scan[static_cast<int64_t>(b) * ntiles + t];
  }
  __syncthreads();
  for (int j = ly; j < 32; j += 8) {
    const int64_t t = t0 + j;
    const int b = b0 + lx;
    if (b < nb && t < ntiles) tb[t * nb + b] = tile[lx][j];
  }
  if (blockIdx.x == 0 && ly == 0) {
    const int b = b0 + lx;
    if (b < nb) bstart[b] = scan[static_cast<int64_t>(b) * ntiles];
    if (b == nb - 1) bstart[nb] = nnz;
  }
}

// tilecol[t] = the column holding entry t * te (largest c < ncol with p[c] <= t * te)
__global__ void split_tilecol_kernel(const int32_t* __restrict__ gp, int32_t ncol, int64_t nnz, int te, int64_t ntiles,
                                     int32_t* __restrict__ tilecol) {
  const int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t > ntiles) return;
  int64_t k = t * te;
  if (k > nnz) k = nnz;
  int32_t lo = 0, hi = ncol - 1;
  while (lo < hi) {
    const int32_t mid = lo + ((hi - lo + 1) >> 1);
    if (gp[mid] <= k)
      lo = mid;
    else
      hi = mid - 1;
  }
  tilecol[t] = lo;
}

// h[(seg << sh) + r] = records of row r (inside its band) in segment seg of the record stream
__global__ void __launch_bounds__(SP_THREADS)
    split_seg_hist_kernel(const Rec* __restrict__ rec, const int32_t* __restrict__ seg, int nseg, int sh, uint32_t* __restrict__ h) {
  extern __shared__ uint32_t hist[];
  const int R = 1 << sh;
  for (int u = blockIdx.x; u < nseg; u += gridDim.x) {
    for (int r = threadIdx.x; r < R; r += SP_THREADS) hist[r] = 0u;
    __syncthreads();
    const int64_t k0 = seg[3 * u + 1], k1 = seg[3 * u + 2];
    for (int64_t k = k0 + threadIdx.x; k < k1; k += SP_THREADS) atomicAdd(&hist[rec[k].r], 1u);
    __syncthreads();
    for (int r = threadIdx.x; r < R; r += SP_THREADS) h[(static_cast<int64_t>(u) << sh) + r] = hist[r];
    __syncthreads();
  }
}

// counts -> cursors: per (band, row), p'[row] then the running sum over the band's segments
__global__ void split_seg_scan_kernel(uint32_t* __restrict__ h, const int32_t* __restrict__ segfirst, const int32_t* __restrict__ rowptr,
                                      int32_t nrow, int sh) {
  const int64_t row = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (row >= nrow) return;
  const int b = static_cast<int>(row >> sh), r = static_cast<int>(row & ((1 << sh) - 1));
  uint32_t run = static_cast<uint32_t>(rowptr[row]);
  for (int u = segfirst[b]; u < segfirst[b + 1]; ++u) {
    uint32_t* cell = h + (static_cast<int64_t>(u) << sh) + r;
    const uint32_t c = *cell;
    *cell = run;
    run += c;
  }
}

// ---- the stable split ---------------------------------------------------------------------------------------------
struct SplitArgs {
  const int32_t* i;  // pass 1 input: the mirror
  const int32_t* p;
  const double* x;
  Rec* rec;          // band-major record stream (pass 1 writes, pass 2 reads)
  int32_t* i_out;    // pass 2 output
  double* x_out;
  const int32_t* tb;
  const int32_t* tilecol;
  const int32_t* seg;
  const uint32_t* segcur;
  int nseg;
  int64_t ntiles;
  int64_t nnz;
  int sh, nb;
  int keys;  // keys of this pass (bands / rows per band)
  int kp;    // table pitch: keys rounded up to a multiple of 8
  unsigned int* counter;
};


// Exclusive scan over the warps of the (warp, key) counts of WPT words (two u16 keys each) of one thread, in place;
// tot receives the totals.  Eight words are in flight before the first store.
template <int WPT, int W>
__device__ __forceinline__ void scan_warps(uint32_t* col, const int pitch, uint32_t (&tot)[4]) {
  constexpr int B = 8 / WPT;  // warps per batch: eight words in flight before the first store
#pragma unroll
  for (int w0 = 0; w0 < W; w0 += B) {
    uint32_t c[B][WPT];
#pragma unroll
    for (int i = 0; i < B; ++i) {
      const uint32_t* src = col + (w0 + i) * pitch;
      if (WPT == 1) {
        c[i][0] = src[0];
      } else if (WPT == 2) {
        const uint2 v = *reinterpret_cast<const uint2*>(src);
        c[i][0] = v.x;
        c[i][WPT - 1] = v.y;
      } else {
        const uint4 v = *reinterpret_cast<const uint4*>(src);
        c[i][0] = v.x;
        c[i][1 % WPT] = v.y;
        c[i][2 % WPT] = v.z;
        c[i][3 % WPT] = v.w;
      }
    }
#pragma unroll
    for (int i = 0; i < B; ++i) {
      uint32_t* dst = col + (w0 + i) * pitch;
      if (WPT == 1)
        dst[0] = tot[0];
      else if (WPT == 2)
        *reinterpret_cast<uint2*>(dst) = make_uint2(tot[0], tot[1]);
      else
        *reinterpret_cast<uint4*>(dst) = make_uint4(tot[0], tot[1], tot[2], tot[3]);
#pragma unroll
      for (int q = 0; q < WPT; ++q) tot[q] += c[i][q];
    }
  }
}

template <int PASS>
size_t split_smem_bytes(int kp, int threads, int te) {
  return static_cast<size_t>(te) * (8 + 4 + 2 + (PASS == 1 ? 2 : 0)) + static_cast<size_t>(kp) * 4 * 3 +
         static_cast<size_t>(threads / 32) * kp * 2;
}

template <int PASS, int THREADS, int EPT>
__global__ void __launch_bounds__(THREADS, (EPT > 8 ? 512 : 1024) / THREADS) split_kernel(const SplitArgs a) {
  constexpr int TE = THREADS * EPT;
  constexpr int W = THREADS / 32, SEG = EPT * 32;
  extern __shared__ __align__(16) unsigned char ssm[];
  __shared__ uint32_t wscan[W];
  __shared__ unsigned int s_unit;

  const int K = a.keys, KP = a.kp;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;

  double* img_x = reinterpret_cast<double*>(ssm);                    // [TE] the chunk's output image: values,
  int32_t* img_c = reinterpret_cast<int32_t*>(img_x + TE);           // [TE] source columns,
  uint32_t* img_kr = reinterpret_cast<uint32_t*>(img_c + TE);        // [TE] pass 1: key << 16 | row inside the band
  uint16_t* img_k = reinterpret_cast<uint16_t*>(img_c + TE);         // [TE] pass 2: keys (to find a slot's global address)
  uint32_t* kbase = reinterpret_cast<uint32_t*>(img_k + (PASS == 1 ? 2 * TE : TE));  // [KP] where a key's piece starts in the image
  int32_t* gdelta = reinterpret_cast<int32_t*>(kbase + KP);          // [KP] global slot - image slot
  uint32_t* cur = reinterpret_cast<uint32_t*>(gdelta + KP);          // [KP] next free global slot of every key
  uint16_t* tbl = reinterpret_cast<uint16_t*>(cur + KP);             // [W*KP] records of (warp, key), then its offset
  const int tbl_vec = (W * KP * 2) / 16;

  for (int e = tid; e < tbl_vec; e += THREADS) reinterpret_cast<uint4*>(tbl)[e] = make_uint4(0u, 0u, 0u, 0u);

  // The records of the chunk in flight: warp w owns records [w * SEG, (w + 1) * SEG), 32 consecutive ones per step.
  uint32_t kr[EPT];  // key << 16 | row inside the band (pass 1)
  uint32_t rk[EPT];  // rank inside (warp, key)
  int32_t cc[EPT];
  double xx[EPT];
  const int seg0 = warp * SEG + lane;

  // records [k0, k0 + n) of unit u into the registers (pass 1: and their columns)
  auto load = [&](const int64_t k0, const int n, const int64_t u) {
#pragma unroll
    for (int j = 0; j < EPT; ++j) {
      const int q = seg0 + j * 32;
      kr[j] = 0xffffffffu;
      cc[j] = 0;
      xx[j] = 0.0;
      if (q < n) {
        if (PASS == 1) {
          const int32_t r = ptx::ld_stream_s32(a.i + k0 + q);
          kr[j] = (static_cast<uint32_t>(r >> a.sh) << 16) | static_cast<uint32_t>(r & ((1 << a.sh) - 1));
          xx[j] = ptx::ld_stream_f64(a.x + k0 + q);
        } else {
          const Rec rc = ld_stream_rec(a.rec + k0 + q);
          kr[j] = rc.r << 16;
          cc[j] = rc.c;
          xx[j] = rc.x;
        }
      }
    }
    if (PASS == 1 && seg0 < n) {
      // column of my first record by bisection inside the tile's columns, then walk: columns are long here
      const int64_t kf = k0 + seg0;
      int32_t lo = __ldg(a.tilecol + u), hi = __ldg(a.tilecol + u + 1);
      while (lo < hi) {
        const int32_t mid = lo + ((hi - lo + 1) >> 1);
        if (__ldg(a.p + mid) <= kf)
          lo = mid;
        else
          hi = mid - 1;
      }
      int32_t c = lo;
      int64_t pend = __ldg(a.p + c + 1);
#pragma unroll
      for (int j = 0; j < EPT; ++j) {
        const int q = seg0 + j * 32;
        if (q < n) {
          const int64_t k = k0 + q;
          while (k >= pend) {
            ++c;
            pend = __ldg(a.p + c + 1);
          }
          cc[j] = c;
        }
      }
    }
  };
  // a unit's records: pass 1 one tile, pass 2 one segment of a band's stream
  auto unit_bounds = [&](const int64_t u, int64_t& lo, int64_t& hi) {
    if (PASS == 1) {
      lo = u * TE;
      hi = (a.nnz - lo < TE) ? a.nnz : lo + TE;
    } else {
      lo = __ldg(a.seg + 3 * u + 1);
      hi = __ldg(a.seg + 3 * u + 2);
    }
  };
  // where every key of unit u starts writing: fetched into registers early, stored to cur[] once the chunk in flight
  // no longer needs it
  constexpr int CPT = (SP_MAX_KEYS + THREADS - 1) / THREADS;
  uint32_t curv[CPT];
  auto fetch_cursors = [&](const int64_t u) {
    const uint32_t* src = PASS == 1 ? reinterpret_cast<const uint32_t*>(a.tb) + u * a.nb : a.segcur + (u << a.sh);
#pragma unroll
    for (int e = 0; e < CPT; ++e) {
      const int key = tid + e * THREADS;
      curv[e] = key < K ? __ldg(src + key) : 0u;
    }
  };
  auto store_cursors = [&]() {
#pragma unroll
    for (int e = 0; e < CPT; ++e) {
      const int key = tid + e * THREADS;
      if (key < K) cur[key] = curv[e];
    }
  };
  // the records two chunks ahead, on their way to L2 (one 128-byte line per thread and array)
  auto prefetch = [&](const int64_t k0, const int n) {
    if (PASS == 1) {
      const int64_t e = (k0 & ~int64_t(15)) + static_cast<int64_t>(tid) * 16;
      if (e < k0 + n) {
        ptx::prefetch_l2(a.x + e);
        if (!(tid & 1)) ptx::prefetch_l2(a.i + e);
      }
    } else {
      for (int64_t e = (k0 & ~int64_t(7)) + static_cast<int64_t>(tid) * 8; e < k0 + n; e += THREADS * 8) ptx::prefetch_l2(a.rec + e);
    }
  };

  const int64_t units = PASS == 1 ? a.ntiles : static_cast<int64_t>(a.nseg);
  if (tid == 0) s_unit = atomicAdd(a.counter, 1u);
  __syncthreads();
  int64_t u = s_unit;
  if (u >= units) return;
  int64_t k0, uend;
  unit_bounds(u, k0, uend);
  int n = static_cast<int>((uend - k0 < TE) ? uend - k0 : TE);
  fetch_cursors(u);
  store_cursors();
  load(k0, n, u);
  __syncthreads();  // s_unit read by everybody, the table clear, the cursors in place

  // One chunk per turn.  The chunk after it is loaded into the registers the placement has just freed, so its global
  // loads (pass 1: and the bisection for its columns) fly while the image is flushed; tickets are taken one unit ahead.
  for (;;) {
    const bool last_of_unit = k0 + n >= uend;
    // ---- rank inside the warp: equal keys of a step in lane order, steps in order ----------------------------------
    // `same` = the lanes of this 32-record step that hold my key.
    //   pass 1  a step inside ONE column has its rows ascending, so equal bands are adjacent: run heads by comparing
    //           with the lane below, one ballot;
    //   else    every lane leaves its lane id in a per-warp claim table indexed by key (it lives in the image, idle until
    //           the placement) and reads it back: the lanes of one key all read the same survivor, a lane alone reads
    //           itself.  Nobody overwritten => every lane is alone (most steps of pass 2: a band's stream interleaves
    //           columns, rows look random); otherwise the groups are the lanes with equal survivors — five ballots, one
    //           per bit of a lane id.  (One ballot per KEY bit was ~45 instructions per record at 1024 keys; match.any is
    //           one instruction and no faster: profiles/r02/prof_split_v1_c2 vs _v2_c2.)
    uint8_t* claim = reinterpret_cast<uint8_t*>(ssm) + warp * KP;
#pragma unroll
    for (int j = 0; j < EPT; ++j) {
      const bool valid = kr[j] != 0xffffffffu;
      const uint32_t key = kr[j] >> 16;
      const unsigned vmask = __ballot_sync(0xffffffffu, valid);
      unsigned same;
      bool runs = false;
      if (PASS == 1) {
        const int32_t c_first = __shfl_sync(0xffffffffu, cc[j], 0);
        runs = __all_sync(0xffffffffu, !valid || cc[j] == c_first);
      }
      if (runs) {
        const uint32_t below = __shfl_up_sync(0xffffffffu, key, 1);
        const unsigned heads = __ballot_sync(0xffffffffu, valid && (lane == 0 || key != below));
        const int start = 31 - __clz(heads & (lt_mask | (1u << lane)));
        const unsigned above = heads & ~(lt_mask | (1u << lane));
        const int end = above ? __ffs(above) - 1 : __popc(vmask);  // valid lanes are a prefix of the step
        same = (end >= 32 ? 0xffffffffu : ((1u << end) - 1u)) & ~((1u << start) - 1u);
      } else {
        if (valid) claim[key] = static_cast<uint8_t>(lane);
        __syncwarp();
        const uint32_t who = valid ? claim[key] : static_cast<uint32_t>(lane);
        if (!__any_sync(0xffffffffu, who != static_cast<uint32_t>(lane))) {
          same = 1u << lane;
        } else {
          same = vmask;
#pragma unroll
          for (int b = 0; b < 5; ++b) {
            const bool bit = (who >> b) & 1u;
            const unsigned bal = __ballot_sync(0xffffffffu, bit);
            same &= bit ? bal : ~bal;
          }
        }
      }
      uint16_t* slot = tbl + warp * KP + (valid ? key : 0u);
      const uint32_t old = *slot;  // every lane of the group reads, its lowest lane writes
      __syncwarp();
      if (valid && (same & lt_mask) == 0u) *slot = static_cast<uint16_t>(old + __popc(same));
      rk[j] = old + __popc(same & lt_mask);
      __syncwarp();
    }
    if (last_of_unit && tid == 0) s_unit = atomicAdd(a.counter, 1u);
    __syncthreads();
    // ---- per key: the warps' pieces in warp order; block scan over the keys -> image layout, destinations ----------
    // A thread owns 2, 4 or 8 consecutive keys (as few as still covers all keys with one thread each: the scan over the
    // warps is a dependent chain, so the more threads share it the shorter the wait of everybody else).  Two u16 counts
    // are one 32-bit word and no sum reaches 65536, so the scan is one plain add per word and warp; eight words are
    // loaded before the first store.
    uint32_t mytot = 0;
    uint32_t totw[4] = {0u, 0u, 0u, 0u};
    const int wpt = (KP <= 2 * THREADS) ? 1 : (KP <= 4 * THREADS) ? 2 : 4;  // words per owner thread
    const bool owner = tid * 2 * wpt < KP;
    if (owner) {
      uint32_t* col = reinterpret_cast<uint32_t*>(tbl) + tid * wpt;
      const int pitch = KP / 2;
      if (wpt == 1)
        scan_warps<1, W>(col, pitch, totw);
      else if (wpt == 2)
        scan_warps<2, W>(col, pitch, totw);
      else
        scan_warps<4, W>(col, pitch, totw);
#pragma unroll
      for (int q = 0; q < 4; ++q) mytot += (totw[q] & 0xffffu) + (totw[q] >> 16);
    }
    uint32_t incl = mytot;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const uint32_t up = __shfl_up_sync(0xffffffffu, incl, off);
      if (lane >= off) incl += up;
    }
    if (lane == 31) wscan[warp] = incl;
    __syncthreads();
    if (owner) {
      uint32_t base = incl - mytot;
#pragma unroll
      for (int w = 0; w < W; ++w)
        if (w < warp) base += wscan[w];
      const int key0 = tid * 2 * wpt;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (q < wpt) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int key = key0 + 2 * q + h;
            const uint32_t tot = h ? (totw[q] >> 16) : (totw[q] & 0xffffu);
            const uint32_t c0 = cur[key];
            kbase[key] = base;
            gdelta[key] = static_cast<int32_t>(c0 - base);
            if (PASS == 2) cur[key] = c0 + tot;
            base += tot;
          }
        }
      }
    }
    __syncthreads();
    // ---- place into the image ---------------------------------------------------------------------------------------
#pragma unroll
    for (int j = 0; j < EPT; ++j) {
      if (kr[j] != 0xffffffffu) {
        const uint32_t key = kr[j] >> 16;
        const uint32_t pos = kbase[key] + tbl[warp * KP + key] + rk[j];
        img_x[pos] = xx[j];
        img_c[pos] = cc[j];
        if (PASS == 1)
          img_kr[pos] = kr[j];
        else
          img_k[pos] = static_cast<uint16_t>(key);
      }
    }
    // ---- the chunk after this one -----------------------------------------------------------------------------------
    int64_t nu = u, nk0 = k0 + TE, nuend = uend;
    bool has_next = true;
    if (last_of_unit) {
      nu = s_unit;
      has_next = nu < units;
      if (has_next) unit_bounds(nu, nk0, nuend);
    }
    const int nn = has_next ? static_cast<int>((nuend - nk0 < TE) ? nuend - nk0 : TE) : 0;
    if (has_next) {
      load(nk0, nn, nu);
      if (last_of_unit) fetch_cursors(nu);
      if (PASS == 1) {
        const int64_t pu = nu + gridDim.x;  // tickets go out in order: about where the tile after that will be
        if (pu < units) prefetch(pu * TE, static_cast<int>((a.nnz - pu * TE < TE) ? a.nnz - pu * TE : TE));
      } else if (nk0 + TE < nuend) {
        prefetch(nk0 + TE, static_cast<int>((nuend - nk0 - TE < TE) ? nuend - nk0 - TE : TE));
      }
    }
    __syncthreads();
    // ---- flush: consecutive image slots of a key are consecutive global slots; clear the table ----------------------------
    for (int pp = tid; pp < n; pp += THREADS) {
      const uint32_t kw = PASS == 1 ? img_kr[pp] : static_cast<uint32_t>(img_k[pp]) << 16;
      const int64_t g = static_cast<int64_t>(static_cast<uint32_t>(gdelta[kw >> 16] + pp));
      if (PASS == 1) {
        st_rec(a.rec + g, img_x[pp], img_c[pp], kw & 0xffffu);
      } else {
        a.i_out[g] = img_c[pp];
        a.x_out[g] = img_x[pp];
      }
    }
    for (int e = tid; e < tbl_vec; e += THREADS) reinterpret_cast<uint4*>(tbl)[e] = make_uint4(0u, 0u, 0u, 0u);
    if (has_next && last_of_unit) store_cursors();
    __syncthreads();
    if (!has_next) break;
    u = nu;
    k0 = nk0;
    n = nn;
    uend = nuend;
  }
}

// geometry: threads per CTA x records per thread.  512x8 (4096-record chunks, 2 CTAs per SM); SB200_SPLIT_CFG=1024x8 =
// 8192-record chunks, one CTA per SM (measured within 10 % of each other, like 256x8 / 256x16 / 1024x4: profiles/r02)
struct SplitCfg {
  int threads, ept;
};
SplitCfg split_cfg(int pass = 1) {
  if (const char* e = getenv(pass == 1 ? "SB200_SPLIT_CFG" : "SB200_SPLIT_CFG2")) {
    if (!strcmp(e, "1024x8")) return {1024, 8};
    if (!strcmp(e, "512x8")) return {512, 8};
  }
  if (pass == 2) return {1024, 8};  // twice the records per row and chunk: half the pieces on the way out (C2 1.55 -> 1.23 ms)
  return {SP_THREADS, SP_TE / SP_THREADS};
}

template <int PASS, int THREADS, int EPT>
cudaError_t launch_split(const SplitArgs& a, int sm_count, int64_t units, cudaStream_t st) {
  const size_t smem = split_smem_bytes<PASS>(a.kp, THREADS, THREADS * EPT);
  auto kern = split_kernel<PASS, THREADS, EPT>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
  if (e != cudaSuccess) return e;
  int per_sm = static_cast<int>((227 * 1024) / (smem + 1024));
  const int by_threads = (EPT > 8 ? 512 : 1024) / THREADS;
  if (per_sm > by_threads) per_sm = by_threads;
  if (per_sm < 1) per_sm = 1;
  int64_t grid = static_cast<int64_t>(sm_count) * per_sm;
  if (grid > units) grid = units;
  if (grid < 1) grid = 1;
  kern<<<static_cast<unsigned>(grid), THREADS, smem, st>>>(a);
  count_launch();
  return cudaGetLastError();
}

template <int PASS>
cudaError_t launch_split_cfg(const SplitArgs& a, int sm_count, int64_t units, cudaStream_t st) {
  SplitCfg c = split_cfg(PASS);
  if (split_smem_bytes<PASS>(a.kp, c.threads, c.threads * c.ept) + 1024 > 227 * 1024) c = {SP_THREADS, SP_TE / SP_THREADS};  // many keys: the small image
  if (c.threads == 1024 && c.ept == 8) return launch_split<PASS, 1024, 8>(a, sm_count, units, st);
  return launch_split<PASS, SP_THREADS, SP_TE / SP_THREADS>(a, sm_count, units, st);
}

int segment_chunks() {
  if (const char* e = getenv("SB200_SPLIT_SEG")) {
    const int v = atoi(e);
    if (v >= 1 && v <= 4096) return v;
  }
  return SP_SEG_CHUNKS;
}

int band_shift(const sb200_matrix* m) {
  int sh = 0;
  while ((static_cast<int64_t>(1) << (2 * sh)) < m->nrow) ++sh;  // 2^sh >= sqrt(nrow): bands ~ rows per band
  while ((1 << sh) > SP_MAX_KEYS) --sh;                          // beyond 2^22 rows: 2048 rows a band, up to 3072 bands
  if (const char* e = getenv("SB200_SPLIT_SHIFT")) {
    const int v = atoi(e);
    if (v >= 0 && v <= 16) sh = v;
  }
  return sh;
}

}  // namespace

void free_split_plan(SplitPlan* sp, cudaStream_t s) {
  if (!sp) return;
  pool_free(sp->d_rowptr, s);
  pool_free(sp->d_tb, s);
  pool_free(sp->d_bstart, s);
  pool_free(sp->d_tilecol, s);
  pool_free(sp->d_seg, s);
  pool_free(sp->d_segfirst, s);
  pool_free(sp->d_segcur, s);
  pool_free(sp->d_counters, s);
  delete sp;
}

int64_t split_plan_bytes(const SplitPlan* sp) { return sp ? static_cast<int64_t>(sp->bytes) : 0; }

// Whether the two-split path can take this matrix: key tables within shared memory, the (tile, band) table and the
// record stream within what the device has left.
bool split_transpose_fits(const sb200_matrix* m) {
  if (m->nnz <= 0 || m->nrow <= 0) return false;
  // a handle that already holds the plan took this path before: no driver query per call (cudaMemGetInfo is not cheap);
  // if the record stream does not fit this time the call comes back with SB200_E_NOMEM and the caller falls back
  if (m->plan_split && m->plan_split->sh == band_shift(m)) return true;
  const int sh = band_shift(m);
  const int64_t rb = static_cast<int64_t>(1) << sh;
  const int64_t nb = (m->nrow + rb - 1) >> sh;
  if (rb > SP_MAX_KEYS || nb > SP_MAX_KEYS) return false;
  const int te_ = split_cfg().threads * split_cfg().ept;
  const int64_t kmax = rb > nb ? rb : nb;
  if (split_smem_bytes<1>(static_cast<int>((kmax + 7) & ~7), SP_THREADS, SP_TE) + 1024 > 227 * 1024) return false;
  const int64_t ntiles = (m->nnz + te_ - 1) / te_;
  const size_t table = sizeof(int32_t) * static_cast<size_t>(nb) * static_cast<size_t>(ntiles);
  const size_t stream = sizeof(Rec) * static_cast<size_t>(m->nnz);
  const size_t need = (m->plan_split ? 0 : 3 * table) + stream + (64ull << 20);
  return device_free_bytes() > need + need / 8;
}

static int build_split_plan(sb200_matrix* m, SplitPlan** out) {
  cudaStream_t st = m->stream;
  SplitPlan* sp = new (std::nothrow) SplitPlan();
  if (!sp) return fail(SB200_E_NOMEM, "transpose: out of host memory");
  sp->sh = band_shift(m);
  sp->nb = static_cast<int>((static_cast<int64_t>(m->nrow) + (1 << sp->sh) - 1) >> sp->sh);
  sp->te = split_cfg().threads * split_cfg().ept;
  sp->ntiles = (m->nnz + sp->te - 1) / sp->te;
  const int nb = sp->nb;
  const int64_t nt = sp->ntiles, cells = static_cast<int64_t>(nb) * nt;
  uint32_t *d_hc = nullptr, *d_rowcnt = nullptr;
  int32_t* d_scan = nullptr;
  void* d_ws = nullptr;
  auto drop = [&]() {
    pool_free(d_hc, st);
    pool_free(d_rowcnt, st);
    pool_free(d_scan, st);
    pool_free(d_ws, st);
  };
  struct Guard {
    SplitPlan** sp;
    cudaStream_t st;
    decltype(drop)& fn;
    bool armed = true;
    ~Guard() {
      fn();
      if (armed) {
        free_split_plan(*sp, st);
        *sp = nullptr;
      }
    }
  } guard{&sp, st, drop};
  WallTrace wt("split plan");  // host wall clock: a stall inside a driver call shows here, not in the device's event times
  const size_t ws_bytes = scan_workspace_bytes(cells > m->nrow ? cells : m->nrow);
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&d_hc), sizeof(uint32_t) * static_cast<size_t>(cells), st));
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&d_rowcnt), sizeof(uint32_t) * static_cast<size_t>(m->nrow), st));
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&d_scan), sizeof(int32_t) * (static_cast<size_t>(cells) + 1), st));
  SB_TRY(pool_alloc(&d_ws, ws_bytes, st));
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&sp->d_rowptr), sizeof(int32_t) * (static_cast<size_t>(m->nrow) + 1), st));
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&sp->d_tb), sizeof(int32_t) * static_cast<size_t>(cells), st));
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&sp->d_bstart), sizeof(int32_t) * (nb + 1), st));
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&sp->d_tilecol), sizeof(int32_t) * (static_cast<size_t>(nt) + 1), st));
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&sp->d_counters), sizeof(unsigned int) * 2, st));
  sp->bytes = sizeof(int32_t) * (static_cast<size_t>(m->nrow) + 1 + static_cast<size_t>(cells) + nb + 1 + static_cast<size_t>(nt) + 1) + 8;

  wt.phase("tables allocated");
  SB_CUDA(cudaMemsetAsync(d_rowcnt, 0, sizeof(uint32_t) * static_cast<size_t>(m->nrow), st));
  int64_t grid = nt < static_cast<int64_t>(m->sm_count) * 4 ? nt : static_cast<int64_t>(m->sm_count) * 4;
  split_hist_kernel<<<static_cast<unsigned>(grid), SP_THREADS, sizeof(uint32_t) * nb, st>>>(m->d_i, m->nnz, sp->sh, nb, sp->te, nt, d_hc, d_rowcnt);
  count_launch();
  SB_CUDA(cudaGetLastError());
  SB_TRY(exclusive_scan_u32(st, d_rowcnt, sp->d_rowptr, m->nrow, nullptr, d_ws, ws_bytes));
  SB_TRY(exclusive_scan_u32(st, d_hc, d_scan, cells, nullptr, d_ws, ws_bytes));
  {
    const dim3 g(static_cast<unsigned>((nt + 31) / 32), static_cast<unsigned>((nb + 31) / 32));
    split_table_kernel<<<g, 256, 0, st>>>(d_scan, nb, nt, static_cast<int32_t>(m->nnz), sp->d_tb, sp->d_bstart);
    count_launch();
    SB_CUDA(cudaGetLastError());
  }
  split_tilecol_kernel<<<static_cast<unsigned>((nt + 1 + 255) / 256), 256, 0, st>>>(m->d_p, m->ncol, m->nnz, sp->te, nt, sp->d_tilecol);
  count_launch();
  SB_CUDA(cudaGetLastError());
  // pass-2 units: every band's stream in segments of SP_SEG_CHUNKS chunks
  std::vector<int32_t> bs(static_cast<size_t>(nb) + 1), seg, segfirst(static_cast<size_t>(nb) + 1);
  wt.phase("kernels enqueued");
  SB_CUDA(cudaMemcpyAsync(bs.data(), sp->d_bstart, sizeof(int32_t) * (nb + 1), cudaMemcpyDeviceToHost, st));
  SB_CUDA(cudaStreamSynchronize(st));
  wt.phase("band starts on the host");
  const int seg_chunks = segment_chunks();
  sp->seg_chunks = seg_chunks;
  const int64_t seglen = static_cast<int64_t>(seg_chunks) * sp->te;
  for (int b = 0; b < nb; ++b) {
    segfirst[b] = static_cast<int32_t>(seg.size() / 3);
    for (int64_t k = bs[b]; k < bs[b + 1]; k += seglen) {
      seg.push_back(b);
      seg.push_back(static_cast<int32_t>(k));
      seg.push_back(static_cast<int32_t>(k + seglen < bs[b + 1] ? k + seglen : bs[b + 1]));
    }
  }
  segfirst[nb] = static_cast<int32_t>(seg.size() / 3);
  sp->nseg = segfirst[nb];
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&sp->d_seg), sizeof(int32_t) * (seg.size() + 3), st));
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&sp->d_segfirst), sizeof(int32_t) * (nb + 1), st));
  SB_TRY(pool_alloc(reinterpret_cast<void**>(&sp->d_segcur), sizeof(uint32_t) * ((static_cast<size_t>(sp->nseg) << sp->sh) + 4), st));
  sp->bytes += sizeof(int32_t) * (seg.size() + nb + 1) + sizeof(uint32_t) * (static_cast<size_t>(sp->nseg) << sp->sh);
  SB_CUDA(cudaMemcpyAsync(sp->d_seg, seg.data(), sizeof(int32_t) * seg.size(), cudaMemcpyHostToDevice, st));
  SB_CUDA(cudaMemcpyAsync(sp->d_segfirst, segfirst.data(), sizeof(int32_t) * (nb + 1), cudaMemcpyHostToDevice, st));
  SB_CUDA(cudaStreamSynchronize(st));
  wt.phase("segments uploaded");
  guard.armed = false;
  *out = sp;
  return SB200_OK;
}

int transpose_split_device(sb200_matrix* m, int32_t* d_p_out, int32_t* d_i_out, double* d_x_out) {
  cudaStream_t st = m->stream;
  PhaseTrace tr(st);
  tr.mark("start");
  if (m->plan_split && (m->plan_split->sh != band_shift(m) || m->plan_split->seg_chunks != segment_chunks() ||
                        m->plan_split->te != split_cfg().threads * split_cfg().ept)) {
    free_split_plan(m->plan_split, st);
    m->plan_split = nullptr;
  }
  const bool cached = m->plan_split != nullptr;
  if (!cached) SB_TRY(build_split_plan(m, &m->plan_split));
  const SplitPlan* sp = m->plan_split;
  tr.mark("plan");
  SB_CUDA(cudaMemcpyAsync(d_p_out, sp->d_rowptr, sizeof(int32_t) * (static_cast<size_t>(m->nrow) + 1), cudaMemcpyDeviceToDevice, st));
  Rec* rec = nullptr;  // per-call scratch: the pool hands the same block back call after call (measured: no jitter from it)
  const size_t n = static_cast<size_t>(m->nnz);
  int rc = pool_alloc(reinterpret_cast<void**>(&rec), padded_bytes(sizeof(Rec) * n), st);
  if (rc == SB200_OK) {
    SplitArgs a;
    memset(&a, 0, sizeof(a));
    a.i = m->d_i;
    a.p = m->d_p;
    a.x = m->d_x;
    a.rec = rec;
    a.i_out = d_i_out;
    a.x_out = d_x_out;
    a.tb = sp->d_tb;
    a.tilecol = sp->d_tilecol;
    a.seg = sp->d_seg;
    a.segcur = sp->d_segcur;
    a.nseg = sp->nseg;
    a.ntiles = sp->ntiles;
    a.nnz = m->nnz;
    a.sh = sp->sh;
    a.nb = sp->nb;
    cudaError_t e = cudaMemsetAsync(sp->d_counters, 0, sizeof(unsigned int) * 2, st);
    if (e == cudaSuccess) {
      a.keys = sp->nb;
      a.kp = (a.keys + 7) & ~7;
      a.counter = sp->d_counters;
      e = launch_split_cfg<1>(a, m->sm_count, sp->ntiles, st);
    }
    tr.mark("pass1");
    if (e == cudaSuccess && !m->plan_split->segcur_ready && sp->nseg > 0) {
      // first call: the cursors every segment starts from, counted from the record stream that now exists
      const int R = 1 << sp->sh;
      const int grid = sp->nseg < m->sm_count * 4 ? sp->nseg : m->sm_count * 4;
      split_seg_hist_kernel<<<grid, SP_THREADS, sizeof(uint32_t) * R, st>>>(rec, sp->d_seg, sp->nseg, sp->sh, sp->d_segcur);
      split_seg_scan_kernel<<<static_cast<unsigned>((static_cast<int64_t>(m->nrow) + 255) / 256), 256, 0, st>>>(sp->d_segcur, sp->d_segfirst, sp->d_rowptr,
                                                                                                          m->nrow, sp->sh);
      count_launch(2);
      e = cudaGetLastError();
      if (e == cudaSuccess) m->plan_split->segcur_ready = true;
    }
    if (e == cudaSuccess) {
      a.keys = 1 << sp->sh;
      a.kp = (a.keys + 7) & ~7;
      a.counter = sp->d_counters + 1;
      e = launch_split_cfg<2>(a, m->sm_count, sp->nseg, st);
    }
    tr.mark("pass2");
    if (e != cudaSuccess) rc = cuda_fail(e, "transpose: stream split launch", __FILE__, __LINE__);
  }
  pool_free(rec, st);
  tr.report("transpose (%s, two stream splits) rows/band=%d bands=%d tiles=%lld plan=%.1f MB:", cached ? "cached plan" : "plan built",
            1 << sp->sh, sp->nb, static_cast<long long>(sp->ntiles), sp->bytes / 1048576.0);
  return rc;
}

}  // namespace sb200
