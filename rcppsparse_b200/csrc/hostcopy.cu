// Host <-> device copies of PAGEABLE memory (R-owned vectors; the reference's Matrix aliases R memory, README.md:7-9).
//
// A cudaMemcpy from pageable memory is staged by the driver through one pinned buffer by one thread: measured on
// the B200 box 11 GB/s up and ~4.5 GB/s down for C2's 1.2 GB, against 55 GB/s from pinned memory; registering
// the caller's pages first (cudaHostRegister) costs more than it saves (123-170 ms vs 108 ms).  Here a few
// worker threads each own two pinned chunks and a stream: a worker copies its chunk into pinned memory with
// memcpy, sends it with cudaMemcpyAsync and meanwhile fills its other chunk, so the CPU copies of all workers
// and the DMA of the previous chunks run together; the link, not one core's memcpy, becomes the limit.
// Buffers, streams and events are created once per process and device.
#include <string.h>

#include <mutex>
#include <thread>
#include <vector>

#include "common.cuh"

namespace sb200 {
namespace {

constexpr int MAX_WORKERS = 16;

// bytes per pinned chunk (SB200_COPY_CHUNK_KB; fixed for the life of the process).  One-shot C2 transpose on B200, 12 workers:
// 512 KB 100 ms, 1 MB 78, 2 MB 62-64, 4 MB 64-66, 8 MB 68-72 (small chunks pay an event wait each, large ones fall out of
// the host's cache between the CPU copy and the DMA).
size_t chunk_bytes() {
  static const size_t n = [] {
    long kb = 2048;
    if (const char* e = getenv("SB200_COPY_CHUNK_KB")) kb = atol(e);
    if (kb < 64) kb = 64;
    if (kb > 65536) kb = 65536;
    return static_cast<size_t>(kb) << 10;
  }();
  return n;
}

struct Worker {
  unsigned char* buf[2] = {nullptr, nullptr};
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[2] = {nullptr, nullptr};
};

struct Pool {
  std::mutex mu;
  int device = -1;
  int n = 0;
  Worker w[MAX_WORKERS];
};

// One set of staging buffers and streams per device: the single-process sharding layer copies to and from several
// devices at once (one worker thread per device, each over its own PCIe link); a single shared set was torn down and
// rebuilt — 16 cudaHostAlloc calls — every time the device changed, and serialised the devices behind one mutex.
constexpr int MAX_DEVICES = 16;
Pool g_pools[MAX_DEVICES];

int worker_count() {
  static const int n = [] {
    int v = 0;
    if (const char* e = getenv("SB200_COPY_THREADS")) v = atoi(e);
    if (v <= 0) {
      const unsigned hc = std::thread::hardware_concurrency();
      v = hc >= 16 ? 12 : (hc >= 8 ? 4 : 2);  // 16-core B200 host, one-shot C2 transpose: 4 threads 92-113 ms, 8 75-85, 12 70-73, 16 68-71
    }
    return v > MAX_WORKERS ? MAX_WORKERS : v;
  }();
  return n;
}

// call with g_pool.mu held
cudaError_t ensure_pool(Pool& g_pool, int device) {
  if (g_pool.device == device && g_pool.n == worker_count()) return cudaSuccess;
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) return e;
  for (int k = 0; k < g_pool.n; ++k) {  // another device before: start over
    Worker& w = g_pool.w[k];
    for (int b = 0; b < 2; ++b) {
      if (w.buf[b]) cudaFreeHost(w.buf[b]);
      if (w.ev[b]) cudaEventDestroy(w.ev[b]);
    }
    if (w.stream) cudaStreamDestroy(w.stream);
    w = Worker();
  }
  g_pool.n = 0;
  g_pool.device = -1;
  const int n = worker_count();
  for (int k = 0; k < n; ++k) {
    Worker& w = g_pool.w[k];
    for (int b = 0; b < 2; ++b) {
      e = cudaHostAlloc(reinterpret_cast<void**>(&w.buf[b]), chunk_bytes(), cudaHostAllocPortable);
      if (e != cudaSuccess) return e;
      e = cudaEventCreateWithFlags(&w.ev[b], cudaEventDisableTiming);
      if (e != cudaSuccess) return e;
    }
    e = cudaStreamCreateWithFlags(&w.stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) return e;
    g_pool.n = k + 1;
  }
  g_pool.device = device;
  return cudaSuccess;
}

// The copy is `runs` runs of `width` bytes, `dpitch` apart on the device and `hpitch` apart on the host (one run: a
// contiguous range).  Chunks never straddle two runs; chunk c of the whole list goes to worker c mod n.
struct Span {
  unsigned char* dev;
  unsigned char* host;
  size_t dpitch, hpitch, width;
  size_t runs;
  size_t per_run() const { return (width + chunk_bytes() - 1) / chunk_bytes(); }
  size_t chunks() const { return runs * per_run(); }
  // device address, host address and length of chunk c
  void at(size_t c, unsigned char** d, unsigned char** h, size_t* len) const {
    const size_t r = c / per_run(), off = (c % per_run()) * chunk_bytes();
    *d = dev + r * dpitch + off;
    *h = host + r * hpitch + off;
    *len = width - off < chunk_bytes() ? width - off : chunk_bytes();
  }
};

void run_h2d(int device, Worker& w, int k, int n, const Span sp, cudaError_t* err) {
  cudaError_t e = cudaSetDevice(device);
  const size_t chunks = sp.chunks();
  int it = 0;
  for (size_t c = k; c < chunks && e == cudaSuccess; c += n, ++it) {
    const int b = it & 1;
    unsigned char *d, *h;
    size_t len;
    sp.at(c, &d, &h, &len);
    if (it >= 2) e = cudaEventSynchronize(w.ev[b]);  // the DMA that last read this buffer is done
    if (e != cudaSuccess) break;
    memcpy(w.buf[b], h, len);
    e = cudaMemcpyAsync(d, w.buf[b], len, cudaMemcpyHostToDevice, w.stream);
    if (e == cudaSuccess) e = cudaEventRecord(w.ev[b], w.stream);
  }
  const cudaError_t es = cudaStreamSynchronize(w.stream);
  *err = e != cudaSuccess ? e : es;
}

void run_d2h(int device, Worker& w, int k, int n, const Span sp, cudaError_t* err) {
  cudaError_t e = cudaSetDevice(device);
  const size_t chunks = sp.chunks();
  // software pipeline: the DMA of my next chunk runs while I memcpy the previous one out of pinned memory
  unsigned char* prev_h = nullptr;
  size_t prev_len = 0;
  int prev_b = -1, it = 0;
  for (size_t c = k; c < chunks && e == cudaSuccess; c += n, ++it) {
    const int b = it & 1;
    unsigned char *d, *h;
    size_t len;
    sp.at(c, &d, &h, &len);
    e = cudaMemcpyAsync(w.buf[b], d, len, cudaMemcpyDeviceToHost, w.stream);
    if (e == cudaSuccess) e = cudaEventRecord(w.ev[b], w.stream);
    if (prev_b >= 0 && e == cudaSuccess) {
      e = cudaEventSynchronize(w.ev[prev_b]);
      if (e == cudaSuccess) memcpy(prev_h, w.buf[prev_b], prev_len);
    }
    prev_b = b;
    prev_h = h;
    prev_len = len;
  }
  if (prev_b >= 0 && e == cudaSuccess) {
    e = cudaEventSynchronize(w.ev[prev_b]);
    if (e == cudaSuccess) memcpy(prev_h, w.buf[prev_b], prev_len);
  }
  *err = e;
}

int staged(int device, const Span& sp, bool up) {
  if (sp.width == 0 || sp.runs == 0) return SB200_OK;
  if (device < 0 || device >= MAX_DEVICES) return fail(SB200_E_INVALID, "staged copy: device index out of range");
  Pool& g_pool = g_pools[device];
  std::lock_guard<std::mutex> lock(g_pool.mu);
  cudaError_t e = ensure_pool(g_pool, device);
  if (e != cudaSuccess) return cuda_fail(e, "pinned staging buffers", __FILE__, __LINE__);
  const int n = g_pool.n;
  cudaError_t errs[MAX_WORKERS];
  std::vector<std::thread> threads;
  threads.reserve(n);
  for (int k = 0; k < n; ++k) {
    errs[k] = cudaSuccess;
    threads.emplace_back(up ? run_h2d : run_d2h, device, std::ref(g_pool.w[k]), k, n, sp, &errs[k]);
  }
  for (auto& t : threads) t.join();
  for (int k = 0; k < n; ++k)
    if (errs[k] != cudaSuccess) return cuda_fail(errs[k], up ? "staged host-to-device copy" : "staged device-to-host copy", __FILE__, __LINE__);
  return SB200_OK;
}

Span span(void* d, const void* h, size_t dpitch, size_t hpitch, size_t width, size_t runs) {
  return Span{static_cast<unsigned char*>(d), static_cast<unsigned char*>(const_cast<void*>(h)), dpitch, hpitch, width, runs};
}

}  // namespace

// true for ordinary malloc'ed / R-allocated memory (neither cudaHostAlloc'ed nor cudaHostRegister'ed nor managed)
bool host_is_pageable(const void* p) {
  cudaPointerAttributes attr;
  const cudaError_t e = cudaPointerGetAttributes(&attr, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return true;
  }
  return attr.type == cudaMemoryTypeUnregistered;
}

// Blocking.  The device range must not be in use by work that has not completed (callers synchronise the stream
// that allocated / produced it first); on return the data has arrived.
int staged_h2d(int device, void* d_dst, const void* h_src, size_t bytes) { return staged(device, span(d_dst, h_src, 0, 0, bytes, 1), true); }
int staged_d2h(int device, void* h_dst, const void* d_src, size_t bytes) {
  return staged(device, span(const_cast<void*>(d_src), h_dst, 0, 0, bytes, 1), false);
}
// Strided forms: `runs` runs of `width` bytes, `dpitch` bytes apart on the device and `hpitch` apart on the host (a
// column-major slice of a host matrix: runs = its columns).
int staged_h2d_2d(int device, void* d_dst, size_t dpitch, const void* h_src, size_t hpitch, size_t width, size_t runs) {
  return staged(device, span(d_dst, h_src, dpitch, hpitch, width, runs), true);
}
int staged_d2h_2d(int device, void* h_dst, size_t hpitch, const void* d_src, size_t dpitch, size_t width, size_t runs) {
  return staged(device, span(const_cast<void*>(d_src), h_dst, dpitch, hpitch, width, runs), false);
}

}  // namespace sb200
