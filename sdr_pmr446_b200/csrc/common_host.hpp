// Host-side plumbing shared by the C-ABI entry points: error reporting, device buffers,
// ring gather / history kernels, and the Frontend object that owns the DC-blocker + multi-stage
// resampler launches (the device counterpart of iirfilt_crcf + msresamp_crcf,
// /root/reference/src/sdr_pmr446.c:422-428,795-796; src/dsd_in.c:97-101,167-168).
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/pmr446_b200.h"
#include "design.hpp"
#include "frontend.cuh"

namespace pmr {

inline std::string& last_error_string() {
  static thread_local std::string s;
  return s;
}
inline int fail(int code, const char* msg) {
  last_error_string() = msg;
  return code;
}
#define CUDA_TRY(expr)                                                                         \
  do {                                                                                         \
    cudaError_t e__ = (expr);                                                                  \
    if (e__ != cudaSuccess) {                                                                  \
      char buf__[256];                                                                         \
      snprintf(buf__, sizeof buf__, "%s:%d: %s", __FILE__, __LINE__, cudaGetErrorString(e__)); \
      return pmr::fail(PMR446_ECUDA, buf__);                                                   \
    }                                                                                          \
  } while (0)

inline int select_device(int device) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return fail(PMR446_ENODEV, "no CUDA device: this library has no CPU fallback");
  if (device >= 0) {
    if (device >= count) return fail(PMR446_ENODEV, "device ordinal out of range");
    CUDA_TRY(cudaSetDevice(device));
  }
  return 0;
}

// The input formats (pmr446_config::in_fmt): bytes per IQ sample and the loader of the front end's first launch.  Every
// value that is not one of the integer formats is read as cf32.
inline int fmt_bytes_per_sample(int in_fmt) {
  switch (in_fmt) {
    case PMR446_FMT_CU8: return 2;
    case PMR446_FMT_CS8: return 2;
    case PMR446_FMT_CS16: return 4;
    default: return 8;
  }
}
inline int fmt_source(int in_fmt) {
  switch (in_fmt) {
    case PMR446_FMT_CU8: return SRC_CU8;
    case PMR446_FMT_CS8: return SRC_CS8;
    case PMR446_FMT_CS16: return SRC_CS16;
    default: return SRC_CF32;
  }
}

inline long long next_pow2(long long v) {
  long long p = 1;
  while (p < v) p <<= 1;
  return p;
}

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  DevBuf() {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), bytes(o.bytes) { o.p = nullptr; o.bytes = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) { release(); p = o.p; bytes = o.bytes; o.p = nullptr; o.bytes = 0; }
    return *this;
  }
  ~DevBuf() { release(); }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
  }
  int alloc(size_t n) {
    release();
    if (n == 0) n = 16;
    if (cudaMalloc(&p, n) != cudaSuccess) {
      p = nullptr;
      cudaGetLastError();
      return fail(PMR446_ENOMEM, "cudaMalloc failed");
    }
    bytes = n;
    return 0;
  }
  int alloc_zero(size_t n) {
    if (int rc = alloc(n)) return rc;
    CUDA_TRY(cudaMemset(p, 0, bytes));
    return 0;
  }
  int ensure(size_t n) { return (p && bytes >= n) ? 0 : alloc(n); }
};

// Row stride of a host-buffer call's input, or PMR446_EINVAL: a single stream may pass a stride smaller than its chunk
// (0, say), several streams may not.
inline long long host_iq_stride(long long iq_stride, unsigned n, size_t bytes_per_sample, int streams) {
  const long long row = (long long)(n * bytes_per_sample);
  if (iq_stride >= row) return iq_stride;
  if (streams > 1) return fail(PMR446_EINVAL, "iq_stride smaller than one stream's chunk");
  return row;
}

// stage(host, buf, bytes): the device buffer, grown to `bytes`, that stages a host-buffer call's output the caller
// requested (host != nullptr); nullptr for one not requested.  A failed allocation must fail the call, not silently
// drop the output: the first one is kept in rc.
struct Staging {
  int rc = 0;
  template <typename T>
  T* operator()(T* host, DevBuf& buf, size_t bytes) {
    if (!host || rc) return nullptr;
    rc = buf.ensure(bytes);
    return rc ? nullptr : (T*)buf.p;
  }
};

// Device -> host copy of columns [col0, col0 + cols) of `rows` rows of elt-byte elements; nothing if the output was not
// requested (host == nullptr) or the range is empty.
inline void copy_back(cudaStream_t st, void* host, const void* dev, long long host_ld, long long dev_ld, size_t elt, long long rows,
                      long long col0, long long cols) {
  if (host && cols > 0)
    cudaMemcpy2DAsync((char*)host + col0 * elt, host_ld * elt, (const char*)dev + col0 * elt, dev_ld * elt, cols * elt, rows,
                      cudaMemcpyDeviceToHost, st);
}

// Frames (channelizer outputs per channel) that the next n input samples complete in a batch chain (closed form).
long long batch_frames_after(const pmr446_batch* b, unsigned n);

// out[row][k] = ring[row][(start + k) & mask], k < count
template <typename T>
__global__ void gather_ring_kernel(const T* ring, long long ring_stride, long long mask, long long start, long long count, T* out, long long out_ld) {
  long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  long long row = blockIdx.y;
  long long n = start + k;
  out[row * out_ld + k] = n >= 0 ? ring[row * ring_stride + (n & mask)] : T();
}

// dst[s][k] = x[new_base + k] taken from the two-source view (history or current chunk)
template <typename T>
__global__ void hist_update_kernel(SrcView v, T* dst, long long dst_stride_elts, long long new_base, int count) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  int s = blockIdx.y;
  long long n = new_base + k;
  T val = T();
  if (n >= v.n0) {
    if (n < v.n1) val = ((const T*)((const char*)v.cur + (long long)s * v.cur_stride))[n - v.n0];
  } else if (n >= v.hist_base) {
    val = ((const T*)((const char*)v.hist + (long long)s * v.hist_stride))[n - v.hist_base];
  }
  dst[(long long)s * dst_stride_elts + k] = val;
}

// Optional per-kernel timing with CUDA events recorded on the launch stream (bench.py's roofline).
// mark(tag) closes the interval since the previous mark and attributes it to `tag`.
enum { TM_START = 0, TM_DC = 1, TM_CASCADE0 = 2, TM_CASCADE1 = 3, TM_CASCADE2 = 4, TM_HIST = 5, TM_CHANNELIZE = 6, TM_AUDIO = 7,
       TM_WATERFALL = 8, TM_GATHER = 9, TM_DSD = 10, TM_NTAGS = 11 };
struct Timer {
  bool enabled = false;
  std::vector<cudaEvent_t> ev;
  std::vector<int> tag;
  size_t used = 0;
  double total_ms[TM_NTAGS] = {0};
  long long count[TM_NTAGS] = {0};
  ~Timer() { for (auto e : ev) cudaEventDestroy(e); }
  void mark(cudaStream_t st, int t) {
    if (!enabled) return;
    if (used == ev.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      ev.push_back(e);
      tag.push_back(0);
    }
    tag[used] = t;
    cudaEventRecord(ev[used++], st);
  }
  // folds the recorded events into the totals; call after the stream has been synchronised
  void collect() {
    for (size_t i = 1; i < used; i++) {
      if (tag[i] == TM_START) continue;
      float ms = 0.0f;
      if (cudaEventElapsedTime(&ms, ev[i - 1], ev[i]) == cudaSuccess) { total_ms[tag[i]] += ms; count[tag[i]]++; }
    }
    used = 0;
  }
  void clear() {
    used = 0;
    for (int i = 0; i < TM_NTAGS; i++) { total_ms[i] = 0; count[i] = 0; }
  }
};

}  // namespace pmr
