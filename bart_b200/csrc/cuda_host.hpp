// cuda_host.hpp -- owners of the host code's CUDA resources: device buffers, pinned host buffers,
// events and the pinned staging of file -> device streams.  Each frees what it holds in its
// destructor, so a fail() that throws (error mode 1) leaks nothing, and none can be copied.
#pragma once
#include "host.hpp"
#include <cuda_runtime.h>
#include <algorithm>
#include <vector>

namespace bart {

#define CUDA_OK(call)                                                                      \
  do {                                                                                     \
    cudaError_t e_ = (call);                                                               \
    if (e_ != cudaSuccess) fail("CUDA error %s at %s:%d (%s)", cudaGetErrorString(e_),     \
                                __FILE__, __LINE__, #call);                                \
  } while (0)

struct DeviceMemory {
  static constexpr const char *name = "cudaMalloc";
  static cudaError_t alloc(void **p, size_t bytes) { return cudaMalloc(p, bytes); }
  static void free(void *p) { cudaFree(p); }
};
struct PinnedMemory {
  static constexpr const char *name = "cudaMallocHost";
  static cudaError_t alloc(void **p, size_t bytes) { return cudaMallocHost(p, bytes); }
  static void free(void *p) { cudaFreeHost(p); }
};

// A grow-only buffer of T.  `p` stays valid until the buffer grows, is released or goes away.
template <class T, class Memory> class CudaBuf {
 public:
  T *p = nullptr;
  size_t cap = 0;                             // elements

  CudaBuf() = default;
  explicit CudaBuf(size_t n) { ensure(n); }
  CudaBuf(CudaBuf &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
  CudaBuf &operator=(CudaBuf &&o) noexcept {
    if (this != &o) { release(); std::swap(p, o.p); std::swap(cap, o.cap); }
    return *this;
  }
  ~CudaBuf() { release(); }

  // at least n elements; a new allocation holds exactly n
  T *ensure(size_t n) {
    if (n > cap) allocate(n * sizeof(T));
    return p;
  }
  // at least max(1, n) elements; a new allocation has 25 % headroom, so that buffers sized per
  // call do not reallocate on every small growth
  T *ensure_grow(size_t n) {
    const size_t bytes = std::max<size_t>(1, n) * sizeof(T);
    if (bytes > cap * sizeof(T)) allocate(bytes + bytes / 4);
    return p;
  }
  void release() {
    if (p) Memory::free(p);
    p = nullptr; cap = 0;
  }

 private:
  void allocate(size_t bytes) {
    release();
    void *q = nullptr;
    const cudaError_t e = Memory::alloc(&q, bytes);
    if (e != cudaSuccess) fail("%s of %zu bytes failed: %s", Memory::name, bytes, cudaGetErrorString(e));
    p = (T *)q; cap = bytes / sizeof(T);
  }
};
template <class T> using DevBuf = CudaBuf<T, DeviceMemory>;
template <class T> using PinnedBuf = CudaBuf<T, PinnedMemory>;

// max(1, size) elements holding v
template <class T> void upload(DevBuf<T> &b, const std::vector<T> &v) {
  b.ensure(v.size() ? v.size() : 1);
  if (!v.empty()) CUDA_OK(cudaMemcpy(b.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
}

struct Event {
  cudaEvent_t e = nullptr;
  Event() { CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); }
  ~Event() { if (e) cudaEventDestroy(e); }
  Event(const Event &) = delete;
  Event &operator=(const Event &) = delete;
};

// File ranges -> device memory through two pinned buffers: the read of one chunk (page cache or
// disk) overlaps the copy, and whatever the caller queues behind it, of the previous one.
class PinnedStage {
 public:
  static constexpr size_t kBytes = (size_t)64 << 20;
  explicit PinnedStage(size_t bytes = kBytes) : buf{PinnedBuf<char>(bytes), PinnedBuf<char>(bytes)} {}
  ~PinnedStage() { for (Event &e : ev) cudaEventSynchronize(e.e); }   // no copy still reads a buffer
  PinnedStage(const PinnedStage &) = delete;
  PinnedStage &operator=(const PinnedStage &) = delete;
  size_t size() const { return buf[0].cap; }
  int next() const { return k; }               // the buffer the next put() fills

  // Reads `bytes` (<= size()) at offset `off` of `fd` into the next buffer, once the work queued
  // behind its previous use is done, then queues its copy to `d_dst` and then() on `s`.  Returns
  // false on a short read.
  template <class Then> bool put(int fd, long long off, size_t bytes, void *d_dst, cudaStream_t s, Then then) {
    CUDA_OK(cudaEventSynchronize(ev[k].e));
    if (!parallel_pread(fd, buf[k].p, bytes, off)) return false;
    CUDA_OK(cudaMemcpyAsync(d_dst, buf[k].p, bytes, cudaMemcpyHostToDevice, s));
    then();
    CUDA_OK(cudaEventRecord(ev[k].e, s));
    k ^= 1;
    return true;
  }
  bool put(int fd, long long off, size_t bytes, void *d_dst, cudaStream_t s) {
    return put(fd, off, bytes, d_dst, s, [] {});
  }

 private:
  PinnedBuf<char> buf[2];
  Event ev[2];
  int k = 0;
};

}  // namespace bart
