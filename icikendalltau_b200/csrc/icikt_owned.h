// icikt_owned.h -- move-only owners of the host code's CUDA resources: device arrays, pinned host arrays, streams and
// events.  Each handle releases what it holds when it dies or is assigned over, so an owner made of handles needs no
// hand-written teardown, and a failed allocation leaves an empty handle that the next call allocates again.  An
// owner whose handles live on a device other than the current one sets that device before they die.
#pragma once

#include <cuda_runtime.h>

#include <algorithm>
#include <cstddef>
#include <utility>

namespace icikt {

namespace owned_detail {

struct DeviceMemory {
  static cudaError_t alloc(void** p, size_t bytes) { return cudaMalloc(p, bytes); }
  static void free(void* p) { cudaFree(p); }
};
struct PinnedMemory {
  static cudaError_t alloc(void** p, size_t bytes) { return cudaMallocHost(p, bytes); }
  static void free(void* p) { cudaFreeHost(p); }
};

// An array of `size()` elements of T in Memory, or empty (null, size 0).
template <typename T, class Memory>
class Array {
 public:
  Array() = default;
  Array(Array&& o) noexcept : ptr_(std::exchange(o.ptr_, nullptr)), count_(std::exchange(o.count_, 0)) {}
  Array& operator=(Array&& o) noexcept {
    if (this != &o) {
      reset();
      ptr_ = std::exchange(o.ptr_, nullptr);
      count_ = std::exchange(o.count_, 0);
    }
    return *this;
  }
  Array(const Array&) = delete;
  Array& operator=(const Array&) = delete;
  ~Array() { reset(); }

  // Room for n elements: the allocation stays if it holds n; otherwise it is freed and max(n, 1) elements are
  // allocated.  The contents do not survive a new allocation.  After a failure the array is empty.
  cudaError_t reserve(size_t n) {
    if (ptr_ && n <= count_) return cudaSuccess;
    reset();
    const size_t count = std::max<size_t>(n, 1);
    void* p = nullptr;
    const cudaError_t e = Memory::alloc(&p, count * sizeof(T));
    if (e != cudaSuccess) return e;
    ptr_ = static_cast<T*>(p);
    count_ = count;
    return cudaSuccess;
  }
  void reset() {
    if (ptr_) Memory::free(ptr_);
    ptr_ = nullptr;
    count_ = 0;
  }
  T* get() const { return ptr_; }
  size_t size() const { return count_; }
  explicit operator bool() const { return ptr_ != nullptr; }

 private:
  T* ptr_ = nullptr;
  size_t count_ = 0;
};

}  // namespace owned_detail

template <typename T>
using DeviceArray = owned_detail::Array<T, owned_detail::DeviceMemory>;
template <typename T>
using PinnedArray = owned_detail::Array<T, owned_detail::PinnedMemory>;

// A non-blocking stream, or none.  Converts to cudaStream_t (none: the legacy default stream, 0).
class Stream {
 public:
  Stream() = default;
  Stream(Stream&& o) noexcept : s_(std::exchange(o.s_, nullptr)) {}
  Stream& operator=(Stream&& o) noexcept {
    if (this != &o) {
      reset();
      s_ = std::exchange(o.s_, nullptr);
    }
    return *this;
  }
  Stream(const Stream&) = delete;
  Stream& operator=(const Stream&) = delete;
  ~Stream() { reset(); }

  cudaError_t create() {
    reset();
    cudaStream_t s = nullptr;
    const cudaError_t e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
    if (e == cudaSuccess) s_ = s;
    return e;
  }
  void reset() {
    if (s_) cudaStreamDestroy(s_);
    s_ = nullptr;
  }
  operator cudaStream_t() const { return s_; }

 private:
  cudaStream_t s_ = nullptr;
};

// An event created with the given flags, or none.  Converts to cudaEvent_t.
class Event {
 public:
  Event() = default;
  Event(Event&& o) noexcept : e_(std::exchange(o.e_, nullptr)) {}
  Event& operator=(Event&& o) noexcept {
    if (this != &o) {
      reset();
      e_ = std::exchange(o.e_, nullptr);
    }
    return *this;
  }
  Event(const Event&) = delete;
  Event& operator=(const Event&) = delete;
  ~Event() { reset(); }

  cudaError_t create(unsigned int flags = cudaEventDefault) {
    reset();
    cudaEvent_t ev = nullptr;
    const cudaError_t e = cudaEventCreateWithFlags(&ev, flags);
    if (e == cudaSuccess) e_ = ev;
    return e;
  }
  void reset() {
    if (e_) cudaEventDestroy(e_);
    e_ = nullptr;
  }
  operator cudaEvent_t() const { return e_; }

 private:
  cudaEvent_t e_ = nullptr;
};

}  // namespace icikt
