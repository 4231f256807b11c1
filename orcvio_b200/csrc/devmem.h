// Owning device (cudaMalloc) and pinned host (cudaMallocHost) buffers of the host code.  Every allocation of the
// library goes through these two types, except the grow-only per-thread Scratch of objects.cu (see there).
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstddef>
#include <cstdio>

#include "kernels.h"

namespace ob {

// ORCVIO_HOST_PROF=3: every growth of a device / pinned buffer after construction (a device-wide synchronisation that
// stalls all the batches of the process) is reported
inline void note_growth(const char* what, size_t bytes) {
  static const bool on = env_int("ORCVIO_HOST_PROF", 0) == 3;
  if (on) std::fprintf(stderr, "[replay prof] growth: %s -> %.1f MB\n", what, bytes / 1048576.0);
}

// live bytes of all the buffers of the process: [0] device, [1] pinned (orcvio_device_bytes_held)
inline std::atomic<long long>* bytes_held() {
  static std::atomic<long long> held[2];
  return held;
}

template <class T, bool Pinned>
class OwnedBuf {
 public:
  OwnedBuf() = default;
  OwnedBuf(const OwnedBuf&) = delete;
  OwnedBuf& operator=(const OwnedBuf&) = delete;
  OwnedBuf(OwnedBuf&& o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr; o.n_ = 0; }
  OwnedBuf& operator=(OwnedBuf&& o) noexcept {
    if (this != &o) {
      release();
      p_ = o.p_; n_ = o.n_;
      o.p_ = nullptr; o.n_ = 0;
    }
    return *this;
  }
  ~OwnedBuf() { release(); }

  T* get() const { return p_; }
  size_t size() const { return n_; }                 // capacity in elements
  size_t bytes() const { return n_ * sizeof(T); }

  // Replaces the contents with n uninitialised elements; false (and empty) when the allocation fails.
  bool alloc(size_t n) {
    release();
    if (n == 0) return true;
    void* p = nullptr;
    const cudaError_t e = Pinned ? cudaMallocHost(&p, n * sizeof(T)) : cudaMalloc(&p, n * sizeof(T));
    if (e != cudaSuccess) return false;
    p_ = static_cast<T*>(p);
    n_ = n;
    bytes_held()[Pinned] += (long long)bytes();
    return true;
  }
  // Nothing when need <= size(); otherwise new_cap elements, contents not preserved.  Each call site keeps its own
  // new_cap: the multi-trajectory replay relies on the exact sizes to avoid growths (see Batch::prereserve).
  bool grow(size_t need, size_t new_cap, const char* what) {
    if (need <= n_) return true;
    note_growth(what, new_cap * sizeof(T));
    return alloc(new_cap);
  }

 private:
  void release() {
    if (!p_) return;
    if (Pinned) cudaFreeHost(p_);
    else cudaFree(p_);
    bytes_held()[Pinned] -= (long long)bytes();
    p_ = nullptr;
    n_ = 0;
  }
  T* p_ = nullptr;
  size_t n_ = 0;
};

template <class T> using DeviceBuf = OwnedBuf<T, false>;
template <class T> using PinnedBuf = OwnedBuf<T, true>;

}  // namespace ob
