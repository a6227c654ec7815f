// Owning handles of the CUDA resources a context holds. Every handle is released by the destructor of its owner, so a
// context releases everything it acquired -- also when nid_create fails half way. An owner converts to its raw handle
// (device and pinned buffers read like the raw pointers they hold).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include <atomic>
#include <string>
#include <type_traits>

#include "../../include/nid_b200.h"

namespace nid {

int check_cuda(cudaError_t e, const char* what);

// handles held by all owners of the process (nid_live_resources)
extern std::atomic<long long> live_handles;

template <typename H, auto Release>
class Owned {
 public:
  Owned() = default;
  Owned(Owned&& o) noexcept : h_(o.h_) { o.h_ = H(); }  // (move-only: no copy, and no assignment)
  ~Owned() { reset(); }

  operator H() const { return h_; }
  H get() const { return h_; }
  // (for an asynchronous copy of the handle value itself, which must outlive the call)
  const H* handle_address() const { return &h_; }

  // releases the handle held, then owns h
  void reset(H h = H()) {
    if (h_) { Release(h_); live_handles--; }
    h_ = h;
    if (h_) live_handles++;
  }
  // releases the handle held, then owns what make(&handle) creates; on an error the owner is empty and the error
  // is reported as check_cuda(error, what)
  template <typename Make>
  int acquire(Make make, const char* what) {
    reset();
    H h = H();
    const cudaError_t e = make(&h);
    if (e != cudaSuccess) return check_cuda(e, what);
    reset(h);
    return NID_OK;
  }

 private:
  H h_ = H();
};

// device (cudaMalloc) or pinned host (cudaMallocHost) memory of T
template <typename T, bool Pinned>
struct Buffer : std::conditional_t<Pinned, Owned<T*, cudaFreeHost>, Owned<T*, cudaFree>> {
  // n elements, at least one; the buffer held is released first
  int alloc(size_t n, const char* what) {
    const size_t bytes = sizeof(T) * (n ? n : 1);
    return this->acquire([bytes](T** p) { return Pinned ? cudaMallocHost((void**)p, bytes) : cudaMalloc((void**)p, bytes); }, what);
  }
};
template <typename T> using DeviceBuffer = Buffer<T, false>;
template <typename T> using PinnedBuffer = Buffer<T, true>;

struct Stream : Owned<cudaStream_t, cudaStreamDestroy> {
  int create(const char* what) {
    return acquire([](cudaStream_t* s) { return cudaStreamCreateWithFlags(s, cudaStreamNonBlocking); }, what);
  }
};

struct Event : Owned<cudaEvent_t, cudaEventDestroy> {
  int create(unsigned flags, const char* what) {
    return acquire([flags](cudaEvent_t* e) { return cudaEventCreateWithFlags(e, flags); }, what);
  }
};

using Graph = Owned<cudaGraph_t, cudaGraphDestroy>;
using GraphExec = Owned<cudaGraphExec_t, cudaGraphExecDestroy>;

// A width x height CUDA array that tex2Dgather can read (cudaArrayTextureGather) and its texture object: clamped, point
// sampled, element reads. The texture is declared after its array, so it is destroyed first.
struct GatherTexture {
  Owned<cudaArray_t, cudaFreeArray> array;
  Owned<cudaTextureObject_t, cudaDestroyTextureObject> tex;

  // errors: "cudaMallocArray (what)", "cudaCreateTextureObject (what)"
  int create(const cudaChannelFormatDesc& cd, size_t width, size_t height, const char* what) {
    tex.reset();
    const std::string w = std::string(" (") + what + ")";
    int r = array.acquire([&](cudaArray_t* a) { return cudaMallocArray(a, &cd, width, height, cudaArrayTextureGather); },
                          ("cudaMallocArray" + w).c_str());
    if (r != NID_OK) return r;
    cudaResourceDesc rd = {};
    rd.resType = cudaResourceTypeArray;
    rd.res.array.array = array;
    cudaTextureDesc td = {};
    td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;
    td.filterMode = cudaFilterModePoint;
    td.readMode = cudaReadModeElementType;
    td.normalizedCoords = 0;
    return tex.acquire([&](cudaTextureObject_t* t) { return cudaCreateTextureObject(t, &rd, &td, nullptr); },
                       ("cudaCreateTextureObject" + w).c_str());
  }
};

}  // namespace nid
