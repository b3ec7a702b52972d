// cuda_handles.h -- owners of CUDA resources: released when the owning object goes away
#pragma once
#include <cuda_runtime.h>

#include <memory>
#include <type_traits>

namespace sffg {

struct CudaFree { void operator()(void *p) const { cudaFree(p); } };
struct CudaFreeHost { void operator()(void *p) const { cudaFreeHost(p); } };
struct StreamDestroy { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
struct EventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
template <class T> using DevPtr = std::unique_ptr<T, CudaFree>;
template <class T> using PinnedPtr = std::unique_ptr<T, CudaFreeHost>;   // cudaHostAllocMapped
using Stream = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, StreamDestroy>;
using Event = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, EventDestroy>;

// hands the handle that `create` writes to the owner, once the call has succeeded
template <class Owner, class Create> cudaError_t make(Owner &o, Create create) {
  typename Owner::pointer h = nullptr;
  const cudaError_t e = create(&h);
  if (e == cudaSuccess) o.reset(h);
  return e;
}
template <class T> cudaError_t dev_alloc(DevPtr<T> &o, size_t bytes) {
  return make(o, [&](T **p) { return cudaMalloc(p, bytes); });
}
template <class T> cudaError_t host_alloc(PinnedPtr<T> &o, size_t bytes) {
  return make(o, [&](T **p) { return cudaHostAlloc(p, bytes, cudaHostAllocMapped); });
}
inline cudaError_t make_stream(Stream &o) {
  return make(o, [](cudaStream_t *s) { return cudaStreamCreateWithFlags(s, cudaStreamNonBlocking); });
}
inline cudaError_t make_event(Event &o) {
  return make(o, [](cudaEvent_t *e) { return cudaEventCreateWithFlags(e, cudaEventDisableTiming); });
}

}  // namespace sffg
