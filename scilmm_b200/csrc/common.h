// Shared error handling for the C-ABI library.
#pragma once
#include <cuda_runtime.h>

#include "../../include/scilmm_b200.h"

#include <cstdint>
#include <cstdio>
#include <memory>
#include <stdexcept>
#include <string>

namespace slmm {

void set_last_error(const std::string& msg);
extern int64_t g_launch_count;   // kernels launched by this library since the last reset

struct CudaError : std::runtime_error {
  explicit CudaError(const std::string& m) : std::runtime_error(m) {}
};

inline void cuda_check(cudaError_t e, const char* what, const char* file, int line) {
  if (e != cudaSuccess) {
    char buf[512];
    snprintf(buf, sizeof(buf), "CUDA error %s at %s:%d (%s)", cudaGetErrorString(e), file, line, what);
    throw CudaError(buf);
  }
}
#define CUDA_OK(x) ::slmm::cuda_check((x), #x, __FILE__, __LINE__)

// Owning handles: device memory, streams, events and graph execs are freed when their owner goes away, on error
// paths too.  Raw pointers taken with .get() are views.
struct CudaFree { void operator()(void* p) const noexcept { cudaFree(p); } };
struct StreamDestroy { void operator()(cudaStream_t s) const noexcept { cudaStreamDestroy(s); } };
struct EventDestroy { void operator()(cudaEvent_t e) const noexcept { cudaEventDestroy(e); } };
struct GraphExecDestroy { void operator()(cudaGraphExec_t g) const noexcept { cudaGraphExecDestroy(g); } };
template <class T> using DevPtr = std::unique_ptr<T[], CudaFree>;
using Stream = std::unique_ptr<CUstream_st, StreamDestroy>;
using Event = std::unique_ptr<CUevent_st, EventDestroy>;
using GraphExec = std::unique_ptr<CUgraphExec_st, GraphExecDestroy>;

template <typename T>
DevPtr<T> dev_alloc(size_t count) {
  T* p = nullptr;
  if (count == 0) count = 1;
  CUDA_OK(cudaMalloc((void**)&p, count * sizeof(T)));
  return DevPtr<T>(p);
}

template <typename T>
DevPtr<T> dev_upload(const T* host, size_t count, cudaStream_t st = 0) {
  DevPtr<T> p = dev_alloc<T>(count);
  if (count) CUDA_OK(cudaMemcpyAsync(p.get(), host, count * sizeof(T), cudaMemcpyHostToDevice, st));
  return p;
}

inline Event make_event(unsigned flags) {
  cudaEvent_t e = nullptr;
  CUDA_OK(cudaEventCreateWithFlags(&e, flags));
  return Event(e);
}

}  // namespace slmm

#define SLMM_TRY try {
#define SLMM_CATCH                                                       \
  }                                                                      \
  catch (const ::slmm::CudaError& e) {                                   \
    ::slmm::set_last_error(e.what());                                    \
    return SLMM_ERR_CUDA;                                                \
  }                                                                      \
  catch (const std::invalid_argument& e) {                               \
    ::slmm::set_last_error(e.what());                                    \
    return SLMM_ERR_INVALID;                                             \
  }                                                                      \
  catch (const std::exception& e) {                                      \
    ::slmm::set_last_error(e.what());                                    \
    return SLMM_ERR_INTERNAL;                                            \
  }
