// rt.cuh — the thin runtime layer under the wavefront driver: device memory, copies, timing and
// "run this stage over n items".  Product build (nvcc): CUDA runtime, one stream per context.
// YB_HOSTSIM build (g++, tests/hostsim only): the same driver code runs the stages as plain loops
// on the CPU so the pipeline can be diffed against oracle/_ref without a GPU.
#pragma once
#include <chrono>
#include <cstdio>
#include <string>

#include "dmath.cuh"

namespace yb {
namespace rt {

#ifdef YB_HOSTSIM
struct Stream {};
struct Event {
  std::chrono::high_resolution_clock::time_point t;
};
inline const char* init(int, Stream&, int& smCount) {
  smCount = 1;
  return nullptr;
}
inline const char* initStream(int, Stream&) { return nullptr; }
inline void destroy(Stream&) {}
inline void useDevice(int) {}
inline const char* alloc(void** p, size_t bytes) {
  *p = malloc(bytes ? bytes : 1);
  return *p ? nullptr : "out of host memory (hostsim)";
}
inline void release(void* p) { free(p); }
inline const char* hostAlloc(void** p, size_t bytes) { return alloc(p, bytes); }
inline void hostRelease(void* p) { free(p); }
inline const char* h2d(Stream&, void* d, const void* s, size_t n) {
  memcpy(d, s, n);
  return nullptr;
}
inline const char* d2h(Stream&, void* d, const void* s, size_t n) {
  memcpy(d, s, n);
  return nullptr;
}
inline const char* zero(Stream&, void* d, size_t n) {
  memset(d, 0, n);
  return nullptr;
}
inline const char* d2d(Stream&, void* d, const void* s, size_t n) {
  memcpy(d, s, n);
  return nullptr;
}
inline const char* sync(Stream&) { return nullptr; }
inline void eventCreate(Event&) {}
inline void eventDestroy(Event&) {}
inline void eventRecord(Stream&, Event& e) { e.t = std::chrono::high_resolution_clock::now(); }
inline void eventSync(Event&) {}
inline bool eventReady(Event&) { return true; }
inline const char* streamCreate(Stream&) { return nullptr; }
inline void streamWaitEvent(Stream&, Event&) {}
inline const char* d2hAsync(Stream&, void* d, const void* s, size_t n) {
  memcpy(d, s, n);
  return nullptr;
}
inline float eventElapsedMs(Event& a, Event& b) { return std::chrono::duration<float, std::milli>(b.t - a.t).count(); }
inline const char* lastError() { return nullptr; }
// peer memory: the CPU build's "devices" are one address space, and there is nothing to map across processes
constexpr bool kOneAddressSpace = true;
constexpr size_t kIpcHandleBytes = 64;
inline const char* ipcExport(void*, void* handle) {
  memset(handle, 0, kIpcHandleBytes);
  return nullptr;
}
inline const char* ipcImport(void**, const void*) { return "no cross-process device memory in the CPU build"; }
inline void ipcClose(void*) {}
inline const char* enablePeer(int, int) { return nullptr; }

template <int MIN_BLOCKS = 1, class F>
inline void launchFor(Stream&, uint32_t n, const F& f) {
  for (uint32_t i = 0; i < n; i++) f(i);
}
template <class... P, class... A>
inline void launch(Stream&, int, int, void (*kernel)(P...), const A&... args) {
  kernel(args...);
}
#else
struct Stream {
  cudaStream_t s = nullptr;
};
struct Event {
  cudaEvent_t e = nullptr;
};
inline const char* errstr(cudaError_t e) { return e == cudaSuccess ? nullptr : cudaGetErrorString(e); }
inline const char* init(int device, Stream& st, int& smCount) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) return cudaGetErrorString(e);
  if (device < 0 || device >= n) return "no such CUDA device";
  if ((e = cudaSetDevice(device)) != cudaSuccess) return cudaGetErrorString(e);
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return cudaGetErrorString(e);
  smCount = prop.multiProcessorCount;
  if ((e = cudaStreamCreateWithFlags(&st.s, cudaStreamNonBlocking)) != cudaSuccess) return cudaGetErrorString(e);
  return nullptr;
}
// A stream on `device` without the device-property query of init() (which costs up to a quarter of a second per call).
inline const char* initStream(int device, Stream& st) {
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) return cudaGetErrorString(e);
  if ((e = cudaStreamCreateWithFlags(&st.s, cudaStreamNonBlocking)) != cudaSuccess) return cudaGetErrorString(e);
  return nullptr;
}
inline void destroy(Stream& st) {
  if (st.s) cudaStreamDestroy(st.s);
  st.s = nullptr;
}
// The current CUDA device is per-thread state: every yc_* entry point re-selects its context's device, so a
// context may be driven from any thread (yr_render's worker) and contexts on several devices may share a process.
inline void useDevice(int device) { cudaSetDevice(device); }
inline const char* alloc(void** p, size_t bytes) { return errstr(cudaMalloc(p, bytes ? bytes : 1)); }
inline void release(void* p) {
  if (p) cudaFree(p);
}
inline const char* hostAlloc(void** p, size_t bytes) { return errstr(cudaMallocHost(p, bytes ? bytes : 1)); }
inline void hostRelease(void* p) {
  if (p) cudaFreeHost(p);
}
inline const char* h2d(Stream& st, void* d, const void* s, size_t n) {
  if (n == 0) return nullptr;
  cudaError_t e = cudaMemcpyAsync(d, s, n, cudaMemcpyHostToDevice, st.s);
  if (e != cudaSuccess) return cudaGetErrorString(e);
  return errstr(cudaStreamSynchronize(st.s));  // the source may be pageable and short-lived
}
inline const char* d2h(Stream& st, void* d, const void* s, size_t n) {
  if (n == 0) return nullptr;
  cudaError_t e = cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToHost, st.s);
  if (e != cudaSuccess) return cudaGetErrorString(e);
  return errstr(cudaStreamSynchronize(st.s));
}
inline const char* zero(Stream& st, void* d, size_t n) { return n ? errstr(cudaMemsetAsync(d, 0, n, st.s)) : nullptr; }
inline const char* d2d(Stream& st, void* d, const void* s, size_t n) {
  return n ? errstr(cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToDevice, st.s)) : nullptr;
}
inline const char* sync(Stream& st) { return errstr(cudaStreamSynchronize(st.s)); }
inline void eventCreate(Event& e) { cudaEventCreate(&e.e); }
inline void eventDestroy(Event& e) {
  if (e.e) cudaEventDestroy(e.e);
  e.e = nullptr;
}
inline void eventRecord(Stream& st, Event& e) { cudaEventRecord(e.e, st.s); }
inline void eventSync(Event& e) { cudaEventSynchronize(e.e); }
inline bool eventReady(Event& e) { return cudaEventQuery(e.e) == cudaSuccess; }
inline const char* streamCreate(Stream& st) { return errstr(cudaStreamCreateWithFlags(&st.s, cudaStreamNonBlocking)); }
inline void streamWaitEvent(Stream& st, Event& e) { cudaStreamWaitEvent(st.s, e.e, 0); }
// dst must be page-locked (hostAlloc) for the copy to be asynchronous
inline const char* d2hAsync(Stream& st, void* d, const void* s, size_t n) {
  return errstr(cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToHost, st.s));
}
inline float eventElapsedMs(Event& a, Event& b) {
  float ms = 0.0f;
  cudaEventElapsedTime(&ms, a.e, b.e);
  return ms;
}
inline const char* lastError() { return errstr(cudaGetLastError()); }
// Peer memory (comm.cuh: finished pixels are stored straight into the root GPU's frame over NVLink).  A cudaMalloc
// block is exported as an opaque handle, imported by another PROCESS (mapping enables peer access), or — for another
// device of the same process — reached through plain peer access.
constexpr bool kOneAddressSpace = false;  // every device has memory of its own
constexpr size_t kIpcHandleBytes = sizeof(cudaIpcMemHandle_t);
inline const char* ipcExport(void* p, void* handle) {
  return errstr(cudaIpcGetMemHandle(static_cast<cudaIpcMemHandle_t*>(handle), p));
}
inline const char* ipcImport(void** p, const void* handle) {
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof h);
  return errstr(cudaIpcOpenMemHandle(p, h, cudaIpcMemLazyEnablePeerAccess));
}
inline void ipcClose(void* p) {
  if (p) cudaIpcCloseMemHandle(p);
}
inline const char* enablePeer(int device, int peer) {
  if (device == peer) return nullptr;
  int can = 0;
  cudaError_t e = cudaDeviceCanAccessPeer(&can, device, peer);
  if (e != cudaSuccess) return cudaGetErrorString(e);
  if (!can) return "no peer access between the two devices";
  e = cudaDeviceEnablePeerAccess(peer, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) {
    cudaGetLastError();
    return nullptr;
  }
  return errstr(e);
}

// MIN_BLOCKS: resident CTAs per SM the register allocation must allow (occupancy vs registers)
template <class F, int MIN_BLOCKS>
__global__ void __launch_bounds__(256, MIN_BLOCKS) forKernel(uint32_t n, F f) {
  const uint32_t i = blockIdx.x * 256u + threadIdx.x;
  if (i < n) f(i);
}
template <int MIN_BLOCKS = 1, class F>
inline void launchFor(Stream& st, uint32_t n, const F& f) {
  if (n == 0) return;
  forKernel<F, MIN_BLOCKS><<<(n + 255u) / 256u, 256, 0, st.s>>>(n, f);
}
// `kernel` over `grid` CTAs of `block` threads (the CPU build calls it once, hostshim.hpp)
template <class... P, class... A>
inline void launch(Stream& st, int grid, int block, void (*kernel)(P...), const A&... args) {
  kernel<<<grid, block, 0, st.s>>>(args...);
}
#endif

}  // namespace rt

// Warp-aggregated "append one item": one atomic per warp instead of one per lane.  Must be called
// by exactly the lanes that append.  Returns the slot index.
YB_DEV uint32_t aggregatedAppend(uint32_t* counter) {
#ifdef YB_HOSTSIM
  return (*counter)++;
#else
  const unsigned mask = __activemask();
  const int lane = threadIdx.x & 31;
  const int leader = __ffs(mask) - 1;
  uint32_t base = 0;
  if (lane == leader) base = atomicAdd(counter, uint32_t(__popc(mask)));
  base = __shfl_sync(mask, base, leader);
  return base + uint32_t(__popc(mask & ((1u << lane) - 1u)));
#endif
}

// Adds `v` (a small per-thread count) into a 64-bit device counter, one atomic per warp.
YB_DEV void aggregatedCount(unsigned long long* counter, uint32_t v) {
#ifdef YB_HOSTSIM
  *counter += v;
#else
  const unsigned mask = __activemask();
  const uint32_t total = __reduce_add_sync(mask, v);
  if ((threadIdx.x & 31) == __ffs(mask) - 1 && total) atomicAdd(counter, (unsigned long long)total);
#endif
}

}  // namespace yb
