// comm.cuh — combining per-GPU accumulation buffers: the transports and the communicator state behind wavefront.cu's
// yc_comm_* entry points.
//
// BASELINE.json north_star: "Work is partitioned across the 8 GPUs of one box by image tile or sample wave, with the
// scene replicated per GPU.  Per-GPU radiance, median-of-means and GMoN accumulation buffers are combined with NCCL
// over NVLink."  The reference's counterpart is the hand-over of finished tiles between worker threads under
// m_bufferMutex (src/cpu/tile-renderer.hpp:205-239).
//
// Three transports behind the same yc_comm_* entry points:
//   * NCCL (product build; the CPU build has none): libnccl.so.2 loaded with dlopen at the first yc_comm_* call — the
//     library has no link-time dependency on it, and a process that already holds NCCL (PyTorch) shares that copy.
//     Collectives run on the context's own stream, so they order after the wave's kernels without a host round trip.
//   * the caller's sum collective (yc_comm_init_custom): MPI, gloo, a test double.
//   * an in-process group: the contexts of yc_comm_init_all meet at a barrier and the last one to arrive adds the
//     buffers with one kernel over the participants' device pointers (groupSumKernel, which the CPU build of the
//     product sources runs as one loop).  Used when two contexts of a communicator share a GPU — NCCL refuses that —
//     and always in the CPU build, whose contexts share one address space; so the multi-GPU renderer logic runs in
//     the CPU test-suite and on a one-GPU box.
// Tile sharding needs no reduction at all where every participant can address the root GPU's memory (NVLink peer
// access: the other devices of the process, or other processes through an exported allocation): the finalize kernel
// stores every finished pixel into the root's combined frame as it produces it, and the per-wave collective shrinks to
// a barrier (yc_comm_reduce_frames, "direct").  Summing the frames is what remains where that is impossible (the
// caller's own collective across processes).
// Every data collective is a SUM over buffers in which each element is non-zero on at most one participant (disjoint
// tiles; disjoint (bucket, pixel) slots, summed as int32), so x + 0 + ... + 0 is exact and the result is bit-identical
// to one GPU whatever order the transport adds in.
#pragma once
#include <condition_variable>
#include <memory>
#include <mutex>
#include <thread>
#include <unistd.h>

#include "rt.cuh"

struct ncclComm;  // what nccl.h's ncclComm_t points to: Comm holds one in both builds

namespace yb {
enum { kCommF32 = 0, kCommI32 = 1, kCommU64 = 2 };
}  // namespace yb

// NCCL behind six calls with the same signatures in both builds, returning nullptr or an error as rt.cuh's calls do.
// The product build resolves the library at the first call; the CPU build has none and says so.
#ifndef YB_HOSTSIM
#include <dlfcn.h>
#include <nccl.h>

namespace yb {
// The handful of NCCL entry points used, resolved once from libnccl.so.2.
struct NcclApi {
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Reduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  std::string error;
  bool ok = false;
};
inline NcclApi& nccl() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) {
      api.error = std::string("cannot load libnccl.so.2: ") + dlerror();
      return;
    }
    bool all = true;
    auto sym = [&](auto& fn, const char* name) {
      fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(dlsym(h, name));
      all = all && fn != nullptr;
    };
    sym(api.GetUniqueId, "ncclGetUniqueId"), sym(api.CommInitRank, "ncclCommInitRank"), sym(api.CommInitAll, "ncclCommInitAll");
    sym(api.CommDestroy, "ncclCommDestroy"), sym(api.AllReduce, "ncclAllReduce"), sym(api.Reduce, "ncclReduce");
    sym(api.GroupStart, "ncclGroupStart"), sym(api.GroupEnd, "ncclGroupEnd"), sym(api.GetErrorString, "ncclGetErrorString");
    api.ok = all;
    if (!all) api.error = "libnccl.so.2 lacks an expected symbol";
  });
  return api;
}
static_assert(sizeof(ncclUniqueId) == YC_COMM_ID_BYTES, "YC_COMM_ID_BYTES must match ncclUniqueId");

inline const char* ncclErrstr(ncclResult_t r) { return r == ncclSuccess ? nullptr : nccl().GetErrorString(r); }
// Why NCCL cannot be used (nullptr: it can).  The other calls assume it can.
inline const char* ncclUnavailable() { return nccl().ok ? nullptr : nccl().error.c_str(); }
inline const char* ncclNewId(void* id128) {
  ncclUniqueId id;
  if (const char* e = ncclErrstr(nccl().GetUniqueId(&id))) return e;
  memcpy(id128, &id, sizeof id);
  return nullptr;
}
inline const char* ncclJoin(ncclComm** comm, int rank, int world, const void* id128) {
  ncclUniqueId id;
  memcpy(&id, id128, sizeof id);
  return ncclErrstr(nccl().CommInitRank(comm, world, id, rank));
}
inline const char* ncclJoinAll(ncclComm** comms, int n, const int* devices) {
  return ncclErrstr(nccl().CommInitAll(comms, n, devices));
}
inline void ncclRelease(ncclComm* comm) {
  if (comm) nccl().CommDestroy(comm);
}
// In place on `st`: into every participant (root < 0, AllReduce) or into `root` only (Reduce).
inline const char* ncclStreamSum(ncclComm* comm, void* buf, size_t count, int dtype, int root, rt::Stream& st) {
  const ncclDataType_t t = dtype == kCommF32 ? ncclFloat32 : dtype == kCommI32 ? ncclInt32 : ncclUint64;
  if (root < 0) return ncclErrstr(nccl().AllReduce(buf, buf, count, t, ncclSum, comm, st.s));
  return ncclErrstr(nccl().Reduce(buf, buf, count, t, ncclSum, root, comm, st.s));
}
}  // namespace yb
#else
namespace yb {
inline const char* ncclUnavailable() { return "the CPU build has no NCCL: use yc_comm_init_custom or yc_comm_init_all"; }
inline const char* ncclNewId(void*) { return ncclUnavailable(); }
inline const char* ncclJoin(ncclComm**, int, int, const void*) { return ncclUnavailable(); }
inline const char* ncclJoinAll(ncclComm**, int, const int*) { return ncclUnavailable(); }
inline void ncclRelease(ncclComm*) {}
inline const char* ncclStreamSum(ncclComm*, void*, size_t, int, int, rt::Stream&) { return ncclUnavailable(); }
}  // namespace yb
#endif

namespace yb {

// In-process group: n participants, each on its own thread, meet per collective.
constexpr int kGroupMax = 16;
struct GroupPtrs {
  void* p[kGroupMax];
};
// The last arrival's add.  One launch covers `count` in both builds: grid-stride on the GPU, one thread on the CPU.
template <typename T>
__global__ void groupSumKernel(GroupPtrs bufs, int n, size_t count, int root) {
  for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < count; i += size_t(gridDim.x) * blockDim.x) {
    T total = T(0);
    for (int r = 0; r < n; r++) total += static_cast<const T*>(bufs.p[r])[i];
    for (int r = 0; r < n; r++)
      if (root < 0 || r == root) static_cast<T*>(bufs.p[r])[i] = total;
  }
}
struct HostGroup {
  std::mutex m;
  std::condition_variable cv;
  int n = 0, arrived = 0;
  uint64_t generation = 0;
  GroupPtrs bufs{};
  const char* error = nullptr;
  // Every participant calls with its buffer (its own stream drained); the last arrival sums all buffers into
  // bufs[root] (root < 0: into all) and releases the others.
  template <class SumFn>
  const char* sum(int rank, void* buf, SumFn&& doSum) {
    std::unique_lock<std::mutex> lk(m);
    bufs.p[rank] = buf;
    const uint64_t gen = generation;
    if (++arrived == n) {
      error = doSum(bufs, n);
      arrived = 0;
      generation++;
      cv.notify_all();
    } else {
      cv.wait(lk, [&] { return generation != gen; });
    }
    return error;
  }
};
struct Comm {
  int rank = 0, world = 1;
  ncclComm* nccl = nullptr;
  yc_collective_fn custom = nullptr;
  void* customUser = nullptr;
  std::shared_ptr<HostGroup> group;
  // Tile sharding: the root's combined frames.  One block holding {hdr, ldr} x 2: the two copies alternate by reduce
  // (`epoch`), so that the root may still be copying wave k's frame out while wave k + 1 is stored into the other.
  float4* block = nullptr;       // root only: the allocation
  float4 *hdrAll[2] = {nullptr, nullptr}, *ldrAll[2] = {nullptr, nullptr};  // as THIS context addresses them (root: its
                                 // own block; others in direct mode: the root's block through peer access)
  void* imported = nullptr;      // cross-process mapping of the root's block (closed with the communicator)
  uint32_t* detached = nullptr;  // kGroupMax words behind the frames in the block: participant r sets word r before it
                                 // closes its mapping, and the root frees the block only when every importer has
  uint32_t importers = 0;        // root: participants that mapped the block from another process
  size_t frameTexels = 0;
  int root = -1;
  bool direct = false;           // every participant reaches the root's block: finished pixels are stored there directly
  bool stale = true;             // direct: this context's pixels in the next copy are not all current (push them)
  bool barrierSinceFinalize = false;  // a collective ran on the stream after the last finalize
  uint32_t epoch = 0;            // reduces completed since the frames were mapped; the next one publishes copy epoch & 1
  int cur = 0;                   // copy the last reduce completed into (yc_resolve_combined reads it)
  uint64_t* scratch = nullptr;   // device staging for small host-value collectives
};

}  // namespace yb
