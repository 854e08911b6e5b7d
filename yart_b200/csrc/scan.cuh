// scan.cuh — inclusive prefix sum of 64-bit words on a stream, in place: the BVH build's packed class counts
// (bvh_build.cuh) and the adaptive-sampling compaction (wavefront.cu) pack two 32-bit counts per word.  n > 0; `sums`
// holds at least n / 2048 + 1 words of scratch.  The CPU build (YB_HOSTSIM) runs one serial loop.
#pragma once
#include "rt.cuh"

namespace yb {

#ifdef YB_HOSTSIM
struct ScanSeqK {
  unsigned long long* v;
  uint32_t n;
  YB_DEV void operator()(uint32_t) const {
    unsigned long long acc = 0ull;
    for (uint32_t i = 0; i < n; i++) acc += v[i], v[i] = acc;
  }
};
inline void inclusiveScan(rt::Stream& st, unsigned long long* v, unsigned long long*, uint32_t n) {
  rt::launchFor(st, 1, ScanSeqK{v, n});
}
#else
constexpr int kScanBlock = 256, kScanPer = 8, kScanTile = kScanBlock * kScanPer;
__device__ inline unsigned long long blockInclusive(unsigned long long x, unsigned long long* shared, unsigned long long& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) shared[warp] = x;
  __syncthreads();
  if (warp == 0) {
    unsigned long long w = lane < kScanBlock / 32 ? shared[lane] : 0ull;
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long y = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += y;
    }
    if (lane < kScanBlock / 32) shared[lane] = w;
  }
  __syncthreads();
  if (warp > 0) x += shared[warp - 1];
  total = shared[kScanBlock / 32 - 1];
  __syncthreads();
  return x;
}
__global__ void __launch_bounds__(kScanBlock) scanTileSumsK(const unsigned long long* v, unsigned long long* sums, uint32_t n) {
  __shared__ unsigned long long sh[kScanBlock / 32];
  const size_t base = size_t(blockIdx.x) * kScanTile + size_t(threadIdx.x) * kScanPer;
  unsigned long long acc = 0ull;
  for (int k = 0; k < kScanPer; k++)
    if (base + k < n) acc += v[base + k];
  unsigned long long total;
  blockInclusive(acc, sh, total);
  if (threadIdx.x == 0) sums[blockIdx.x] = total;
}
__global__ void __launch_bounds__(kScanBlock) scanSumsK(unsigned long long* sums, uint32_t nTiles) {
  // one block: exclusive scan of the tile sums, kScanBlock at a time with a running carry
  __shared__ unsigned long long sh[kScanBlock / 32];
  unsigned long long carry = 0ull;
  for (uint32_t base = 0; base < nTiles; base += kScanBlock) {
    const uint32_t i = base + threadIdx.x;
    const unsigned long long x = i < nTiles ? sums[i] : 0ull;
    unsigned long long total;
    const unsigned long long incl = blockInclusive(x, sh, total);
    if (i < nTiles) sums[i] = carry + incl - x;
    carry += total;
  }
}
__global__ void __launch_bounds__(kScanBlock) scanApplyK(unsigned long long* v, const unsigned long long* sums, uint32_t n) {
  __shared__ unsigned long long sh[kScanBlock / 32];
  const size_t base = size_t(blockIdx.x) * kScanTile + size_t(threadIdx.x) * kScanPer;
  unsigned long long x[kScanPer], acc = 0ull;
  for (int k = 0; k < kScanPer; k++) {
    x[k] = base + k < n ? v[base + k] : 0ull;
    acc += x[k];
  }
  unsigned long long total;
  const unsigned long long incl = blockInclusive(acc, sh, total);
  unsigned long long run = sums[blockIdx.x] + incl - acc;
  for (int k = 0; k < kScanPer; k++) {
    run += x[k];
    if (base + k < n) v[base + k] = run;
  }
}
inline void inclusiveScan(rt::Stream& st, unsigned long long* v, unsigned long long* sums, uint32_t n) {
  const uint32_t tiles = (n + kScanTile - 1) / kScanTile;
  scanTileSumsK<<<tiles, kScanBlock, 0, st.s>>>(v, sums, n);
  scanSumsK<<<1, kScanBlock, 0, st.s>>>(sums, tiles);
  scanApplyK<<<tiles, kScanBlock, 0, st.s>>>(v, sums, n);
}
#endif

}  // namespace yb
