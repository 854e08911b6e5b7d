// hostshim.hpp — lets the device headers and the wavefront driver compile with plain g++
// (-DYB_HOSTSIM) so that tests/hostsim can run the SAME code on the CPU, single-threaded, and
// compare it bit for bit with oracle/_ref where no GPU is available.  Test infrastructure only:
// the product library (libyart_b200.so) is always built by nvcc without this file.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>

struct float4 {
  float x, y, z, w;
};
struct uint2 {
  uint32_t x, y;
};
struct uint3 {
  uint32_t x, y, z;
};
static inline float4 make_float4(float x, float y, float z, float w) { return float4{x, y, z, w}; }
// A kernel is a plain function that rt::launch calls once: one thread of one block runs the whole launch.
#define __global__
#define __launch_bounds__(...)
static const uint3 threadIdx = {0, 0, 0}, blockIdx = {0, 0, 0}, blockDim = {1, 1, 1}, gridDim = {1, 1, 1};
static inline void __syncwarp() {}
static inline unsigned long long atomicAdd(unsigned long long* p, unsigned long long v) {
  const unsigned long long old = *p;
  *p = old + v;
  return old;
}
template <typename T>
static inline T __ldg(const T* p) { return *p; }
static inline uint32_t __brev(uint32_t v) {
  v = ((v >> 1) & 0x55555555u) | ((v & 0x55555555u) << 1);
  v = ((v >> 2) & 0x33333333u) | ((v & 0x33333333u) << 2);
  v = ((v >> 4) & 0x0f0f0f0fu) | ((v & 0x0f0f0f0fu) << 4);
  v = ((v >> 8) & 0x00ff00ffu) | ((v & 0x00ff00ffu) << 8);
  return (v >> 16) | (v << 16);
}
// PRMT: result byte i = byte (selector nibble i) of the eight bytes {x (0-3), y (4-7)}
static inline uint32_t __byte_perm(uint32_t x, uint32_t y, uint32_t s) {
  const uint64_t v = (uint64_t(y) << 32) | x;
  uint32_t r = 0;
  for (int i = 0; i < 4; i++) r |= uint32_t((v >> (8 * ((s >> (4 * i)) & 7u))) & 0xffu) << (8 * i);
  return r;
}
static inline uint32_t __float_as_uint(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  return u;
}
static inline float __uint_as_float(uint32_t u) {
  float f;
  memcpy(&f, &u, 4);
  return f;
}
static inline float __fdiv_rn(float a, float b) { return a / b; }
