// host_shim.h -- TEST INFRASTRUCTURE. Lets g++ compile the game-logic half of
// csrc/inversus_kernels.cuh (everything up to the kernel template) for the CPU, so that the
// product's own step logic -- not a restatement of it -- can be replayed against the golden
// fixtures in the CPU test suite and run under AddressSanitizer / UBSan (compute-sanitizer is
// closed on this pool). Only tests/host_kernel/harness.cpp includes this. The product never does:
// INV_HOST_BUILD is defined nowhere else.
#pragma once
#include <stdint.h>
#include <string.h>

#include <cstdlib>

#define __device__
#define __host__
#define __forceinline__ inline
#define __constant__ static const
#define __restrict__

struct uint4 { uint32_t x, y, z, w; };
struct uint2 { uint32_t x, y; };
struct float4 { float x, y, z, w; };
static inline uint4 make_uint4(uint32_t x, uint32_t y, uint32_t z, uint32_t w) { return uint4{x, y, z, w}; }
static inline float4 make_float4(float x, float y, float z, float w) { return float4{x, y, z, w}; }

static inline uint32_t __umulhi(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
static inline int __popc(uint32_t v) { return __builtin_popcount(v); }
// compiled with -ffp-contract=off: plain IEEE operations, like the _rn intrinsics
static inline double __dadd_rn(double a, double b) { return a + b; }
static inline double __dmul_rn(double a, double b) { return a * b; }
static inline float __double2float_rn(double a) { return (float)a; }
static inline uint32_t atomicOr(uint32_t *p, uint32_t v) { const uint32_t o = *p; *p |= v; return o; }
using std::abs;
