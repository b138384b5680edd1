// TEST INFRASTRUCTURE -- lets practical-path-guiding_b200/csrc/ppg_device.cuh (the product's CUDA device functions) compile for the HOST with g++, so that the
// arithmetic the kernels are written with can be compared on the CPU with the reference's own code (oracle/_ref/libmicrofacet_ref.so) and with the oracle:
// +, -, *, / and sqrt are IEEE on both sides (the kernels are built with -fmad=false -prec-div=true -prec-sqrt=true, this harness with -ffp-contract=off);
// only the libm calls (expf, sincosf, ...) are the host's here and the device's there.  Built by tests/test_device_source_on_host.py:
//   g++ -D__device__= -D__host__= -D__global__= -D__shared__= -D__forceinline__=inline -D__noinline__= -I$CUDA/include ...
// CUDA's own headers supply float3 / float4 / make_float3 / __half2float for host compilers; the intrinsics the device code uses are given host meanings here.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
using std::isfinite; using std::min; using std::max;
template <class T> static inline T __ldg(const T *p) { return *p; }
template <class T> static inline T __ldcs(const T *p) { return *p; }
template <class T> static inline void __stcs(T *p, T v) { *p = v; }
static inline unsigned __float_as_uint(float f) { unsigned u; memcpy(&u, &f, 4); return u; }
static inline int __float_as_int(float f) { int u; memcpy(&u, &f, 4); return u; }
static inline float __uint_as_float(unsigned u) { float f; memcpy(&f, &u, 4); return f; }
static inline float __int_as_float(int u) { float f; memcpy(&f, &u, 4); return f; }
static inline unsigned __funnelshift_r(unsigned lo, unsigned hi, unsigned s) { s &= 31; return s ? (lo >> s) | (hi << (32 - s)) : lo; }
static inline double __dmul_rn(double a, double b) { return a * b; }          // (no contraction: -ffp-contract=off)
static inline double __dadd_rn(double a, double b) { return a + b; }
static inline double __dsub_rn(double a, double b) { return a - b; }
#define __expf(x) expf(x)                                                      /* fast-math exp on the device (only where stated in the kernels); glibc declares but does not export the name */
static inline float __fdividef(float a, float b) { return a / b; }            // approximate on the device (<= 2 ulp): the conservative pre-filter of the tiny-scene test and the Adam chain (fraction_link) use it
static inline unsigned __ballot_sync(unsigned, int p) { return p ? 1u : 0u; }
static inline unsigned __match_any_sync(unsigned, unsigned long long) { return 1u; }
template <class T> static inline T __shfl_sync(unsigned, T v, int) { return v; }
template <class T> static inline T __shfl_xor_sync(unsigned, T, int) { return T(); }   // a one-lane warp: the other lane of a butterfly does not exist (only compiled, never run here)
static inline double atomicAdd(double *a, double v) { const double o = *a; *a += v; return o; }
static inline int __popc(unsigned v) { return __builtin_popcount(v); }
static inline int __ffs(int v) { return __builtin_ffs(v); }
static inline unsigned __activemask() { return 1u; }
static inline void __syncwarp(unsigned = 0xffffffffu) {}
static inline void __syncthreads() {}
static inline float atomicAdd(float *a, float v) { const float o = *a; *a += v; return o; }
static inline unsigned atomicAdd(unsigned *a, unsigned v) { const unsigned o = *a; *a += v; return o; }
static inline unsigned long long atomicAdd(unsigned long long *a, unsigned long long v) { const unsigned long long o = *a; *a += v; return o; }
struct HostDim3 { unsigned x, y, z; };
static HostDim3 threadIdx = {0, 0, 0}, blockIdx = {0, 0, 0}, blockDim = {1, 1, 1}, gridDim = {1, 1, 1};
