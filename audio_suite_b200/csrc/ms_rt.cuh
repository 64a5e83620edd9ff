// ms_rt.cuh -- thin portability layer so every kernel body in this library is written once
// and can be compiled two ways:
//   * nvcc, sm_100a: the product.  Ctx::sync() is __syncthreads(), smem is dynamic shared memory.
//   * g++ with -DMS_HOST_EMUL: a cooperative-fibre block emulator (tests/host_emul/) that runs the
//     same kernel bodies on the CPU, one fibre per CUDA thread, so index arithmetic is unit-tested
//     in the build container where there is no GPU.  This is test infrastructure, never a fallback:
//     the shipped shared library contains no host compute path.
#pragma once
#include <stdint.h>
#include <math.h>

#ifdef MS_HOST_EMUL
  #include <cmath>
  #include <cstring>
  #include <algorithm>
  #define MS_DEV inline
  #define MS_DEV_NOINLINE static __attribute__((noinline))
  #define MS_HD inline
  #define MS_RESTRICT
  struct float2 { float x, y; };
  struct float4 { float x, y, z, w; };
  struct double2 { double x, y; };
  static inline float2 make_float2(float x, float y) { float2 r; r.x = x; r.y = y; return r; }
  static inline double2 make_double2(double x, double y) { double2 r; r.x = x; r.y = y; return r; }
  static inline float __ldg(const float* p) { return *p; }
  static inline double __ldg(const double* p) { return *p; }
  static inline float2 __ldg(const float2* p) { return *p; }
  static inline int __ldg(const int* p) { return *p; }
  static inline float __fmaf_rn(float a, float b, float c) { return std::fma(a, b, c); }
  static inline unsigned int __umulhi(unsigned int a, unsigned int b) { return (unsigned int)(((unsigned long long)a * b) >> 32); }
  static inline double cospi(double a) { return std::cos(M_PI * a); }
  namespace msemu { void yield_barrier(); void yield_warp_barrier(); }
  struct Ctx {
      int tid, nthr, bx, by;
      char* smem;
      void sync() const { msemu::yield_barrier(); }
      // warp-level barrier among the 32 fibres of a warp (counting barrier in the emulator's scheduler)
      void syncwarp() const { msemu::yield_warp_barrier(); }
  };
#else
  #include <cuda_runtime.h>
  #define MS_DEV __device__ __forceinline__
  #define MS_DEV_NOINLINE static __device__ __noinline__
  #define MS_HD __host__ __device__ __forceinline__
  #define MS_RESTRICT __restrict__
  struct Ctx {
      int tid, nthr, bx, by;
      char* smem;
      __device__ __forceinline__ void sync() const { __syncthreads(); }
      __device__ __forceinline__ void syncwarp() const { __syncwarp(); }
  };
#endif

// ---- complex helpers, stamped for float2 and double2 -----------------------------------------------
#define MS_STAMP_CPX(C, T, MK) \
MS_DEV C c_mul(C a, C b) { return MK(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); } \
MS_DEV C c_mulc(C a, C b) { return MK(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y); } \
MS_DEV C c_add(C a, C b) { return MK(a.x + b.x, a.y + b.y); } \
MS_DEV C c_sub(C a, C b) { return MK(a.x - b.x, a.y - b.y); } \
MS_DEV C c_scale(C a, T s) { return MK(a.x * s, a.y * s); } \
MS_DEV C c_swap(C a) { return MK(a.y, a.x); } \
MS_DEV C c_conj(C a) { return MK(a.x, -a.y); } \
MS_DEV C c_mul_mi(C a) { return MK(a.y, -a.x); }
MS_STAMP_CPX(float2, float, make_float2)
MS_STAMP_CPX(double2, double, make_double2)
#ifdef MS_HOST_EMUL
static inline double2 __ldg(const double2* p) { return *p; }
#endif

// ---- math wrappers overloaded on precision ---------------------------------------------------------------
#ifdef MS_HOST_EMUL
MS_DEV void r_sincospi(float a, float* s, float* c) { *s = (float)std::sin(M_PI * (double)a); *c = (float)std::cos(M_PI * (double)a); }
MS_DEV void r_sincospi(double a, double* s, double* c) { *s = std::sin(M_PI * a); *c = std::cos(M_PI * a); }
MS_DEV float r_cospi(float a) { return (float)std::cos(M_PI * (double)a); }
MS_DEV double r_cospi(double a) { return std::cos(M_PI * a); }
MS_DEV float r_sinpi(float a) { return (float)std::sin(M_PI * (double)a); }
MS_DEV double r_sinpi(double a) { return std::sin(M_PI * a); }
MS_DEV void r_sincos(float a, float* s, float* c) { *s = std::sin(a); *c = std::cos(a); }
MS_DEV void r_sincos(double a, double* s, double* c) { *s = std::sin(a); *c = std::cos(a); }
#else
MS_DEV void r_sincospi(float a, float* s, float* c) { sincospif(a, s, c); }
MS_DEV void r_sincospi(double a, double* s, double* c) { sincospi(a, s, c); }
MS_DEV float r_cospi(float a) { return cospif(a); }
MS_DEV double r_cospi(double a) { return cospi(a); }
MS_DEV float r_sinpi(float a) { return sinpif(a); }
MS_DEV double r_sinpi(double a) { return sinpi(a); }
MS_DEV void r_sincos(float a, float* s, float* c) { sincosf(a, s, c); }
MS_DEV void r_sincos(double a, double* s, double* c) { sincos(a, s, c); }
#endif
MS_DEV float r_exp(float a) { return expf(a); }
MS_DEV double r_exp(double a) { return exp(a); }
MS_DEV float r_pow(float a, float b) { return powf(a, b); }
MS_DEV double r_pow(double a, double b) { return pow(a, b); }
MS_DEV float r_tanh(float a) { return tanhf(a); }
MS_DEV double r_tanh(double a) { return tanh(a); }
MS_DEV float r_abs(float a) { return fabsf(a); }
MS_DEV double r_abs(double a) { return fabs(a); }
MS_DEV float r_max(float a, float b) { return fmaxf(a, b); }
MS_DEV double r_max(double a, double b) { return fmax(a, b); }
