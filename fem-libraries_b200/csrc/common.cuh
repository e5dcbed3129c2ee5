// common.cuh -- shared host/device helpers of libfemb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/femb200.h"

namespace femb {

// ---- error plumbing: no exceptions cross the C ABI -------------------------
extern thread_local char g_err[512];
int set_error(const char *fmt, ...);

#define FEMB_CUDA(call)                                                                                  \
   do                                                                                                    \
   {                                                                                                     \
      cudaError_t e__ = (call);                                                                          \
      if (e__ != cudaSuccess)                                                                            \
         return femb::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
   } while (0)

#define FEMB_CHECK(cond, ...)                      \
   do                                              \
   {                                               \
      if (!(cond)) return femb::set_error(__VA_ARGS__); \
   } while (0)

#define FEMB_LAUNCH_CHECK() FEMB_CUDA(cudaGetLastError())

static inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

static inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// device properties cached per process (one process per GPU)
struct DevInfo
{
   int sm_count = 0, cc_major = 0, cc_minor = 0;
   size_t smem_optin = 0;
};
const DevInfo &devinfo();

// opt-in dynamic shared memory of a kernel, set once per growth (not on every launch)
template <auto Kernel>
static inline int ensure_dynamic_smem(size_t smem)
{
   static size_t have = 0;
   if (smem > have)
   {
      FEMB_CUDA(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      have = smem;
   }
   return 0;
}

// ---- element tables --------------------------------------------------------
// FEMB200_Q1 is a pattern-only family (coarse multigrid levels): nd = nv = 4, 9 points that no kernel uses
__host__ __device__ constexpr int elem_nd(int etype)
{
   return etype == FEMB200_P1 ? 3 : (etype == FEMB200_P2 ? 6 : (etype == FEMB200_Q1 ? 4 : 9));
}
__host__ __device__ constexpr int elem_nv(int etype) { return (etype == FEMB200_Q2 || etype == FEMB200_Q1) ? 4 : 3; }
__host__ __device__ constexpr int elem_nq(int etype) { return etype == FEMB200_P1 ? 1 : (etype == FEMB200_P2 ? 3 : 9); }
__host__ __device__ constexpr bool elem_is_triangle(int etype) { return etype == FEMB200_P1 || etype == FEMB200_P2; }
// every element-level entry point (tabulation, assembly, residual, lifting, PA, output fields) refuses Q1
#define FEMB_REFUSE_Q1(etype, who) \
   FEMB_CHECK((etype) != FEMB200_Q1, who ": the Q1 family is pattern only (coarse multigrid levels), it has no element kernel")

// ---- exclusive scans on the device (hand-written, multi-level) --------------
// out[i] = sum_{k<i} in[k], i in [0, n]; out has n+1 entries.
int exclusive_scan_i32_i64(const int32_t *d_in, int64_t *d_out, int64_t n, cudaStream_t st);
int exclusive_scan_i32_i32(const int32_t *d_in, int32_t *d_out, int64_t n, cudaStream_t st);

// ---- streaming loads / stores ----------------------------------------------
__device__ __forceinline__ double2 ld_stream_d2(const double *p)
{
   double2 v;
   asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
   return v;
}
__device__ __forceinline__ void st_stream_d2(double *p, double2 v)
{
   asm volatile("st.global.cs.v2.f64 [%0], {%1,%2};" ::"l"(p), "d"(v.x), "d"(v.y) : "memory");
}

// 256-bit global load (PTX ISA 8.8, sm_100+): one request, one line for a 32-byte record
__device__ __forceinline__ void ld_d4(const double *p, double &a, double &b, double &c, double &d)
{
   asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
}

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
   for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
   return v;
}

}  // namespace femb
