// kge_common.cuh -- shared device helpers and host-side error plumbing for libkge_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/kge_b200.h"
#include "kge_math.h"

namespace kge {

// ---- error plumbing (no exceptions across the C ABI) --------------------------------------------
void set_error(const char *fmt, ...);
int check_model(const kge_model_t *m);
// Makes `device` current for the duration of an ABI call and restores the caller's current device on return (a model
// on cuda:1 must not silently change the calling thread's device for later allocations).
struct DeviceGuard {
  int prev = -1;
  bool changed = false;
  int enter(int device);
  ~DeviceGuard() { if (changed) cudaSetDevice(prev); }
};

#define KGE_CUDA_OK(expr)                                                                   \
  do {                                                                                      \
    cudaError_t e__ = (expr);                                                               \
    if (e__ != cudaSuccess) {                                                               \
      kge::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
      return KGE_ERR_CUDA;                                                                  \
    }                                                                                       \
  } while (0)

#define KGE_REQUIRE(cond, ...)              \
  do {                                      \
    if (!(cond)) {                          \
      kge::set_error(__VA_ARGS__);          \
      return KGE_ERR_INVALID;               \
    }                                       \
  } while (0)

// ---- per-candidate inner operations --------------------------------------------------------------
// Every (model, mode) folds the fixed side of the triple into a query vector q (model.py:166-249);
// what is left per candidate row x is one of these element operations followed by a sum over k.
enum Op {
  OP_SUBABS = 0,   // TransE tail-batch/single: |(h+r) - t|      q = h + r
  OP_ADDABS = 1,   // TransE head-batch:        |h + (r-t)|      q = r - t
  OP_MUL = 2,      // DistMult:                 q * x            q = h*r or r*t
  OP_CMUL = 3,     // ComplEx:                  q_re x_re + q_im x_im
  OP_CDIST = 4,    // RotatE:                   |q - x| (complex modulus)
  OP_SUBSIN = 5,   // pRotatE tail/single:      |sin((ph+pr) - pt)|
  OP_ADDSIN = 6,   // pRotatE head-batch:       |sin(ph + (pr-pt))|
  OP_SQDIFF = 7    // similarity search, l2:    (q - x)^2        (no model scores with it)
};

__host__ __device__ constexpr bool op_is_complex(int op) { return op == OP_CMUL || op == OP_CDIST; }

__host__ __device__ constexpr int op_of(int model, bool head_batch) {
  return model == KGE_TRANSE ? (head_batch ? OP_ADDABS : OP_SUBABS)
         : model == KGE_DISTMULT ? OP_MUL
         : model == KGE_COMPLEX ? OP_CMUL
         : model == KGE_ROTATE ? OP_CDIST
                               : (head_batch ? OP_ADDSIN : OP_SUBSIN);
}

// rho/pi as the fp32 scalar torch divides by (`relation/(self.embedding_range.item()/pi)`)
inline float phase_scale(const kge_model_t *m) {
  const double pi = m->model == KGE_PROTATE ? 3.14159262358979323846 : 3.14159265358979323846;
  return (float)((double)m->embedding_range / pi);
}

#if defined(__CUDACC__)
// ---- warp / block reductions --------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---- 128-bit global access ----------------------------------------------------------------------
__device__ __forceinline__ float4 ldg_stream4(const float *p) {   // read-only, do not pollute L1
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void red_add4(float *p, float a, float b, float c, float d) {
  // sm_90+ vector reduction: one 16-byte fire-and-forget atomic add per lane
  asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d)
               : "memory");
}
__device__ __forceinline__ void red_add1(float *p, float a) {
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(a) : "memory");
}
__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// 1/sqrt(x) on the MUFU pipe, one instruction (flush-to-zero: callers guard x >= FLT_MIN)
__device__ __forceinline__ float rsqrt_fast(float x) {
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
constexpr float kFltMin = 1.17549435e-38f;

// ---- L2 residency hints (createpolicy + .L2::cache_hint) -------------------------------------------------------
// The 120 MB entity table of FB15k-sized models almost fits the 126 MB L2, but every train step also streams the two
// Adam moment tables (240 MB read + 240 MB written) through it.  Tagging the moment traffic evict_first and the entity
// rows evict_last keeps the table that the NEXT step gathers at random resident.  kind: 0 normal, 1 evict_first, 2 evict_last.
__device__ __forceinline__ uint64_t l2_policy(int kind) {
  uint64_t p;
  if (kind == 1) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  else if (kind == 2) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ float4 ld4_hint(const float *p, uint64_t pol) {
  float4 r;
  asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p), "l"(pol));
  return r;
}
__device__ __forceinline__ void st4_hint(float *p, float4 v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w),
               "l"(pol)
               : "memory");
}

// ---- NVSwitch multicast stores (NVLS): one store writes the same address in every rank's replica of a multicast-mapped
// allocation (the local one included) ----------------------------------------------------------------------------
__device__ __forceinline__ void multimem_st_b32(void *mc, uint32_t v) {
  asm volatile("multimem.st.relaxed.sys.global.b32 [%0], %1;" ::"l"(mc), "r"(v) : "memory");
}
__device__ __forceinline__ void multimem_st_v4(float *mc, float4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}

// ---- packed FP32 pairs (Blackwell FADD2 / FMUL2 / FFMA2): one issue slot for two IEEE-rn operations ------------
struct f2 { unsigned long long v; };
__device__ __forceinline__ f2 pack2(float lo, float hi) {
  f2 r;
  asm("mov.b64 %0, {%1,%2};" : "=l"(r.v) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(f2 a, float &lo, float &hi) {
  asm("mov.b64 {%0,%1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a.v));
}
__device__ __forceinline__ f2 sub2(f2 a, f2 b) {
  f2 r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
  return r;
}
__device__ __forceinline__ f2 add2(f2 a, f2 b) {
  f2 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
  return r;
}
__device__ __forceinline__ f2 mul2(f2 a, f2 b) {
  f2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
  return r;
}
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) {
  f2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r.v) : "l"(a.v), "l"(b.v), "l"(c.v));
  return r;
}

__device__ __forceinline__ float log_sigmoid(float x) {     // F.logsigmoid: min(x,0) - log1p(exp(-|x|))
  return fminf(x, 0.f) - log1pf(expf(-fabsf(x)));
}
__device__ __forceinline__ float sigmoid(float x) {
  float e = expf(-fabsf(x));
  return x >= 0.f ? 1.f / (1.f + e) : e / (1.f + e);
}
// 2^x and 1/x on the MUFU pipe, one instruction each; flush-to-zero (without it, ex2 is wrapped in a subnormal range
// check and two rescaling multiplies)
__device__ __forceinline__ float ex2_ftz(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float rcp_ftz(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
constexpr float kLog2e = 1.44269504088896341f;
// sigmoid on the MUFU pipe (ex2 + rcp, ~2^-21 relative): the per-candidate softmax weight of the train kernel sits on the
// warp's serial path, where the IEEE division of sigmoid() costs ~40 cycles of latency
__device__ __forceinline__ float sigmoid_fast(float x) {
  const float e = ex2_ftz(-kLog2e * fabsf(x));
  const float r = rcp_ftz(1.f + e);
  return x >= 0.f ? r : e * r;
}
#endif

}  // namespace kge
