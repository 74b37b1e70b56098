// Shared device/host helpers for libtmf (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/tmf.h"

namespace tmf {

void set_error(const char* fmt, ...);

#define TMF_REQUIRE(cond, ...)      \
  do {                              \
    if (!(cond)) {                  \
      tmf::set_error(__VA_ARGS__);  \
      return TMF_E_INVALID;         \
    }                               \
  } while (0)

#define TMF_CUDA(expr)                                                              \
  do {                                                                              \
    cudaError_t _e = (expr);                                                        \
    if (_e != cudaSuccess) {                                                        \
      tmf::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return TMF_E_CUDA;                                                            \
    }                                                                               \
  } while (0)

#define TMF_LAUNCH_CHECK() TMF_CUDA(cudaGetLastError())

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline cudaStream_t as_stream(tmf_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }
inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

constexpr int kNumSMs = 148;  // B200

// blocks of a grid-stride launch that needs `blocks` to cover its range: at most per_sm resident per SM, the loop does the rest
inline unsigned grid_stride_blocks(int64_t blocks, int per_sm) {
  const int64_t cap = (int64_t)kNumSMs * per_sm;
  return (unsigned)(blocks < cap ? blocks : cap);
}

// ---- sub-warp "row groups": LPR lanes (power of two) cooperate on one embedding row,
//      each lane owning one float4 (128-bit) column slice.
template <int LPR>
__device__ __forceinline__ unsigned group_mask() {
  if constexpr (LPR == 32) {
    return 0xffffffffu;
  } else {
    const unsigned lane = threadIdx.x & 31u;
    return ((1u << LPR) - 1u) << (lane & ~(unsigned)(LPR - 1));
  }
}

template <int LPR>
__device__ __forceinline__ float group_sum(float v, unsigned mask) {
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o, LPR);
  return v;
}

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

__device__ __forceinline__ float dot4(const float4& a, const float4& b) {
  return fmaf(a.w, b.w, fmaf(a.z, b.z, fmaf(a.y, b.y, a.x * b.x)));
}

__device__ __forceinline__ void fma4(float4& acc, float c, const float4& r) {
  acc.x = fmaf(c, r.x, acc.x);
  acc.y = fmaf(c, r.y, acc.y);
  acc.z = fmaf(c, r.z, acc.z);
  acc.w = fmaf(c, r.w, acc.w);
}

// ---- packed fp32x2 arithmetic (sm_100: FADD2 / FFMA2, two IEEE fp32 results per issue slot)
__device__ __forceinline__ float2 fadd2(const float2 a, const float2 b) {
  float2 r;
  asm("{ .reg .b64 ra, rb, rc; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; add.rn.f32x2 rc, ra, rb; mov.b64 {%0,%1}, rc; }"
      : "=f"(r.x), "=f"(r.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return r;
}

__device__ __forceinline__ float2 ffma2(const float2 a, const float2 b, const float2 c) {
  float2 r;
  asm("{ .reg .b64 ra, rb, rc, rd; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; mov.b64 rc, {%6,%7};"
      " fma.rn.f32x2 rd, ra, rb, rc; mov.b64 {%0,%1}, rd; }"
      : "=f"(r.x), "=f"(r.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return r;
}

__device__ __forceinline__ float rcp_approx(float x) {  // MUFU.RCP, 1 ulp; callers guarantee a normal x
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// Keras Adam, step 1 from zero moments (a NEW optimizer every epoch, matrix_factorization.py:176), in the un-simplified
// m / v / alpha form in fp32 (SURVEY A.6).  One definition for the stand-alone update (tmf_adam1) and the update fused into
// the multi-GPU gradient exchange (tmf_peer_reduce_push): replicas must receive identical bits.
__device__ __forceinline__ float adam1_alpha(float lr) { return lr * sqrtf(1.0f - 0.999f) / (1.0f - 0.9f); }
__device__ __forceinline__ float adam1_apply(float w, float g, float alpha) {
  const float one_m_b1 = 1.0f - 0.9f;
  const float one_m_b2 = 1.0f - 0.999f;
  const float eps = 1e-7f;
  const float m = g * one_m_b1;
  const float v = (g * g) * one_m_b2;
  return w - __fdiv_rn(alpha * m, sqrtf(v) + eps);
}

// 16-byte global -> shared asynchronous copy (LDGSTS: no register staging); both addresses 16-byte aligned
__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gmem_src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

__device__ __forceinline__ void add4(float4& acc, const float4& r) {
  acc.x += r.x;
  acc.y += r.y;
  acc.z += r.z;
  acc.w += r.w;
}

}  // namespace tmf
