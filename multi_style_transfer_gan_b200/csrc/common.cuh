// Shared helpers for the msg_b200 kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/msg_b200.h"

namespace msg {

void set_error(const char* fmt, ...);
int check_launch(const char* what);  // cudaGetLastError -> MSG_ERR_CUDA

#define MSG_REQUIRE(cond, code, ...)   \
  do {                                 \
    if (!(cond)) {                     \
      ::msg::set_error(__VA_ARGS__);   \
      return (code);                   \
    }                                  \
  } while (0)

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

template <typename T>
__device__ __forceinline__ float to_f(T v);
template <>
__device__ __forceinline__ float to_f<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T>
__device__ __forceinline__ T from_f(float v);
template <>
__device__ __forceinline__ float from_f<float>(float v) { return v; }
template <>
__device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// 4-element vector access (16 B for fp32, 8 B for bf16). Pointers must be 4-element aligned.
__device__ __forceinline__ void load4(const float* p, float (&v)[4]) {
  float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void load4(const __nv_bfloat16* p, float (&v)[4]) {
  uint2 t = *reinterpret_cast<const uint2*>(p);
  __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&t.x);
  __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&t.y);
  v[0] = __low2float(a); v[1] = __high2float(a); v[2] = __low2float(b); v[3] = __high2float(b);
}
__device__ __forceinline__ void store4(float* p, const float (&v)[4]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
__device__ __forceinline__ void store4(__nv_bfloat16* p, const float (&v)[4]) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]);
  __nv_bfloat162 b = __floats2bfloat162_rn(v[2], v[3]);
  uint2 t;
  t.x = *reinterpret_cast<uint32_t*>(&a);
  t.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = t;
}

// 8 x bf16 <-> 8 floats (one 16-byte access)
__device__ __forceinline__ void unpack8(const uint4& t, float (&v)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
  for (int i = 0; i < 4; ++i) { v[2 * i] = __low2float(h[i]); v[2 * i + 1] = __high2float(h[i]); }
}
__device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
  uint4 t;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&t);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
  return t;
}

// Running sum kept as an unevaluated (hi, lo) pair of floats (Knuth TwoSum): ~2^-44 relative, in the 8 bytes of the double it
// replaces.  The conv epilogues add their fixed-order 32-row fp32 partial sums into per-warp running column sums once per tile;
// as fp64 adds those were the hottest stall of the 7x7 input conv's epilogue ("math pipe throttle" on the two DADDs: 26 % of
// all stall samples, ncu) -- B200's FP64 pipe is narrow.  The pair is converted to fp64 only when a CTA flushes an image.
__device__ __forceinline__ void f2sum_add(float2& s, float x) {
  const float a = s.x;
  const float t = __fadd_rn(a, x);
  const float bb = __fsub_rn(t, a);
  const float err = __fadd_rn(__fsub_rn(a, __fsub_rn(t, bb)), __fsub_rn(x, bb));
  s.x = t;
  s.y = __fadd_rn(s.y, err);
}
__device__ __forceinline__ double f2sum_value(float2 s) { return (double)s.x + (double)s.y; }

__device__ __forceinline__ float apply_act(float v, int act) {
  switch (act) {
    case MSG_ACT_RELU: return v > 0.f ? v : 0.f;
    case MSG_ACT_LRELU: return v > 0.f ? v : 0.2f * v;
    case MSG_ACT_TANH: return tanhf(v);
    default: return v;
  }
}
// derivative of act w.r.t. its input, expressed with the pre-activation value z
__device__ __forceinline__ float act_grad_from_pre(float z, int act) {
  switch (act) {
    case MSG_ACT_RELU: return z > 0.f ? 1.f : 0.f;
    case MSG_ACT_LRELU: return z > 0.f ? 1.f : 0.2f;
    default: return 1.f;
  }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

constexpr float kInEps = 1e-5f;

// raw plane sums (kept in fp64: E[x^2]-mean^2 then has no cancellation problem and the fp64 atomics
// make the statistics order-independent to ~1e-16) -> (mean, rstd) in fp32
__device__ __forceinline__ void finalize_stats(double s, double ss, double inv_hw, float& mean, float& rstd) {
  double m = s * inv_hw;
  double var = ss * inv_hw - m * m;
  var = var > 0.0 ? var : 0.0;
  mean = (float)m;
  rstd = (float)(1.0 / sqrt(var + (double)kInEps));
}

// The one place that turns statistics and an affine into the constants every InstanceNorm apply site uses,
// z = fmaf(x, scale, shift):  scale = rstd * gamma,  shift = beta - mean * scale.
// gamma = 1, beta = 0 (no affine) gives scale = rstd and shift = -mean * rstd bit for bit.
__device__ __forceinline__ void in_scale_shift(const double* st, double inv_hw, float gamma, float beta,
                                               float& mean, float& rstd, float& scale, float& shift) {
  finalize_stats(st[0], st[1], inv_hw, mean, rstd);
  scale = rstd * gamma;
  shift = beta - mean * scale;
}

// An affine is passed as (gamma, beta, img_stride): element ai = n * img_stride + c is indexed like the statistics it
// accompanies (channel offsets included); img_stride 0 is one [C] affine for the whole batch; a null gamma is no affine.
__device__ __forceinline__ void in_affine(const float* gamma, const float* beta, size_t ai, float& g, float& b) {
  g = 1.f;
  b = 0.f;
  if (gamma != nullptr) { g = gamma[ai]; b = beta[ai]; }
}

int sm_count();

// once-per-device latch for cudaFuncSetAttribute (a function attribute belongs to the current device's context, so a
// process-wide flag would leave the second GPU of a multi-device process without its shared-memory opt-in)
struct DeviceOnce {
  unsigned long long mask = 0;
  int dev = 0;
  bool needed() {
    cudaGetDevice(&dev);
    return !((__atomic_load_n(&mask, __ATOMIC_ACQUIRE) >> (dev & 63)) & 1ull);
  }
  void done() { __atomic_fetch_or(&mask, 1ull << (dev & 63), __ATOMIC_RELEASE); }
};

}  // namespace msg
