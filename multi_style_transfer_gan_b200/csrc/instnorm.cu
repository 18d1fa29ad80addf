// InstanceNorm2d (eps 1e-5, biased variance) on NHWC tensors: statistics, fused apply (+ optional affine -- a blend of
// per-style gammas / betas shared by the batch, or a per-image table -- activation, residual add) and backward.
// Bandwidth-bound: 16-byte vector accesses, per-thread channel groups fixed across the pixel loop
// (so scale/shift live in registers), block reduction in shared memory, one atomic per
// (block, channel).   Reference: nn.InstanceNorm2d at enhanced_generator.py:54..129, 242..263.
#include <stdlib.h>

#include "common.cuh"

namespace msg {
namespace {

template <typename T> struct Vec;
template <> struct Vec<float> { static constexpr int W = 4; };
template <> struct Vec<__nv_bfloat16> { static constexpr int W = 8; };

template <int W> struct VecIO;
template <> struct VecIO<4> {
  static __device__ __forceinline__ void ld(const float* p, float (&v)[4]) { load4(p, v); }
  static __device__ __forceinline__ void st(float* p, const float (&v)[4]) { store4(p, v); }
};
template <> struct VecIO<8> {
  static __device__ __forceinline__ void ld(const __nv_bfloat16* p, float (&v)[8]) {
    uint4 t = *reinterpret_cast<const uint4*>(p);
    unpack8(t, v);
  }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, const float (&v)[8]) {
    *reinterpret_cast<uint4*>(p) = pack8(v);
  }
};

constexpr int TPB = 256;

// ---- statistics -----------------------------------------------------------------------------
// x: [N][HW][C]; requires C % W == 0 and (TPB*W) % C == 0 (C a power of two <= TPB*W).
template <typename T>
__global__ void __launch_bounds__(TPB)
in_stats_kernel(const T* __restrict__ x, long long HW, int C, double* __restrict__ stats) {
  constexpr int W = Vec<T>::W;
  __shared__ float red[TPB][2 * W + 1];
  const int n = blockIdx.y;
  const long long nvec = HW * C / W;                       // vectors in this image
  const T* xn = x + (size_t)n * HW * C;
  float s[W], ss[W];
#pragma unroll
  for (int e = 0; e < W; ++e) { s[e] = 0.f; ss[e] = 0.f; }
  const long long stride = (long long)gridDim.x * TPB;
  for (long long v = (long long)blockIdx.x * TPB + threadIdx.x; v < nvec; v += stride) {
    float t[W];
    VecIO<W>::ld(xn + v * W, t);
#pragma unroll
    for (int e = 0; e < W; ++e) { s[e] += t[e]; ss[e] = fmaf(t[e], t[e], ss[e]); }
  }
#pragma unroll
  for (int e = 0; e < W; ++e) { red[threadIdx.x][e] = s[e]; red[threadIdx.x][W + e] = ss[e]; }
  __syncthreads();
  const int groups = C / W;            // distinct channel groups; thread t owns group t % groups
  for (int c = threadIdx.x; c < C; c += TPB) {
    int g = c / W, e = c - g * W;
    float ts = 0.f, tss = 0.f;
    for (int t = g; t < TPB; t += groups) { ts += red[t][e]; tss += red[t][W + e]; }
    double* st = stats + ((size_t)n * C + c) * 2;
    atomicAdd(st, (double)ts);
    atomicAdd(st + 1, (double)tss);
  }
}

// generic fallback: one block per (n, c) plane
template <typename T>
__global__ void __launch_bounds__(TPB)
in_stats_generic_kernel(const T* __restrict__ x, long long HW, int C, double* __restrict__ stats) {
  __shared__ float rs[TPB / 32], rss[TPB / 32];
  const int n = blockIdx.y, c = blockIdx.x;
  const T* xp = x + (size_t)n * HW * C + c;
  float s = 0.f, ss = 0.f;
  for (long long p = threadIdx.x; p < HW; p += TPB) {
    float v = to_f<T>(xp[(size_t)p * C]);
    s += v; ss = fmaf(v, v, ss);
  }
  s = warp_sum(s); ss = warp_sum(ss);
  if ((threadIdx.x & 31) == 0) { rs[threadIdx.x >> 5] = s; rss[threadIdx.x >> 5] = ss; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, b = 0.f;
    for (int i = 0; i < TPB / 32; ++i) { a += rs[i]; b += rss[i]; }
    double* st = stats + ((size_t)n * C + c) * 2;
    st[0] += (double)a; st[1] += (double)b;
  }
}

// ---- apply ----------------------------------------------------------------------------------
// The affine of channel c: with S > 0 the blend gamma = sum_s w[s] * gammas[s][c] (beta alike) as an fmaf chain over s in
// ascending order from 0 -- msg_style_affine's chain, so its per-image tables reproduce these bits --, else the (agamma,
// abeta) table at row offset `row` (in_affine: null = none).
__device__ __forceinline__ void blend_or_affine(int S, const float* gammas, const float* betas, const float* w, int C,
                                                const float* agamma, const float* abeta, size_t row, int c, float& g, float& b) {
  if (S > 0) {
    g = 0.f;
    b = 0.f;
    for (int s = 0; s < S; ++s) {
      g = fmaf(w[s], gammas[(size_t)s * C + c], g);
      b = fmaf(w[s], betas[(size_t)s * C + c], b);
    }
  } else {
    in_affine(agamma, abeta, row + c, g, b);
  }
}

template <typename T, bool FAST>
__global__ void __launch_bounds__(TPB)
in_apply_kernel(const T* __restrict__ x, const double* __restrict__ stats, long long HW, int C,
                int act, const T* __restrict__ residual, int S, const float* __restrict__ gammas,
                const float* __restrict__ betas, const float* __restrict__ w, const float* __restrict__ agamma,
                const float* __restrict__ abeta, int astride, T* __restrict__ y) {
  constexpr int W = FAST ? Vec<T>::W : 1;
  const int n = blockIdx.y;
  const double inv_hw = 1.0 / (double)HW;
  const size_t base = (size_t)n * HW * C;
  const long long nvec = HW * C / W;
  const long long stride = (long long)gridDim.x * TPB;
  long long v0 = (long long)blockIdx.x * TPB + threadIdx.x;
  float scale[W], shift[W];
  int c_cached = -1;
  for (long long v = v0; v < nvec; v += stride) {
    int c0 = (int)((v * W) % C);
    if (c0 != c_cached) {   // FAST: executes once (channel group is loop-invariant)
      c_cached = c0;
#pragma unroll
      for (int e = 0; e < W; ++e) {
        float g, b, mean, rstd;
        blend_or_affine(S, gammas, betas, w, C, agamma, abeta, (size_t)n * astride, c0 + e, g, b);
        in_scale_shift(stats + ((size_t)n * C + c0 + e) * 2, inv_hw, g, b, mean, rstd, scale[e], shift[e]);
      }
    }
    float t[W], r[W];
    if constexpr (FAST) {
      VecIO<Vec<T>::W>::ld(x + base + v * W, reinterpret_cast<float(&)[Vec<T>::W]>(t));
      if (residual) VecIO<Vec<T>::W>::ld(residual + base + v * W, reinterpret_cast<float(&)[Vec<T>::W]>(r));
    } else {
      t[0] = to_f<T>(x[base + v]);
      if (residual) r[0] = to_f<T>(residual[base + v]);
    }
#pragma unroll
    for (int e = 0; e < W; ++e) {
      float o = apply_act(fmaf(t[e], scale[e], shift[e]), act);
      if (residual) o += r[e];
      t[e] = o;
    }
    if constexpr (FAST) VecIO<Vec<T>::W>::st(y + base + v * W, reinterpret_cast<float(&)[Vec<T>::W]>(t));
    else y[base + v] = from_f<T>(t[0]);
  }
}

// ---- apply, fast path (C power of two): activation / residual are template parameters, the channel
// group of a thread is computed ONCE (no per-iteration 64-bit modulo), four independent 16-byte loads
// are in flight per thread per iteration.
template <typename T> __device__ __forceinline__ void raw_unpack(const uint4& t, float (&v)[Vec<T>::W]);
template <> __device__ __forceinline__ void raw_unpack<float>(const uint4& t, float (&v)[4]) {
  v[0] = __uint_as_float(t.x); v[1] = __uint_as_float(t.y); v[2] = __uint_as_float(t.z); v[3] = __uint_as_float(t.w);
}
template <> __device__ __forceinline__ void raw_unpack<__nv_bfloat16>(const uint4& t, float (&v)[8]) { unpack8(t, v); }
template <typename T> __device__ __forceinline__ uint4 raw_pack(const float (&v)[Vec<T>::W]);
template <> __device__ __forceinline__ uint4 raw_pack<float>(const float (&v)[4]) {
  return make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3]));
}
template <> __device__ __forceinline__ uint4 raw_pack<__nv_bfloat16>(const float (&v)[8]) { return pack8(v); }

template <typename T, int ACT, bool HAS_RES>
__global__ void __launch_bounds__(TPB, 3)
in_apply_fast_kernel(const T* __restrict__ x, const double* __restrict__ stats, long long HW, int C,
                     const T* __restrict__ residual, int S, const float* __restrict__ gammas,
                     const float* __restrict__ betas, const float* __restrict__ w, const float* __restrict__ agamma,
                     const float* __restrict__ abeta, int astride, T* __restrict__ y) {
  constexpr int W = Vec<T>::W;
  constexpr int U = 4;
  const int n = blockIdx.y;
  const double inv_hw = 1.0 / (double)HW;
  const size_t base = (size_t)n * HW * C;
  const long long nvec = HW * C / W;
  const long long stride = (long long)gridDim.x * TPB;
  const long long v0 = (long long)blockIdx.x * TPB + threadIdx.x;
  const int c0 = (int)((v0 * W) % C);          // loop-invariant: stride * W is a multiple of C
  float scale[W], shift[W];
#pragma unroll
  for (int e = 0; e < W; ++e) {
    float g, b, mean, rstd;
    blend_or_affine(S, gammas, betas, w, C, agamma, abeta, (size_t)n * astride, c0 + e, g, b);
    in_scale_shift(stats + ((size_t)n * C + c0 + e) * 2, inv_hw, g, b, mean, rstd, scale[e], shift[e]);
  }
  const T* xb = x + base;
  const T* rb = HAS_RES ? residual + base : nullptr;
  T* yb = y + base;
  // Loads stay RAW 16-byte vectors until they are consumed (unpacked floats would triple the registers that are live
  // while the loads are in flight): 2 x U x 16 B in flight per thread at 3 CTAs per SM.
  for (long long v = v0; v < nvec; v += U * stride) {
    uint4 tx[U], rx[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long vv = v + u * stride;
      if (vv < nvec) {
        tx[u] = *reinterpret_cast<const uint4*>(xb + vv * W);
        if (HAS_RES) rx[u] = *reinterpret_cast<const uint4*>(rb + vv * W);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long vv = v + u * stride;
      if (vv < nvec) {
        float t[W], r[W];
        raw_unpack<T>(tx[u], t);
        if (HAS_RES) raw_unpack<T>(rx[u], r);
#pragma unroll
        for (int e = 0; e < W; ++e) {
          float o = fmaf(t[e], scale[e], shift[e]);
          if (ACT == MSG_ACT_RELU) o = fmaxf(o, 0.f);
          else if (ACT == MSG_ACT_LRELU) o = o > 0.f ? o : 0.2f * o;
          if (HAS_RES) o += r[e];
          t[e] = o;
        }
        *reinterpret_cast<uint4*>(yb + vv * W) = raw_pack<T>(t);
      }
    }
  }
}

// ---- backward -------------------------------------------------------------------------------
// Per-channel constants of the backward.  xhat = (x - mean) * rstd.  With an affine (gamma, beta at element ai =
// n * img_stride + c) the activation's input is rebuilt as z = fmaf(x, scale, shift) by in_scale_shift: the arithmetic of
// the forward apply, so the ReLU / LeakyReLU mask is the sign of the stored forward output bit for bit.  Without one,
// z = xhat and scale = rstd.
template <bool AFFINE>
__device__ __forceinline__ void bwd_channel(const double* st, double inv_hw, const float* gamma, const float* beta, size_t ai,
                                            float& mean, float& rstd, float& scale, float& shift) {
  float g = 1.f, b = 0.f;
  if constexpr (AFFINE) { g = gamma[ai]; b = beta[ai]; }
  in_scale_shift(st, inv_hw, g, b, mean, rstd, scale, shift);
}

// g = dy * act'(z)
template <bool AFFINE>
__device__ __forceinline__ float bwd_grad(float t, float dy, float xh, float scale, float shift, int act) {
  return dy * act_grad_from_pre(AFFINE ? fmaf(t, scale, shift) : xh, act);
}

// pass 1: scratch[n][c] += (sum g, sum g*xhat); scratch rows are img_stride apart for a per-image affine, else C
template <typename T, bool FAST, bool AFFINE>
__global__ void __launch_bounds__(TPB)
in_bwd_reduce_kernel(const T* __restrict__ x, const double* __restrict__ stats,
                     const T* __restrict__ dy, long long HW, int C, int act, const float* __restrict__ gamma,
                     const float* __restrict__ beta, int astride, double* __restrict__ scratch) {
  constexpr int W = FAST ? Vec<T>::W : 1;
  __shared__ float red[TPB][2 * W + 1];
  const int n = blockIdx.y;
  const double inv_hw = 1.0 / (double)HW;
  const size_t base = (size_t)n * HW * C;
  const int sstride = astride ? astride : C;      // sums rows follow a per-image affine table
  if constexpr (FAST) {
    const long long nvec = HW * C / W;
    const long long stride = (long long)gridDim.x * TPB;
    long long v0 = (long long)blockIdx.x * TPB + threadIdx.x;
    float mean[W], rstd[W], scale[W], shift[W], sg[W], sgx[W];
    int c0 = (int)((v0 * W) % C);
#pragma unroll
    for (int e = 0; e < W; ++e) {
      bwd_channel<AFFINE>(stats + ((size_t)n * C + c0 + e) * 2, inv_hw, gamma, beta, (size_t)n * astride + c0 + e, mean[e], rstd[e], scale[e], shift[e]);
      sg[e] = 0.f; sgx[e] = 0.f;
    }
    constexpr int U = 4;          // 2 x U raw 16-byte loads in flight per thread (unpacked only when consumed)
    for (long long v = v0; v < nvec; v += U * stride) {
      uint4 tx[U], gx[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long vv = v + u * stride;
        if (vv < nvec) {
          tx[u] = *reinterpret_cast<const uint4*>(x + base + vv * W);
          gx[u] = *reinterpret_cast<const uint4*>(dy + base + vv * W);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (v + u * stride < nvec) {
          float t[Vec<T>::W], g[Vec<T>::W];
          raw_unpack<T>(tx[u], t);
          raw_unpack<T>(gx[u], g);
#pragma unroll
          for (int e = 0; e < W; ++e) {
            float xh = (t[e] - mean[e]) * rstd[e];
            float gg = bwd_grad<AFFINE>(t[e], g[e], xh, scale[e], shift[e], act);
            sg[e] += gg; sgx[e] = fmaf(gg, xh, sgx[e]);
          }
        }
      }
    }
#pragma unroll
    for (int e = 0; e < W; ++e) { red[threadIdx.x][e] = sg[e]; red[threadIdx.x][W + e] = sgx[e]; }
    __syncthreads();
    const int groups = C / W;
    for (int c = threadIdx.x; c < C; c += TPB) {
      int gi = c / W, e = c - gi * W;
      float a = 0.f, b = 0.f;
      for (int t = gi; t < TPB; t += groups) { a += red[t][e]; b += red[t][W + e]; }
      double* sc = scratch + ((size_t)n * sstride + c) * 2;
      atomicAdd(sc, (double)a);
      atomicAdd(sc + 1, (double)b);
    }
  } else {
    // generic: grid.x == C, one block per plane
    const int c = blockIdx.x;
    float mean, rstd, scale, shift;
    bwd_channel<AFFINE>(stats + ((size_t)n * C + c) * 2, inv_hw, gamma, beta, (size_t)n * astride + c, mean, rstd, scale, shift);
    float sg = 0.f, sgx = 0.f;
    for (long long p = threadIdx.x; p < HW; p += TPB) {
      float t = to_f<T>(x[base + (size_t)p * C + c]);
      float xh = (t - mean) * rstd;
      float gg = bwd_grad<AFFINE>(t, to_f<T>(dy[base + (size_t)p * C + c]), xh, scale, shift, act);
      sg += gg; sgx = fmaf(gg, xh, sgx);
    }
    sg = warp_sum(sg); sgx = warp_sum(sgx);
    if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5][0] = sg; red[threadIdx.x >> 5][1] = sgx; }
    __syncthreads();
    if (threadIdx.x == 0) {
      float a = 0.f, b = 0.f;
      for (int i = 0; i < TPB / 32; ++i) { a += red[i][0]; b += red[i][1]; }
      double* sc = scratch + ((size_t)n * sstride + c) * 2;
      sc[0] += (double)a; sc[1] += (double)b;
    }
  }
}

// pass 2: dx = gamma * rstd * (g - mean(g) - xhat * mean(g*xhat)), the means taken from scratch / HW
template <typename T, bool FAST, bool AFFINE>
__global__ void __launch_bounds__(TPB)
in_bwd_apply_kernel(const T* __restrict__ x, const double* __restrict__ stats,
                    const T* __restrict__ dy, long long HW, int C, int act, const float* __restrict__ gamma,
                    const float* __restrict__ beta, int astride, const double* __restrict__ scratch, T* __restrict__ dx) {
  constexpr int W = FAST ? Vec<T>::W : 1;
  const int n = blockIdx.y;
  const double inv_hw = 1.0 / (double)HW;
  const size_t base = (size_t)n * HW * C;
  const long long nvec = HW * C / W;
  const long long stride = (long long)gridDim.x * TPB;
  long long v0 = (long long)blockIdx.x * TPB + threadIdx.x;
  const int sstride = astride ? astride : C;
  float mean[W], rstd[W], scale[W], shift[W], mg[W], mgx[W];
  if constexpr (FAST) {
    // channel group of a thread is loop-invariant (stride * W is a multiple of C); 2 x U raw loads in flight per thread
    const int c0 = (int)((v0 * W) % C);
#pragma unroll
    for (int e = 0; e < W; ++e) {
      bwd_channel<AFFINE>(stats + ((size_t)n * C + c0 + e) * 2, inv_hw, gamma, beta, (size_t)n * astride + c0 + e, mean[e], rstd[e], scale[e], shift[e]);
      const double* sc = scratch + ((size_t)n * sstride + c0 + e) * 2;
      mg[e] = (float)(sc[0] * inv_hw); mgx[e] = (float)(sc[1] * inv_hw);
    }
    constexpr int U = 4;
    for (long long v = v0; v < nvec; v += U * stride) {
      uint4 tx[U], gx[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long vv = v + u * stride;
        if (vv < nvec) {
          tx[u] = *reinterpret_cast<const uint4*>(x + base + vv * W);
          gx[u] = *reinterpret_cast<const uint4*>(dy + base + vv * W);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long vv = v + u * stride;
        if (vv < nvec) {
          float t[Vec<T>::W], g[Vec<T>::W];
          raw_unpack<T>(tx[u], t);
          raw_unpack<T>(gx[u], g);
#pragma unroll
          for (int e = 0; e < W; ++e) {
            float xh = (t[e] - mean[e]) * rstd[e];
            float gg = bwd_grad<AFFINE>(t[e], g[e], xh, scale[e], shift[e], act);
            t[e] = scale[e] * (gg - mg[e] - xh * mgx[e]);
          }
          *reinterpret_cast<uint4*>(dx + base + vv * W) = raw_pack<T>(t);
        }
      }
    }
    return;
  }
  int c_cached = -1;
  for (long long v = v0; v < nvec; v += stride) {
    int c0 = (int)((v * W) % C);
    if (c0 != c_cached) {
      c_cached = c0;
#pragma unroll
      for (int e = 0; e < W; ++e) {
        bwd_channel<AFFINE>(stats + ((size_t)n * C + c0 + e) * 2, inv_hw, gamma, beta, (size_t)n * astride + c0 + e, mean[e], rstd[e], scale[e], shift[e]);
        const double* sc = scratch + ((size_t)n * sstride + c0 + e) * 2;
        mg[e] = (float)(sc[0] * inv_hw); mgx[e] = (float)(sc[1] * inv_hw);
      }
    }
    float t[W], g[W];
    if constexpr (FAST) {
      VecIO<Vec<T>::W>::ld(x + base + v * W, reinterpret_cast<float(&)[Vec<T>::W]>(t));
      VecIO<Vec<T>::W>::ld(dy + base + v * W, reinterpret_cast<float(&)[Vec<T>::W]>(g));
    } else {
      t[0] = to_f<T>(x[base + v]); g[0] = to_f<T>(dy[base + v]);
    }
#pragma unroll
    for (int e = 0; e < W; ++e) {
      float xh = (t[e] - mean[e]) * rstd[e];
      float gg = bwd_grad<AFFINE>(t[e], g[e], xh, scale[e], shift[e], act);
      t[e] = scale[e] * (gg - mg[e] - xh * mgx[e]);
    }
    if constexpr (FAST) VecIO<Vec<T>::W>::st(dx + base + v * W, reinterpret_cast<float(&)[Vec<T>::W]>(t));
    else dx[base + v] = from_f<T>(t[0]);
  }
}

template <typename T>
bool fast_ok(int C, long long HW) {
  constexpr int W = Vec<T>::W;
  return C % W == 0 && (TPB * W) % C == 0;
}

unsigned blocks_per_image(int N, long long nvec) {
  long long want = (8LL * sm_count() + N - 1) / N;
  long long maxb = (nvec + TPB - 1) / TPB;
  if (want > maxb) want = maxb;
  if (want < 1) want = 1;
  return (unsigned)want;
}

template <typename T>
int stats_impl(const T* x, int N, long long HW, int C, double* stats, cudaStream_t st) {
  if (fast_ok<T>(C, HW)) {
    dim3 grid(blocks_per_image(N, HW * C / Vec<T>::W), N);
    in_stats_kernel<T><<<grid, TPB, 0, st>>>(x, HW, C, stats);
  } else {
    dim3 grid(C, N);
    in_stats_generic_kernel<T><<<grid, TPB, 0, st>>>(x, HW, C, stats);
  }
  return check_launch("in_stats_kernel");
}

template <typename T>
int apply_impl(const T* x, const double* stats, int N, long long HW, int C, int act, const T* res,
               int S, const float* gammas, const float* betas, const float* w, const float* agamma, const float* abeta,
               int astride, T* y, cudaStream_t st) {
  if (fast_ok<T>(C, HW)) {
    const long long nvec = HW * C / Vec<T>::W;
    static const int ctas_per_sm = [] { const char* e = getenv("MSG_IN_CTAS"); return e ? atoi(e) : 12; }();
    // CTAs per SM over the whole launch (3 resident at 80 registers; measured plateau from 8 up on 537 MB tensors), but
    // at least 32 vectors per thread: every thread pays an fp64 statistics finalisation for its 8 channels up front
    long long total_ctas = (long long)ctas_per_sm * sm_count();
    const long long by_work = ((long long)N * nvec) / (TPB * 32);
    if (total_ctas > by_work) total_ctas = by_work > 4LL * sm_count() ? by_work : 4LL * sm_count();
    long long want = (total_ctas + N - 1) / N;
    long long maxb = (nvec + TPB * 4 - 1) / (TPB * 4);         // >= 4 vectors per thread
    if (want > maxb) want = maxb;
    if (want < 1) want = 1;
    dim3 grid((unsigned)want, N);
#define MSG_IN_APPLY(ACT, RES) in_apply_fast_kernel<T, ACT, RES><<<grid, TPB, 0, st>>>(x, stats, HW, C, res, S, gammas, betas, w, agamma, abeta, astride, y)
    if (res) {
      if (act == MSG_ACT_RELU) MSG_IN_APPLY(MSG_ACT_RELU, true);
      else if (act == MSG_ACT_LRELU) MSG_IN_APPLY(MSG_ACT_LRELU, true);
      else MSG_IN_APPLY(MSG_ACT_NONE, true);
    } else {
      if (act == MSG_ACT_RELU) MSG_IN_APPLY(MSG_ACT_RELU, false);
      else if (act == MSG_ACT_LRELU) MSG_IN_APPLY(MSG_ACT_LRELU, false);
      else MSG_IN_APPLY(MSG_ACT_NONE, false);
    }
#undef MSG_IN_APPLY
  } else {
    dim3 grid(blocks_per_image(N, HW * C), N);
    in_apply_kernel<T, false><<<grid, TPB, 0, st>>>(x, stats, HW, C, act, res, S, gammas, betas, w, agamma, abeta, astride, y);
  }
  return check_launch("in_apply_kernel");
}

template <typename T>
int bwd_reduce_impl(const T* x, const double* stats, const T* dy, int N, long long HW, int C, int act,
                    const float* gamma, const float* beta, int astride, double* scratch, cudaStream_t st) {
  if (astride == 0 || astride == C) cudaMemsetAsync(scratch, 0, (size_t)N * C * 2 * sizeof(double), st);
  else cudaMemset2DAsync(scratch, (size_t)astride * 2 * sizeof(double), 0, (size_t)C * 2 * sizeof(double), N, st);
  if (fast_ok<T>(C, HW)) {
    dim3 grid(blocks_per_image(N, HW * C / Vec<T>::W), N);
    if (gamma) in_bwd_reduce_kernel<T, true, true><<<grid, TPB, 0, st>>>(x, stats, dy, HW, C, act, gamma, beta, astride, scratch);
    else in_bwd_reduce_kernel<T, true, false><<<grid, TPB, 0, st>>>(x, stats, dy, HW, C, act, nullptr, nullptr, 0, scratch);
  } else {
    dim3 grid(C, N);
    if (gamma) in_bwd_reduce_kernel<T, false, true><<<grid, TPB, 0, st>>>(x, stats, dy, HW, C, act, gamma, beta, astride, scratch);
    else in_bwd_reduce_kernel<T, false, false><<<grid, TPB, 0, st>>>(x, stats, dy, HW, C, act, nullptr, nullptr, 0, scratch);
  }
  return check_launch("in_bwd_reduce_kernel");
}

template <typename T>
int bwd_apply_impl(const T* x, const double* stats, const T* dy, int N, long long HW, int C, int act,
                   const float* gamma, const float* beta, int astride, const double* scratch, T* dx, cudaStream_t st) {
  if (fast_ok<T>(C, HW)) {
    dim3 grid(blocks_per_image(N, HW * C / Vec<T>::W), N);
    if (gamma) in_bwd_apply_kernel<T, true, true><<<grid, TPB, 0, st>>>(x, stats, dy, HW, C, act, gamma, beta, astride, scratch, dx);
    else in_bwd_apply_kernel<T, true, false><<<grid, TPB, 0, st>>>(x, stats, dy, HW, C, act, nullptr, nullptr, 0, scratch, dx);
  } else {
    dim3 grid(blocks_per_image(N, HW * C), N);
    if (gamma) in_bwd_apply_kernel<T, false, true><<<grid, TPB, 0, st>>>(x, stats, dy, HW, C, act, gamma, beta, astride, scratch, dx);
    else in_bwd_apply_kernel<T, false, false><<<grid, TPB, 0, st>>>(x, stats, dy, HW, C, act, nullptr, nullptr, 0, scratch, dx);
  }
  return check_launch("in_bwd_apply_kernel");
}

template <typename T>
int bwd_impl(const T* x, const double* stats, const T* dy, int N, long long HW, int C, int act,
             double* scratch, T* dx, cudaStream_t st) {
  int rc = bwd_reduce_impl<T>(x, stats, dy, N, HW, C, act, nullptr, nullptr, 0, scratch, st);
  return rc ? rc : bwd_apply_impl<T>(x, stats, dy, N, HW, C, act, nullptr, nullptr, 0, scratch, dx, st);
}

}  // namespace
}  // namespace msg

using namespace msg;

extern "C" int msg_instnorm_stats(int dtype, const void* x, int N, long long HW, int C,
                                  double* stats, void* stream) {
  MSG_REQUIRE(N > 0 && HW > 0 && C > 0, MSG_ERR_SHAPE, "instnorm_stats: bad shape");
  if (dtype == MSG_F32) return stats_impl<float>((const float*)x, N, HW, C, stats, as_stream(stream));
  if (dtype == MSG_BF16) return stats_impl<__nv_bfloat16>((const __nv_bfloat16*)x, N, HW, C, stats, as_stream(stream));
  MSG_REQUIRE(false, MSG_ERR_UNSUPPORTED, "instnorm_stats: bad dtype");
}

extern "C" int msg_instnorm_apply_affine(int dtype, const void* x, const double* stats, int N, long long HW, int C, int act,
                                         const void* residual, int S, const float* gammas, const float* betas, const float* w,
                                         const float* gamma, const float* beta, int img_stride, void* y, void* stream) {
  MSG_REQUIRE(N > 0 && HW > 0 && C > 0, MSG_ERR_SHAPE, "instnorm_apply: bad shape");
  MSG_REQUIRE(act == MSG_ACT_NONE || act == MSG_ACT_RELU || act == MSG_ACT_LRELU, MSG_ERR_UNSUPPORTED, "instnorm_apply: bad act");
  MSG_REQUIRE(S == 0 || (gammas && betas && w), MSG_ERR_SHAPE, "instnorm_apply: S>0 needs gammas/betas/w");
  MSG_REQUIRE((gamma == nullptr) == (beta == nullptr), MSG_ERR_SHAPE, "instnorm_apply: gamma and beta go together");
  MSG_REQUIRE(gamma == nullptr || S == 0, MSG_ERR_SHAPE, "instnorm_apply: a style blend (S > 0) and an affine table exclude each other");
  MSG_REQUIRE(img_stride == 0 || img_stride >= C, MSG_ERR_SHAPE, "instnorm_apply: img_stride must be 0 or >= C");
  if (dtype == MSG_F32)
    return apply_impl<float>((const float*)x, stats, N, HW, C, act, (const float*)residual, S, gammas, betas, w, gamma, beta, img_stride,
                             (float*)y, as_stream(stream));
  if (dtype == MSG_BF16)
    return apply_impl<__nv_bfloat16>((const __nv_bfloat16*)x, stats, N, HW, C, act, (const __nv_bfloat16*)residual, S, gammas, betas, w,
                                     gamma, beta, img_stride, (__nv_bfloat16*)y, as_stream(stream));
  MSG_REQUIRE(false, MSG_ERR_UNSUPPORTED, "instnorm_apply: bad dtype");
}

extern "C" int msg_instnorm_apply(int dtype, const void* x, const double* stats, int N, long long HW,
                                  int C, int act, const void* residual, int S, const float* gammas,
                                  const float* betas, const float* w, void* y, void* stream) {
  return msg_instnorm_apply_affine(dtype, x, stats, N, HW, C, act, residual, S, gammas, betas, w, nullptr, nullptr, 0, y, stream);
}

extern "C" int msg_instnorm_bwd(int dtype, const void* x, const double* stats, const void* dy, int N,
                                long long HW, int C, int act, double* scratch, void* dx, void* stream) {
  MSG_REQUIRE(N > 0 && HW > 0 && C > 0, MSG_ERR_SHAPE, "instnorm_bwd: bad shape");
  MSG_REQUIRE(act == MSG_ACT_NONE || act == MSG_ACT_RELU || act == MSG_ACT_LRELU, MSG_ERR_UNSUPPORTED, "instnorm_bwd: bad act");
  if (dtype == MSG_F32)
    return bwd_impl<float>((const float*)x, stats, (const float*)dy, N, HW, C, act, scratch, (float*)dx, as_stream(stream));
  if (dtype == MSG_BF16)
    return bwd_impl<__nv_bfloat16>((const __nv_bfloat16*)x, stats, (const __nv_bfloat16*)dy, N, HW, C, act, scratch, (__nv_bfloat16*)dx, as_stream(stream));
  MSG_REQUIRE(false, MSG_ERR_UNSUPPORTED, "instnorm_bwd: bad dtype");
}

extern "C" int msg_instnorm_bwd_reduce_affine(int dtype, const void* x, const double* stats, const void* dy, int N, long long HW, int C,
                                              int act, const float* gamma, const float* beta, int img_stride, double* sums,
                                              void* stream) {
  MSG_REQUIRE(N > 0 && HW > 0 && C > 0, MSG_ERR_SHAPE, "instnorm_bwd_reduce: bad shape");
  MSG_REQUIRE(act == MSG_ACT_NONE || act == MSG_ACT_RELU || act == MSG_ACT_LRELU, MSG_ERR_UNSUPPORTED, "instnorm_bwd_reduce: bad act");
  MSG_REQUIRE((gamma == nullptr) == (beta == nullptr), MSG_ERR_SHAPE, "instnorm_bwd_reduce: gamma and beta go together");
  MSG_REQUIRE(img_stride == 0 || (gamma != nullptr && img_stride >= C), MSG_ERR_SHAPE, "instnorm_bwd_reduce: img_stride must be 0 or >= C");
  if (dtype == MSG_F32)
    return bwd_reduce_impl<float>((const float*)x, stats, (const float*)dy, N, HW, C, act, gamma, beta, img_stride, sums, as_stream(stream));
  if (dtype == MSG_BF16)
    return bwd_reduce_impl<__nv_bfloat16>((const __nv_bfloat16*)x, stats, (const __nv_bfloat16*)dy, N, HW, C, act, gamma, beta, img_stride,
                                          sums, as_stream(stream));
  MSG_REQUIRE(false, MSG_ERR_UNSUPPORTED, "instnorm_bwd_reduce: bad dtype");
}

extern "C" int msg_instnorm_bwd_reduce(int dtype, const void* x, const double* stats, const void* dy, int N,
                                       long long HW, int C, int act, const float* gamma, const float* beta,
                                       double* sums, void* stream) {
  return msg_instnorm_bwd_reduce_affine(dtype, x, stats, dy, N, HW, C, act, gamma, beta, 0, sums, stream);
}

extern "C" int msg_instnorm_bwd_apply_affine(int dtype, const void* x, const double* stats, const void* dy, int N, long long HW, int C,
                                             int act, const float* gamma, const float* beta, int img_stride, const double* sums,
                                             void* dx, void* stream) {
  MSG_REQUIRE(N > 0 && HW > 0 && C > 0, MSG_ERR_SHAPE, "instnorm_bwd_apply: bad shape");
  MSG_REQUIRE(act == MSG_ACT_NONE || act == MSG_ACT_RELU || act == MSG_ACT_LRELU, MSG_ERR_UNSUPPORTED, "instnorm_bwd_apply: bad act");
  MSG_REQUIRE((gamma == nullptr) == (beta == nullptr), MSG_ERR_SHAPE, "instnorm_bwd_apply: gamma and beta go together");
  MSG_REQUIRE(img_stride == 0 || (gamma != nullptr && img_stride >= C), MSG_ERR_SHAPE, "instnorm_bwd_apply: img_stride must be 0 or >= C");
  if (dtype == MSG_F32)
    return bwd_apply_impl<float>((const float*)x, stats, (const float*)dy, N, HW, C, act, gamma, beta, img_stride, sums, (float*)dx,
                                 as_stream(stream));
  if (dtype == MSG_BF16)
    return bwd_apply_impl<__nv_bfloat16>((const __nv_bfloat16*)x, stats, (const __nv_bfloat16*)dy, N, HW, C, act, gamma, beta, img_stride,
                                         sums, (__nv_bfloat16*)dx, as_stream(stream));
  MSG_REQUIRE(false, MSG_ERR_UNSUPPORTED, "instnorm_bwd_apply: bad dtype");
}

extern "C" int msg_instnorm_bwd_apply(int dtype, const void* x, const double* stats, const void* dy, int N,
                                      long long HW, int C, int act, const float* gamma, const float* beta,
                                      const double* sums, void* dx, void* stream) {
  return msg_instnorm_bwd_apply_affine(dtype, x, stats, dy, N, HW, C, act, gamma, beta, 0, sums, dx, stream);
}
