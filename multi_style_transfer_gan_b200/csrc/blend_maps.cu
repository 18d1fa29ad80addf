// Per-pixel multi-style blend (enhanced_local_style.py:126-176, 232-236): the style weights of each output pixel are sampled
// bilinearly from low-resolution weight maps, optionally normalised, and applied to every channel of the pixel; plus the
// separable Gaussian blur that feathers those maps.  Semantics in include/msg_b200.h.
#include <math.h>

#include "common.cuh"

namespace msg {
namespace {

constexpr int BM_TPB = 256;
constexpr int BM_MAX_STYLES = 8;
constexpr int BM_MAX_K = BM_MAX_STYLES + 1;
constexpr int GB_MAX_TAPS = 256;  // taps[0..r] of a symmetric kernel: radius <= 255

struct BlendMapsArgs {
  const float* src[BM_MAX_K];  // the S style outputs, then the input image when K == S+1 (map k weights plane k)
  const float* maps;  // [Bm][K][h][w]
  float* out;         // fp32 NCHW or null
  uint8_t* out_u8;    // uint8 NCHW or null
  int K, map_batch, h, w, N, C, H, W;
  int normalize, do_clip;
  float gain, lo, hi;
  float scale_h, scale_w;  // (float)h / H, (float)w / W
};

// F.interpolate(mode="bilinear", align_corners=False) source coordinate of output index `o`
__device__ __forceinline__ void src_index(float scale, int o, int n, int& i0, int& i1, float& t) {
  float s = fmaxf(scale * ((float)o + 0.5f) - 0.5f, 0.f);
  i0 = (int)s;
  i1 = min(i0 + 1, n - 1);
  t = s - (float)i0;
}

// Each thread owns V consecutive pixels of one row: it samples the K weights of each pixel once, then walks the C channels,
// reading the S style planes (and x) with one V-wide load per plane.  V = 4 needs W % 4 == 0 and 16-byte aligned planes.
// MK >= K bounds the planes: the K weights of V pixels live in registers, so K <= 4 (three styles and the input) gets its own
// instantiation instead of paying the registers of nine planes.  Without a minimum-blocks bound ptxas spills the MK = 9
// kernels (80 registers); with one the V = 4, MK = 4 kernel spills at 80 instead of fitting 64 (full occupancy) without it.
template <int V, int MK>
__global__ void __launch_bounds__(BM_TPB, MK <= 4 ? 0 : 2) blend_maps_kernel(BlendMapsArgs a) {
  const int groups = a.W / V;
  const long long total = (long long)a.N * a.H * groups;
  const long long plane = (long long)a.H * a.W;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
    const int j0 = (int)(g % groups) * V;
    const long long row = g / groups;
    const int i = (int)(row % a.H);
    const int n = (int)(row / a.H);

    int r0, r1;
    float ty;
    src_index(a.scale_h, i, a.h, r0, r1, ty);
    int c0[V], c1[V];
    float tx[V];
#pragma unroll
    for (int v = 0; v < V; ++v) src_index(a.scale_w, j0 + v, a.w, c0[v], c1[v], tx[v]);

    // sample: rows first (lerp between map rows r0 and r1 at both columns), then columns
    const float* mb = a.maps + (size_t)(a.map_batch == 1 ? 0 : n) * a.K * a.h * a.w;
    float m[MK][V];
#pragma unroll
    for (int k = 0; k < MK; ++k) {
      if (k < a.K) {
        const float* p0 = mb + ((size_t)k * a.h + r0) * a.w;
        const float* p1 = mb + ((size_t)k * a.h + r1) * a.w;
#pragma unroll
        for (int v = 0; v < V; ++v) {
          const float a0 = __ldg(p0 + c0[v]), b0 = __ldg(p1 + c0[v]);
          const float a1 = __ldg(p0 + c1[v]), b1 = __ldg(p1 + c1[v]);
          const float l = a0 + ty * (b0 - a0);
          const float r = a1 + ty * (b1 - a1);
          m[k][v] = l + tx[v] * (r - l);
        }
      } else {
#pragma unroll
        for (int v = 0; v < V; ++v) m[k][v] = 0.f;
      }
    }
    if (a.normalize) {
#pragma unroll
      for (int v = 0; v < V; ++v) {
        float sum = 0.f;
#pragma unroll
        for (int k = 0; k < MK; ++k)
          if (k < a.K) sum += m[k][v];
#pragma unroll
        for (int k = 0; k < MK; ++k) m[k][v] = sum != 0.f ? m[k][v] / sum : 0.f;
      }
    }
    const long long base = (long long)n * a.C * plane + (long long)i * a.W + j0;
    for (int c = 0; c < a.C; ++c) {
      const long long off = base + (long long)c * plane;
      float acc[V];
#pragma unroll
      for (int v = 0; v < V; ++v) acc[v] = 0.f;
      // the operation order of blend_kernel (elementwise.cu): styles in order, then x; constant maps equal to (w, w_x)
      // reproduce msg_blend_outputs bit for bit
#pragma unroll
      for (int k = 0; k < MK; ++k) {
        if (k < a.K) {
          float y[V];
          if constexpr (V == 4) load4(a.src[k] + off, y);
          else y[0] = a.src[k][off];
#pragma unroll
          for (int v = 0; v < V; ++v) acc[v] = fmaf(m[k][v], y[v], acc[v]);
        }
      }
      uint8_t u[V];
#pragma unroll
      for (int v = 0; v < V; ++v) {
        float t = acc[v] * a.gain;
        if (a.do_clip) t = fminf(fmaxf(t, a.lo), a.hi);
        acc[v] = t;
        u[v] = (uint8_t)(fminf(fmaxf((t + 1.f) * 0.5f, 0.f), 1.f) * 255.f);  // truncation, as blend_kernel
      }
      if (a.out) {
        if constexpr (V == 4) store4(a.out + off, acc);
        else a.out[off] = acc[0];
      }
      if (a.out_u8) {
        if constexpr (V == 4) *reinterpret_cast<uchar4*>(a.out_u8 + off) = make_uchar4(u[0], u[1], u[2], u[3]);
        else a.out_u8[off] = u[0];
      }
    }
  }
}

// half-sample-symmetric reflection (scipy.ndimage mode="reflect") of any index into [0, n)
__device__ __forceinline__ int reflect(int i, int n) {
  const int n2 = 2 * n;
  i %= n2;
  if (i < 0) i += n2;
  return i >= n ? n2 - 1 - i : i;
}

struct GaussTaps {
  float t[GB_MAX_TAPS];  // t[|d|], d in [-r, r]
};

// VERT: out[p][i][j] = sum_d taps[|d|] * in[p][reflect(i + d)][j]; otherwise the same along j.  Summed from d = -r up.
template <bool VERT>
__global__ void __launch_bounds__(BM_TPB) gauss_pass_kernel(const float* __restrict__ in, long long planes, int h, int w, int r,
                                                            GaussTaps taps, float* __restrict__ out) {
  const long long total = planes * h * w;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(idx % w);
    const long long t = idx / w;
    const int i = (int)(t % h);
    const float* src = in + (t / h) * h * w;
    float acc = 0.f;
    for (int d = -r; d <= r; ++d) {
      const float v = VERT ? src[(size_t)reflect(i + d, h) * w + j] : src[(size_t)i * w + reflect(j + d, w)];
      acc = fmaf(taps.t[d < 0 ? -d : d], v, acc);
    }
    out[idx] = acc;
  }
}

inline unsigned grid_for(long long n) {
  long long b = (n + BM_TPB - 1) / BM_TPB;
  const long long cap = 32LL * sm_count();
  return (unsigned)(b > cap ? cap : (b < 1 ? 1 : b));
}

inline bool aligned16(const void* p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace
}  // namespace msg

using namespace msg;

extern "C" int msg_blend_maps(const float* const* ys, int S, const float* x, const float* maps, int map_batch, int K, int h,
                              int w, int N, int C, int H, int W, int normalize, float gain, int do_clip, float clip_lo,
                              float clip_hi, float* out_f32, uint8_t* out_u8, void* stream) {
  MSG_REQUIRE(ys != nullptr && S >= 1 && S <= BM_MAX_STYLES, MSG_ERR_SHAPE, "blend_maps: S must be in [1,%d]", BM_MAX_STYLES);
  MSG_REQUIRE(N > 0 && C > 0 && H > 0 && W > 0, MSG_ERR_SHAPE, "blend_maps: empty image [%d,%d,%d,%d]", N, C, H, W);
  MSG_REQUIRE(K == S || K == S + 1, MSG_ERR_SHAPE, "blend_maps: K = %d maps for %d styles (need S or S+1)", K, S);
  MSG_REQUIRE(map_batch == 1 || map_batch == N, MSG_ERR_SHAPE, "blend_maps: map batch %d for %d images (need 1 or N)",
              map_batch, N);
  MSG_REQUIRE(h >= 1 && h <= H && w >= 1 && w <= W, MSG_ERR_SHAPE, "blend_maps: %dx%d maps for %dx%d images (need 1 <= map <= image)",
              h, w, H, W);
  MSG_REQUIRE(maps != nullptr && (out_f32 || out_u8), MSG_ERR_SHAPE, "blend_maps: null maps or no output");
  MSG_REQUIRE(K == S || x != nullptr, MSG_ERR_SHAPE, "blend_maps: K = S+1 maps need the input image x");
  BlendMapsArgs a;
  bool vec = W % 4 == 0 && aligned16(out_f32) && (reinterpret_cast<uintptr_t>(out_u8) & 3) == 0;
  for (int k = 0; k < BM_MAX_K; ++k) {
    a.src[k] = k < S ? ys[k] : (k < K ? x : nullptr);
    MSG_REQUIRE(k >= K || a.src[k] != nullptr, MSG_ERR_SHAPE, "blend_maps: style %d is null", k);
    vec = vec && aligned16(a.src[k]);
  }
  a.maps = maps;
  a.out = out_f32;
  a.out_u8 = out_u8;
  a.K = K; a.map_batch = map_batch; a.h = h; a.w = w; a.N = N; a.C = C; a.H = H; a.W = W;
  a.normalize = normalize != 0;
  a.do_clip = do_clip != 0;
  a.gain = gain; a.lo = clip_lo; a.hi = clip_hi;
  a.scale_h = (float)h / (float)H;
  a.scale_w = (float)w / (float)W;
  const long long pix = (long long)N * H * W;
  if (vec && K <= 4) blend_maps_kernel<4, 4><<<grid_for(pix / 4), BM_TPB, 0, as_stream(stream)>>>(a);
  else if (vec) blend_maps_kernel<4, BM_MAX_K><<<grid_for(pix / 4), BM_TPB, 0, as_stream(stream)>>>(a);
  else if (K <= 4) blend_maps_kernel<1, 4><<<grid_for(pix), BM_TPB, 0, as_stream(stream)>>>(a);
  else blend_maps_kernel<1, BM_MAX_K><<<grid_for(pix), BM_TPB, 0, as_stream(stream)>>>(a);
  return check_launch("blend_maps_kernel");
}

extern "C" int msg_gaussian_blur(const float* in, long long planes, int h, int w, float sigma, float* tmp, float* out,
                                 void* stream) {
  MSG_REQUIRE(in && tmp && out && planes > 0 && h > 0 && w > 0, MSG_ERR_SHAPE, "gaussian_blur: bad arguments");
  MSG_REQUIRE(isfinite(sigma) && sigma >= 0.f, MSG_ERR_SHAPE, "gaussian_blur: sigma must be finite and >= 0 (got %g)",
              (double)sigma);
  // scipy.ndimage.gaussian_filter(truncate=4.0): radius int(4 sigma + 0.5), taps exp(-x^2 / 2 sigma^2) normalised to sum 1
  const int r = (int)(4.0 * (double)sigma + 0.5);
  MSG_REQUIRE(r < GB_MAX_TAPS, MSG_ERR_SHAPE, "gaussian_blur: radius %d (sigma %g) exceeds %d", r, (double)sigma,
              GB_MAX_TAPS - 1);
  GaussTaps taps;
  double e[GB_MAX_TAPS], sum = 0.0;
  for (int d = 0; d <= r; ++d) {
    e[d] = r == 0 ? 1.0 : exp(-0.5 * (double)d * d / ((double)sigma * sigma));
    sum += d == 0 ? e[d] : 2.0 * e[d];
  }
  for (int d = 0; d < GB_MAX_TAPS; ++d) taps.t[d] = d <= r ? (float)(e[d] / sum) : 0.f;
  const long long total = planes * h * w;
  gauss_pass_kernel<true><<<grid_for(total), BM_TPB, 0, as_stream(stream)>>>(in, planes, h, w, r, taps, tmp);
  int rc = check_launch("gauss_pass_kernel<vertical>");
  if (rc != 0) return rc;
  gauss_pass_kernel<false><<<grid_for(total), BM_TPB, 0, as_stream(stream)>>>(tmp, planes, h, w, r, taps, out);
  return check_launch("gauss_pass_kernel<horizontal>");
}
