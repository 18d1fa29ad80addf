// Per-image InstanceNorm affine tables of a style-conditional generator (Dumoulin et al.'s conditional instance norm with a
// style mix): forward gamma_n[c] = sum_s w[n][s] * gammas[s][c] (beta alike), and the backward of that blend.
// Tiny and launch-bound: one thread per output element, one launch each for all the normalisation sites of a forward.
#include "common.cuh"

namespace msg {
namespace {

constexpr int TPB = 256;

// gamma_out[n][c] = fmaf chain over s in ascending order from 0: the chain msg_instnorm_apply runs over its own w[S], so a
// table row built from the same w reproduces that apply bit for bit
__global__ void __launch_bounds__(TPB)
style_affine_kernel(const float* __restrict__ w, int N, int S, const float* __restrict__ gammas, const float* __restrict__ betas,
                    int Ct, float* __restrict__ gamma_out, float* __restrict__ beta_out) {
  const long long i = (long long)blockIdx.x * TPB + threadIdx.x;
  if (i >= (long long)N * Ct) return;
  const int n = (int)(i / Ct), c = (int)(i - (long long)n * Ct);
  float g = 0.f, b = 0.f;
  for (int s = 0; s < S; ++s) {
    const float ws = w[(size_t)n * S + s];
    g = fmaf(ws, gammas[(size_t)s * Ct + c], g);
    b = fmaf(ws, betas[(size_t)s * Ct + c], b);
  }
  gamma_out[i] = g;
  beta_out[i] = b;
}

// dgammas[s][c] += sum_n w[n][s] * sums[n][c][1], dbetas[s][c] += sum_n w[n][s] * sums[n][c][0] (sums: the IN backward's
// per-(image, channel) (sum g, sum g * xhat) = (d beta_n, d gamma_n)), summed over n in ascending order in fp64
__global__ void __launch_bounds__(TPB)
style_affine_bwd_kernel(const double* __restrict__ sums, const float* __restrict__ w, int N, int S, int Ct,
                        float* __restrict__ dgammas, float* __restrict__ dbetas) {
  const long long i = (long long)blockIdx.x * TPB + threadIdx.x;
  if (i >= (long long)S * Ct) return;
  const int s = (int)(i / Ct), c = (int)(i - (long long)s * Ct);
  double dg = 0.0, db = 0.0;
  for (int n = 0; n < N; ++n) {
    const double ws = (double)w[(size_t)n * S + s];
    const double* sm = sums + ((size_t)n * Ct + c) * 2;
    db += ws * sm[0];
    dg += ws * sm[1];
  }
  dgammas[i] += (float)dg;
  dbetas[i] += (float)db;
}

unsigned blocks(long long n) { return (unsigned)((n + TPB - 1) / TPB); }

}  // namespace
}  // namespace msg

using namespace msg;

extern "C" int msg_style_affine(const float* w, int N, int S, const float* gammas, const float* betas, int Ct, float* gamma_out,
                                float* beta_out, void* stream) {
  MSG_REQUIRE(w && gammas && betas && gamma_out && beta_out, MSG_ERR_SHAPE, "style_affine: null pointer");
  MSG_REQUIRE(N > 0 && S > 0 && Ct > 0 && (long long)N * Ct < (1LL << 40), MSG_ERR_SHAPE, "style_affine: bad shape");
  style_affine_kernel<<<blocks((long long)N * Ct), TPB, 0, as_stream(stream)>>>(w, N, S, gammas, betas, Ct, gamma_out, beta_out);
  return check_launch("style_affine_kernel");
}

extern "C" int msg_style_affine_bwd(const double* sums, const float* w, int N, int S, int Ct, float* dgammas, float* dbetas,
                                    void* stream) {
  MSG_REQUIRE(sums && w && dgammas && dbetas, MSG_ERR_SHAPE, "style_affine_bwd: null pointer");
  MSG_REQUIRE(N > 0 && S > 0 && Ct > 0 && (long long)S * Ct < (1LL << 40), MSG_ERR_SHAPE, "style_affine_bwd: bad shape");
  style_affine_bwd_kernel<<<blocks((long long)S * Ct), TPB, 0, as_stream(stream)>>>(sums, w, N, S, Ct, dgammas, dbetas);
  return check_launch("style_affine_bwd_kernel");
}
