// C-ABI glue: error reporting, device capability check, conv dispatch (tcgen05 vs SIMT engine).
#include <stdarg.h>

#include "common.cuh"

namespace msg {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return MSG_ERR_CUDA;
  }
  return MSG_OK;
}

// immutable per-device capability cache (the only global state)
struct DevInfo { int major = -1, minor = 0, sms = 0; };
static DevInfo g_dev[64];
static const DevInfo& dev_info() {
  int dev = 0;
  cudaGetDevice(&dev);
  DevInfo& d = g_dev[dev & 63];
  if (d.major < 0) {
    int major = 0, minor = 0, sms = 0;
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    d.minor = minor; d.sms = sms > 0 ? sms : 148;
    d.major = major;
  }
  return d;
}
int sm_count() { return dev_info().sms; }

int conv_validate(const msg_conv_desc* d);
int conv2d_simt(const msg_conv_desc* d, const void* x, const void* w, const float* bias, void* y,
                double* stats, const double* in_stats, cudaStream_t st);
bool conv2d_tma_supported(const msg_conv_desc* d, const void* x, const void* w, const void* y);
int conv2d_tma(const msg_conv_desc* d, const void* x, const void* w, const float* bias, void* y,
               double* stats, const double* in_stats, const float* in_gamma, const float* in_beta, int in_img_stride, cudaStream_t st);
bool conv2d_tc_supported(const msg_conv_desc* d, const void* x, const void* w, const void* y);
int conv2d_tc(const msg_conv_desc* d, const void* x, const void* w, const float* bias, void* y,
              double* stats, const double* in_stats, cudaStream_t st);

bool conv2d_dot_supported(const msg_conv_desc* d, const void* x, const void* w);
int conv2d_dot(const msg_conv_desc* d, const void* x, const void* w, const float* bias, void* y, cudaStream_t st);

int conv2d_dispatch(const msg_conv_desc* d, const void* x, const void* w, const float* bias, void* y,
                    double* stats, const double* in_stats, cudaStream_t st) {
  int rc = conv_validate(d);
  if (rc) return rc;
  MSG_REQUIRE(!(d->flags & MSG_CONV_STATS) || stats != nullptr, MSG_ERR_SHAPE, "conv: MSG_CONV_STATS without a stats buffer");
  MSG_REQUIRE(!(d->flags & MSG_CONV_IN_NORM) || in_stats != nullptr, MSG_ERR_SHAPE, "conv: MSG_CONV_IN_NORM without in_stats");
  if (!(d->flags & MSG_CONV_FORCE_SIMT)) {
    if (!(d->flags & MSG_CONV_FORCE_GATHER) && conv2d_dot_supported(d, x, w))
      return conv2d_dot(d, x, w, bias, y, st);                              // one useful GEMM column: warp-per-pixel dot products
    if (!(d->flags & MSG_CONV_FORCE_GATHER) && conv2d_tma_supported(d, x, w, y))
      return conv2d_tma(d, x, w, bias, y, stats, in_stats, nullptr, nullptr, 0, st);   // persistent TMA + tcgen05 kernel
    MSG_REQUIRE(!(d->flags & MSG_CONV_PER_IMAGE_W), MSG_ERR_UNSUPPORTED,
                "conv: MSG_CONV_PER_IMAGE_W needs the TMA kernel (bf16, Cin % 64 == 0, plane a multiple of 128 pixels)");
    if (conv2d_tc_supported(d, x, w, y))
      return conv2d_tc(d, x, w, bias, y, stats, in_stats, st);   // cp.async gather + tcgen05 kernel
  }
  MSG_REQUIRE(!(d->flags & MSG_CONV_PER_IMAGE_W), MSG_ERR_UNSUPPORTED, "conv: MSG_CONV_PER_IMAGE_W needs the TMA kernel");
  return conv2d_simt(d, x, w, bias, y, stats, in_stats, st);
}

}  // namespace msg

using namespace msg;

extern "C" const char* msg_last_error(void) { return g_err; }
extern "C" int msg_version(void) { return 100; }
extern "C" int msg_sm_count(void) { return sm_count(); }
extern "C" int msg_check_device(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  MSG_REQUIRE(e == cudaSuccess && n > 0, MSG_ERR_ARCH, "no CUDA device: %s", cudaGetErrorString(e));
  const DevInfo& d = dev_info();
  MSG_REQUIRE(d.major == 10, MSG_ERR_ARCH,
              "msg_b200 kernels are built for sm_100a only; device is sm_%d%d (no fallback)", d.major, d.minor);
  return MSG_OK;
}

extern "C" int msg_conv2d_path(const msg_conv_desc* d, const void* x, const void* w, const void* y) {
  MSG_REQUIRE(d != nullptr, MSG_ERR_SHAPE, "conv: null descriptor");
  int rc = conv_validate(d);
  if (rc) return rc;
  if (!(d->flags & MSG_CONV_FORCE_SIMT)) {
    if (!(d->flags & MSG_CONV_FORCE_GATHER) && conv2d_tma_supported(d, x, w, y)) return 2;
    if (conv2d_tc_supported(d, x, w, y)) return 1;
  }
  return 0;
}

extern "C" int msg_conv2d_affine(const msg_conv_desc* d, const void* x, const void* w, const float* bias, void* y, double* stats,
                                 const double* in_stats, const float* in_gamma, const float* in_beta, int in_img_stride, void* stream) {
  if (in_gamma == nullptr && in_beta == nullptr) return conv2d_dispatch(d, x, w, bias, y, stats, in_stats, as_stream(stream));
  // only the TMA kernel's transform warps apply an input affine: every other engine refuses one instead of dropping it
  MSG_REQUIRE(d != nullptr, MSG_ERR_SHAPE, "conv: null descriptor");
  int rc = conv_validate(d);
  if (rc) return rc;
  MSG_REQUIRE(in_gamma && in_beta && in_img_stride >= 0 && (d->flags & MSG_CONV_IN_NORM) && in_stats != nullptr, MSG_ERR_SHAPE,
              "conv: an input affine needs gamma, beta and MSG_CONV_IN_NORM with in_stats");
  MSG_REQUIRE(!(d->flags & MSG_CONV_STATS) || stats != nullptr, MSG_ERR_SHAPE, "conv: MSG_CONV_STATS without a stats buffer");
  MSG_REQUIRE(!(d->flags & (MSG_CONV_FORCE_SIMT | MSG_CONV_FORCE_GATHER)) && !conv2d_dot_supported(d, x, w) &&
              conv2d_tma_supported(d, x, w, y), MSG_ERR_SHAPE,
              "conv: an input affine runs only on the TMA kernel (bf16 1x1, Cin %% 64 == 0, tiles inside one image)");
  return conv2d_tma(d, x, w, bias, y, stats, in_stats, in_gamma, in_beta, in_img_stride, as_stream(stream));
}

extern "C" int msg_conv2d(const msg_conv_desc* d, const void* x, const void* w, const float* bias,
                          void* y, double* stats, const double* in_stats, void* stream) {
  return msg_conv2d_affine(d, x, w, bias, y, stats, in_stats, nullptr, nullptr, 0, stream);
}
