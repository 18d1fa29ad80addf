// The generator's output layer (enhanced_generator.py:130-133: Conv2d(c, 3, 7, padding 3) + Tanh) fused with the InstanceNorm + ReLU
// + residual of the MultiScaleBlock in front of it (enhanced_generator.py:78-84), as a ROW RING of tensor-memory accumulators
// (sm_100a, bf16 operands, fp32 accumulate; c = 64) -- the third member of the msb_ring.cu / convt_ring.cu family (shared mechanics in
// ring.cuh).
//
//   a2 = a1 + ReLU(IN(f))        f: raw output of the block's 1x1 fusion conv with its plane statistics, a1: the block's input
//   y  = tanh(conv7x7(a2) + b)   fp32 NCHW, 3 channels
//
// Until now that was an HBM-bound apply kernel (read f, read a1, write a2: 1.6 GB per 16 images at 512^2) followed by the taps-as-N
// kernel of conv_shift.cu, which re-reads every input row four times and shifts its accumulators through shared memory.  Here a CTA
// walks DOWN a 128-pixel column strip:
//   * the f and a1 row slabs [136 pixels x 64 ch] are loaded ONCE by TMA; four transform warps rewrite the f slab in place as the
//     bf16 operand a2 with the apply kernel's exact arithmetic (fmaf(f, rstd, -mean rstd), max 0, + a1, round to nearest), pixels
//     outside the plane forced to 0 (the conv's zero padding applies to a2, not to f): a2 never exists in HBM;
//   * input row r feeds the output rows r-3 .. r+3 (ky = 6..0), whose accumulators are adjacent 16-column slots (3 channels padded
//     to 16: N of an M = 128 tcgen05.mma is a multiple of 16) of a 32-slot ring: for each of the 7 horizontal taps (shifted views of the
//     slab) the 7 vertical taps are ONE MMA of N = 112 -- 28 MMAs per input row and K step instead of the 49 x (re-reads) of a
//     per-tap kernel, and no accumulator shifting in the epilogue;
//   * input row r completes output row r-3: four epilogue warps read its 3 live columns, zero the slot, add the bias, tanh, and
//     write the fp32 NCHW planes (consecutive lanes = consecutive pixels: full 128-byte lines).
// Schedule stated and run on tensors in slab.py (out7_ring_row_mmas) / tests/test_out7_ring_cpu.py.
//
//   warp 0      TMA producer: the weight stacks once, then the f and a1 slabs of one input row per stage
//   warp 1      MMA issuer (also allocates TMEM)
//   warps 4-7   epilogue
//   warps 8-11  transform
#include "ring.cuh"

namespace msg {
namespace {
using namespace ring;

constexpr int NCOL = 16;                // columns per row accumulator (3 output channels padded)
constexpr int SLOTS = 32;
constexpr int HV = 3;                   // input rows above / below a piece
constexpr uint32_t LEAD = 6;            // a slot is touched again 26 steps after its row completed: any lead <= NBAR would do
constexpr int W_ROWS = 7 * 128;         // per horizontal tap: 8 entries (7 vertical taps + one zero block) x 16 rows
constexpr int NTHREADS = 32 * 12;
constexpr int XF0 = 8;
// weights [7 kx][8 e][16 co][128 B] | stages [f slab | a1 slab]; full / empty / transformed per stage
__host__ __device__ constexpr Shape o7_shape() { return Shape{W_ROWS * 128, 2 * SLAB_BYTES, 0, 0, 3}; }

struct O7Params {
  int N, H, W;
  int segs;
  long long total_rows;
  int stages;
  const float* bias;                    // [3]
  const double* in_stats;               // [N][Cs_total][2] raw plane sums of f
  int Cs_total, cs_off;
  const float* in_gamma;                // optional affine of f's norm (common.cuh: in_affine), or null
  const float* in_beta;
  int in_img_stride;
  float* y;                             // fp32 NCHW [N][3][H][W]
};

__global__ void __launch_bounds__(NTHREADS, 1)
out7_ring_kernel(const __grid_constant__ CUtensorMap mapF, const __grid_constant__ CUtensorMap mapR,
                 const __grid_constant__ CUtensorMap mapB, const O7Params p) {
  constexpr Shape SH = o7_shape();
  using Walk = Pieces<1, HV>;
  extern __shared__ uint8_t smem_raw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const Smem sm(smem_raw, SH, p.stages);
  const Bars& bars = sm.b;
  const uint32_t tmem_base = prologue(sm, warp, lane, 1, 4, 4, &mapF, &mapR, &mapB);
  const Walk pieces(p.total_rows, p.H, p.segs);

  if (warp == 0) {
    if (lane == 0)
      producer(sm, pieces, p.H, &mapB, SH.w_bytes, 0, SH.stage_bytes, [&](const Walk& pc, int r, uint32_t dst, uint32_t bar) {
        tma_load_4d(dst, &mapF, bar, 0, pc.seg * BM - HALO, r, pc.img);
        tma_load_4d(dst + SLAB_BYTES, &mapR, bar, 0, pc.seg * BM - HALO, r, pc.img);
      });
  } else if (warp == 1) {
    const bool leader = elect_one();
    const uint32_t hi = (uint32_t)(make_sw128_desc(0) >> 32);
    const uint32_t b_base = sm.sB() >> 4;
    // (waits for the transform warps to have turned the landed f slab into the operand)
    issuer<LEAD, true>(bars, pieces, p.H, leader, [&](const Walk& pc, int r, int s) {
      const uint32_t a0 = sm.sA(s, SH.stage_bytes) >> 4;
      // entries e = 0..6 = output rows r-3 .. r+3 (ky = 6 - e); those of this piece are an interval of adjacent ring slots
      const int o_lo = r - 3 > pc.y0 ? r - 3 : pc.y0, o_hi = r + 3 < pc.y1 - 1 ? r + 3 : pc.y1 - 1;      // inclusive
      if (o_lo <= o_hi)
        runs(o_hi - o_lo + 1, o_lo & (SLOTS - 1), SLOTS, [&](int e, int nrun, int slot) {
          const uint32_t idesc = idesc_bf16(NCOL * nrun);
          const uint32_t dcol = tmem_base + (uint32_t)(slot * NCOL);
#pragma unroll
          for (int kx = 0; kx < 7; ++kx) {
            const uint32_t av = a0 + (uint32_t)((HALO + kx - 3) * 8);
            const uint32_t bv = b_base + (uint32_t)((kx * 128 + NCOL * (o_lo - (r - 3) + e)) * 8);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) umma_bf16_lo(dcol, av + (uint32_t)(2 * ks), bv + (uint32_t)(2 * ks), hi, idesc, true);
          }
        });
    });
  } else if (warp >= EPI0 && warp < XF0) {
    // ===================================== epilogue =====================================
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const float b0 = p.bias ? p.bias[0] : 0.f, b1 = p.bias ? p.bias[1] : 0.f, b2 = p.bias ? p.bias[2] : 0.f;
    uint32_t k = 0;
    const size_t plane = (size_t)p.H * p.W;
    for (Walk pc = pieces; pc.next();) {
      const int xcol = pc.seg * BM + row;
      const bool valid = xcol < p.W;
      for (int r = pc.r0; r < pc.r1; ++r, ++k) {
        bars.wait_rowdone(k);
        const int o = r - 3;                                         // the output row this input row completed
        const bool okr = o >= pc.y0 && o < pc.y1;                    // (warp-uniform)
        float v[4];
        if (okr) {
          tc_fence_after();
          const uint32_t taddr = tmem_base + lane_addr + (uint32_t)((o & (SLOTS - 1)) * NCOL);
          tmem_ld4(taddr, v);
          tmem_ld_wait();
          tmem_zero<16>(taddr);                                      // (columns 3..15 only ever received zero weights)
          tmem_st_wait();
          tc_fence_before();
        }
        arrive_drained(bars, k, lane);
        if (okr && valid) {
          float* y = p.y + (size_t)pc.img * 3 * plane + (size_t)o * p.W + xcol;
          y[0] = tanhf(v[0] + b0);
          y[plane] = tanhf(v[1] + b1);
          y[2 * plane] = tanhf(v[2] + b2);
        }
      }
    }
  } else if (warp >= XF0) {
    // ===================================== transform: f slab -> a2 operand, in place =====================================
    const int xt = tid - 32 * XF0;                     // 0..127
    const int pchunk = xt & 7, rbase = xt >> 3;
    const int lchunk = pchunk ^ (rbase & 7);
    const double inv_hw = 1.0 / ((double)p.H * (double)p.W);
    float sc[8], sh[8];
    int cur_img = -1;
    SlabRing ring(bars.S);
    for (Walk pc = pieces; pc.next();) {
      if (pc.img != cur_img) {
        load_scale_shift(p.in_stats, p.in_gamma, p.in_beta, p.in_img_stride, pc.img, p.Cs_total, p.cs_off, lchunk, inv_hw, sc, sh);
        cur_img = pc.img;
      }
      const int r_lo = pc.r0 < 0 ? 0 : pc.r0, r_hi = pc.r1 > p.H ? p.H : pc.r1;
      const int x0 = pc.seg * BM - HALO;               // image column of slab pixel 0
      for (int r = r_lo; r < r_hi; ++r) {
        mbar_wait(bars.full(ring.s), ring.parity());
        uint8_t* fs = sm.stage_ptr(ring.s, SH.stage_bytes) + rbase * 128 + pchunk * 16;
        // (loads batched ahead of the arithmetic, no branches: rows 128..135 exist only for rbase < 8 -- those threads' ninth chunk --
        // and out-of-plane pixels are forced to 0 by a select: the conv's zero padding is a padding of a2)
        {
          uint4 raw[9], res[9];
#pragma unroll
          for (int i = 0; i < 9; ++i)
            if (i < 8 || rbase < 8) {
              raw[i] = *reinterpret_cast<const uint4*>(fs + i * (16 * 128));
              res[i] = *reinterpret_cast<const uint4*>(fs + SLAB_BYTES + i * (16 * 128));
            }
#pragma unroll
          for (int i = 0; i < 9; ++i) {
            const int x = x0 + rbase + 16 * i;
            const bool inside = x >= 0 && x < p.W;
            uint32_t w4[4] = {raw[i].x, raw[i].y, raw[i].z, raw[i].w};
            const uint32_t r4[4] = {res[i].x, res[i].y, res[i].z, res[i].w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              // packed f32x2 arithmetic with the apply kernel's roundings: fmaf, max 0, + residual, one bf16 RN pack
              const float2 x2 = make_float2(__uint_as_float(w4[j] << 16), __uint_as_float(w4[j] & 0xffff0000u));
              const float2 a2 = make_float2(__uint_as_float(r4[j] << 16), __uint_as_float(r4[j] & 0xffff0000u));
              float2 o2 = __ffma2_rn(x2, make_float2(sc[2 * j], sc[2 * j + 1]), make_float2(sh[2 * j], sh[2 * j + 1]));
              o2 = __fadd2_rn(make_float2(fmaxf(o2.x, 0.f), fmaxf(o2.y, 0.f)), a2);
              const __nv_bfloat162 pk = __floats2bfloat162_rn(o2.x, o2.y);
              w4[j] = inside ? *reinterpret_cast<const uint32_t*>(&pk) : 0u;
            }
            raw[i] = make_uint4(w4[0], w4[1], w4[2], w4[3]);
          }
#pragma unroll
          for (int i = 0; i < 9; ++i)
            if (i < 8 || rbase < 8) *reinterpret_cast<uint4*>(fs + i * (16 * 128)) = raw[i];
        }
        fence_proxy_async();                           // generic-proxy writes -> visible to the tensor core
        __syncwarp();
        if (lane == 0) mbar_arrive(bars.xf(ring.s));
        ring.advance();
      }
    }
  }
  teardown(warp, tmem_base);
}

}  // namespace
}  // namespace msg

using namespace msg;

extern "C" int msg_out7_ring_affine(const msg_out7_ring_desc* d, const void* f, const double* in_stats, const float* in_gamma,
                                    const float* in_beta, int in_img_stride, const void* residual, const void* w_stacks, const float* bias,
                                    float* y, void* stream) {
  cudaStream_t st = as_stream(stream);
  MSG_REQUIRE(d != nullptr && f && in_stats && residual && w_stacks && y, MSG_ERR_SHAPE, "out7_ring: null argument");
  MSG_REQUIRE(d->dtype == MSG_BF16, MSG_ERR_UNSUPPORTED, "out7_ring: bf16 only");
  MSG_REQUIRE(d->N > 0 && d->H > 0 && d->W > 0, MSG_ERR_SHAPE, "out7_ring: bad plane");
  MSG_REQUIRE((d->Cf_total & 7) == 0 && (d->cf_off & 7) == 0 && d->cf_off + 64 <= d->Cf_total, MSG_ERR_SHAPE, "out7_ring: f channel layout");
  MSG_REQUIRE((d->Cr_total & 7) == 0 && (d->cr_off & 7) == 0 && d->cr_off + 64 <= d->Cr_total, MSG_ERR_SHAPE, "out7_ring: residual channel layout");
  MSG_REQUIRE(d->cs_off >= 0 && d->cs_off + 64 <= d->Cs_total, MSG_ERR_SHAPE, "out7_ring: stats layout");
  MSG_REQUIRE((in_gamma == nullptr) == (in_beta == nullptr) && in_img_stride >= 0, MSG_ERR_SHAPE, "out7_ring: gamma and beta go together");
  MSG_REQUIRE((((uintptr_t)f | (uintptr_t)residual | (uintptr_t)w_stacks) & 15) == 0, MSG_ERR_ALIGN, "out7_ring: operands must be 16-byte aligned");
  MSG_REQUIRE(get_encode() != nullptr, MSG_ERR_CUDA, "out7_ring: cuTensorMapEncodeTiled unavailable");

  O7Params p;
  p.N = d->N; p.H = d->H; p.W = d->W;
  p.segs = (d->W + BM - 1) / BM;
  p.total_rows = (long long)d->N * p.segs * d->H;
  MSG_REQUIRE(p.total_rows < (1LL << 40), MSG_ERR_SHAPE, "out7_ring: too many rows");
  p.bias = bias; p.in_stats = in_stats; p.Cs_total = d->Cs_total; p.cs_off = d->cs_off; p.y = y;
  p.in_gamma = in_gamma; p.in_beta = in_beta; p.in_img_stride = in_img_stride;

  CUtensorMap mapF, mapR, mapB;
  CUresult r = encode_slab(&mapF, (const __nv_bfloat16*)f + d->cf_off, 64, d->Cf_total, d->W, d->H, d->N);
  MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "out7_ring: cuTensorMapEncodeTiled(f) failed with %d", (int)r);
  r = encode_slab(&mapR, (const __nv_bfloat16*)residual + d->cr_off, 64, d->Cr_total, d->W, d->H, d->N);
  MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "out7_ring: cuTensorMapEncodeTiled(residual) failed with %d", (int)r);
  r = encode_weights(&mapB, w_stacks, W_ROWS);
  MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "out7_ring: cuTensorMapEncodeTiled(w) failed with %d", (int)r);
  return launch<out7_ring_kernel>("out7_ring_kernel", o7_shape(), NTHREADS, p.total_rows, 8, p, mapF, mapR, mapB, st);
}

extern "C" int msg_out7_ring(const msg_out7_ring_desc* d, const void* f, const double* in_stats, const void* residual,
                             const void* w_stacks, const float* bias, float* y, void* stream) {
  return msg_out7_ring_affine(d, f, in_stats, nullptr, nullptr, 0, residual, w_stacks, bias, y, stream);
}
