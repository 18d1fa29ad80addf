// The first down-sampling conv of the encoder (enhanced_generator.py:99-104: Conv2d(c, 2c, 4, stride 2, padding 1), c = 64) fused with
// the InstanceNorm + ReLU of the 7x7 input layer in front of it (enhanced_generator.py:93-97), as a ROW RING of tensor-memory
// accumulators (sm_100a, bf16 operands, fp32 accumulate) -- the stride-2 member of the msb_ring.cu / convt_ring.cu / out7_ring.cu family
// (shared mechanics in ring.cuh).
//
//   a = ReLU(IN(x))              x: raw output of the 7x7 input conv with its plane statistics
//   y[o, u] = sum a[2o - 1 + ky, 2u - 1 + kx] w[ky, kx] + b      (+ IN statistics of y)
//
// Until now: an HBM-bound apply kernel (read x, write a: 1.07 GB per 16 images at 512^2) and the per-tap implicit GEMM of conv_tma.cu
// (16 taps, each an M = 128 x N = 128 MMA per K step, every input pixel fetched four times from L2).  Here a CTA walks DOWN a column
// strip of 128 output pixels = 256 input pixels, one launch per 64 output channels (the launch's 16 taps x 64 x 64 weights = 128 KB
// stay resident in shared memory):
//   * every input row is loaded ONCE per launch as two slabs, its even and its odd pixels (one TMA each through a tensor map that
//     views the row as [W/2][2] pixels), so that the stride-2 taps become SHIFTED VIEWS: kx = 0, 2 read the odd slab at pixel u - 1, u
//     and kx = 1, 3 the even slab at u, u + 1; four transform warps normalise the landed slabs in place with the apply kernel's
//     arithmetic (pixels outside the plane forced to 0: the conv pads a, not x), so a never exists in HBM;
//   * input row r feeds two output rows -- (r-1)/2 rounded down and the next one -- whose accumulators are adjacent 64-column slots of
//     an eight-slot ring: per horizontal tap the two vertical taps are ONE MMA of N = 128 (full rate on the tensor pipe), 16 MMAs per
//     input row at c = 64;
//   * every second input row completes an output row: eight epilogue warps (lane quarter x channel half) drain it and hand
//     [32 px x 32 ch] pieces to the TMA store.
// A piece [y0, y1) of OUTPUT rows reads the input rows 2 y0 - 1 .. 2 y1, one step each.
// Schedule stated and run on tensors in slab.py (down_ring_row_mmas) / tests/test_down_ring_cpu.py.
//
//   warp 0       TMA producer: the launch's weight stacks once, then the even / odd slabs of one input row per stage
//   warp 1       MMA issuer (also allocates TMEM)
//   warps 4-11   epilogue
//   warps 12-15  transform
#include "ring.cuh"

namespace msg {
namespace {
using namespace ring;

constexpr int NC = 64;                  // output channels per launch = columns per row accumulator
constexpr int NEW = 8, XF0 = 12;
constexpr uint32_t LEAD = 8;            // a slot is touched again 13 steps after its row completed
constexpr int W_ROWS = 4 * 2 * 2 * NC;  // [kx][input-row parity][entry][64 co] rows of 64 input channels
constexpr int NTHREADS = 32 * 16;
constexpr int OUT_B = 2048;             // per-warp scratch: [16 ch][32 px] fp32 for the statistics, then the [32 px][32 ch] bf16 piece
// weights | stages of the even | odd pixels of one input row, 64 channels | bias | scratch; full / empty / transformed per stage
__host__ __device__ constexpr Shape dn_shape() { return Shape{W_ROWS * 128, 2 * SLAB_BYTES, NC, NEW * OUT_B, 3}; }

struct DnParams {
  int N, H, W;                          // input plane (H, W even); output H/2 x W/2
  int Co_total, co_off;
  int segs;
  long long total_rows;                 // N * segs * (H/2) output rows
  int stages;
  int w_row0;
  const float* bias;                    // [64] of this launch's channels, or null
  double* stats;
  const double* in_stats;               // [N][Cs_total][2] raw plane sums of x, or null (x is used as it is)
  int Cs_total, cs_off;
};

__global__ void __launch_bounds__(NTHREADS, 1)
down_ring_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                 const __grid_constant__ CUtensorMap mapY, const DnParams p) {
  constexpr Shape SH = dn_shape();
  using Walk = Pieces<2, 1>;
  extern __shared__ uint8_t smem_raw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int Ho = p.H >> 1, Wo = p.W >> 1;
  const Smem sm(smem_raw, SH, p.stages);
  const Bars& bars = sm.b;
  float* sbias = sm.bias();

  if (tid < NC) sbias[tid] = p.bias ? p.bias[tid] : 0.f;
  const uint32_t tmem_base = prologue(sm, warp, lane, 1, NEW, 4, &mapA, &mapB, &mapY);
  const Walk pieces(p.total_rows, Ho, p.segs);

  if (warp == 0) {
    if (lane == 0)
      producer(sm, pieces, p.H, &mapB, SH.w_bytes, p.w_row0, SH.stage_bytes, [&](const Walk& pc, int r, uint32_t dst, uint32_t bar) {
        tma_load_5d(dst, &mapA, bar, 0, 0, pc.seg * BM - HALO, r, pc.img);                  // even pixels
        tma_load_5d(dst + SLAB_BYTES, &mapA, bar, 0, 1, pc.seg * BM - HALO, r, pc.img);     // odd pixels
      });
  } else if (warp == 1) {
    const bool leader = elect_one();
    const uint32_t hi = (uint32_t)(make_sw128_desc(0) >> 32);
    const uint32_t b_base = sm.sB() >> 4;
    issuer<LEAD, true>(bars, pieces, p.H, leader, [&](const Walk& pc, int r, int s) {
      const uint32_t a0 = sm.sA(s, SH.stage_bytes) >> 4;
      const int par = r & 1;
      // entries e = 0, 1 = output rows of = (r - 1) >> 1 and of + 1 (vertical taps ky = 3 - par, 1 - par)
      const int of = (r - 1) >> 1;                             // (arithmetic shift: r = 0 -> -1)
      const int o_lo = of > pc.y0 ? of : pc.y0, o_hi = of + 1 < pc.y1 - 1 ? of + 1 : pc.y1 - 1;      // inclusive
      if (o_lo <= o_hi)
        runs(o_hi - o_lo + 1, o_lo & 7, 8, [&](int e, int nrun, int slot) {
          const uint32_t idesc = idesc_bf16(NC * nrun);
          const uint32_t dcol = tmem_base + (uint32_t)(slot * NC);
#pragma unroll
          for (int kx = 0; kx < 4; ++kx) {
            // kx = 0: odd pixels at u - 1; 1: even at u; 2: odd at u; 3: even at u + 1
            const uint32_t av = a0 + (uint32_t)(((kx & 1) ? 0 : (SLAB_BYTES >> 4)) + (HALO + (kx == 0 ? -1 : (kx == 3 ? 1 : 0))) * 8);
            const uint32_t bv = b_base + (uint32_t)((((kx * 2 + par) * 2 + (o_lo - of + e)) * NC) * 8);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) umma_bf16_lo(dcol, av + (uint32_t)(2 * ks), bv + (uint32_t)(2 * ks), hi, idesc, true);
          }
        });
    });
  } else if (warp >= EPI0 && warp < XF0) {
    // ===================================== epilogue: warp = (lane quarter q, channel half h) =====================================
    const int q = warp & 3;
    const int ew = warp - EPI0;
    const int h = ew >> 2;
    const int row = q * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    uint8_t* buf = sm.scratch(ew, OUT_B);
    Stats stats;
    const bool do_stats = p.stats != nullptr;
    uint32_t k = 0;
    bool stored = false;
    for (Walk pc = pieces; pc.next();) {
      const bool valid = pc.seg * BM + row < Wo;
      if (do_stats && pc.img != stats.img) { stats.flush<32>(p.stats, p.Co_total, p.co_off + 32 * h, lane); stats.img = pc.img; }
      for (int r = pc.r0; r < pc.r1; ++r, ++k) {
        bars.wait_rowdone(k);
        // an even input row r completes the output row r / 2 - 1 (its last tap is ky = 3)
        const int o = (r >> 1) - 1;
        const bool okr = !(r & 1) && o >= pc.y0 && o < pc.y1;        // (warp-uniform)
        float v[32];
        if (okr) {
          tc_fence_after();
          const uint32_t ta = tmem_base + lane_addr + (uint32_t)((o & 7) * NC + 32 * h);
          tmem_ld32(ta, v);
          tmem_ld_wait();
          tmem_zero<32>(ta);
          tmem_st_wait();
          tc_fence_before();
        }
        arrive_drained(bars, k, lane);
        if (!okr) continue;
#pragma unroll
        for (int c = 0; c < 32; ++c) v[c] += sbias[32 * h + c];
        if (stored) wait_store_read<0>(lane);
        if (do_stats) piece_stats<32>(reinterpret_cast<float*>(buf), v, valid, lane, stats);
        store_piece_bf16<32>(buf, v, lane, &mapY, p.co_off + 32 * h, pc.seg * BM + q * 32, o, pc.img);
        stored = true;
      }
    }
    if (do_stats) stats.flush<32>(p.stats, p.Co_total, p.co_off + 32 * h, lane);
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  } else if (warp >= XF0) {
    // ===================================== transform: x slabs -> ReLU(IN(x)), in place =====================================
    const int xt = tid - 32 * XF0;                     // 0..127
    const int pchunk = xt & 7, rbase = xt >> 3;
    const int lchunk = pchunk ^ (rbase & 7);
    const double inv_hw = 1.0 / ((double)p.H * (double)p.W);
    const bool xform = p.in_stats != nullptr;
    float sc[8], sh[8];
    int cur_img = -1;
    SlabRing ring(bars.S);
    for (Walk pc = pieces; pc.next();) {
      if (xform && pc.img != cur_img) {
        load_scale_shift(p.in_stats, pc.img, p.Cs_total, p.cs_off, lchunk, inv_hw, sc, sh);
        cur_img = pc.img;
      }
      const int r_lo = pc.r0 < 0 ? 0 : pc.r0, r_hi = pc.r1 > p.H ? p.H : pc.r1;
      const int j0 = pc.seg * BM - HALO;               // pixel-pair index of slab pixel 0
      for (int r = r_lo; r < r_hi; ++r) {
        mbar_wait(bars.full(ring.s), ring.parity());
        if (xform) {
          uint8_t* fs = sm.stage_ptr(ring.s, SH.stage_bytes) + rbase * 128 + pchunk * 16;
          // (loads of a slab batched ahead of the arithmetic, no branches: rows 128..135 exist only for rbase < 8 -- those threads'
          // ninth chunk -- and out-of-plane pixels are forced to 0 by a select)
          const __nv_bfloat162 zero2 = __floats2bfloat162_rn(0.f, 0.f);
#pragma unroll
          for (int par = 0; par < 2; ++par) {
            uint4 raw[9];
#pragma unroll
            for (int i = 0; i < 9; ++i)
              if (i < 8 || rbase < 8) raw[i] = *reinterpret_cast<const uint4*>(fs + par * SLAB_BYTES + i * (16 * 128));
#pragma unroll
            for (int i = 0; i < 9; ++i) {
              const int x = 2 * (j0 + rbase + 16 * i) + par;
              const bool inside = x >= 0 && x < p.W;
              uint32_t w4[4] = {raw[i].x, raw[i].y, raw[i].z, raw[i].w};
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                // packed path of conv_tma.cu's fused input norm: two fmaf per FFMA2 (the apply kernel's roundings), bf16 RN pack,
                // ReLU as a packed bf16 max AFTER rounding (rounding is monotone and keeps 0)
                const float2 x2 = make_float2(__uint_as_float(w4[j] << 16), __uint_as_float(w4[j] & 0xffff0000u));
                const float2 o2 = __ffma2_rn(x2, make_float2(sc[2 * j], sc[2 * j + 1]), make_float2(sh[2 * j], sh[2 * j + 1]));
                __nv_bfloat162 pk = __hmax2(__floats2bfloat162_rn(o2.x, o2.y), zero2);
                w4[j] = inside ? *reinterpret_cast<uint32_t*>(&pk) : 0u;     // the conv's zero padding is a padding of a
              }
              raw[i] = make_uint4(w4[0], w4[1], w4[2], w4[3]);
            }
#pragma unroll
            for (int i = 0; i < 9; ++i)
              if (i < 8 || rbase < 8) *reinterpret_cast<uint4*>(fs + par * SLAB_BYTES + i * (16 * 128)) = raw[i];
          }
          fence_proxy_async();
        }
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

extern "C" int msg_down_ring(const msg_down_ring_desc* d, const void* x, const double* in_stats, const void* w_stacks, const float* bias,
                             void* y, double* stats, void* stream) {
  cudaStream_t st = as_stream(stream);
  MSG_REQUIRE(d != nullptr && x && w_stacks && y, MSG_ERR_SHAPE, "down_ring: null argument");
  MSG_REQUIRE(d->dtype == MSG_BF16, MSG_ERR_UNSUPPORTED, "down_ring: bf16 only");
  MSG_REQUIRE(d->Cout > 0 && d->Cout % 64 == 0, MSG_ERR_UNSUPPORTED, "down_ring: Cout must be a multiple of 64 (got %d)", d->Cout);
  MSG_REQUIRE(d->N > 0 && d->H > 0 && d->W > 0 && (d->H & 1) == 0 && (d->W & 1) == 0, MSG_ERR_SHAPE, "down_ring: the plane must have even sides");
  MSG_REQUIRE((d->Ci_total & 7) == 0 && (d->ci_off & 7) == 0 && d->ci_off + 64 <= d->Ci_total, MSG_ERR_SHAPE, "down_ring: input channel layout (Cin = 64)");
  MSG_REQUIRE((d->Co_total & 7) == 0 && (d->co_off & 7) == 0 && d->co_off + d->Cout <= d->Co_total, MSG_ERR_SHAPE, "down_ring: output channel layout");
  MSG_REQUIRE(in_stats == nullptr || (d->cs_off >= 0 && d->cs_off + 64 <= d->Cs_total), MSG_ERR_SHAPE, "down_ring: stats layout");
  MSG_REQUIRE((((uintptr_t)x | (uintptr_t)w_stacks | (uintptr_t)y) & 15) == 0, MSG_ERR_ALIGN, "down_ring: operands must be 16-byte aligned");
  MSG_REQUIRE(!(d->flags & MSG_CONV_STATS) || stats != nullptr, MSG_ERR_SHAPE, "down_ring: stats buffer missing");
  MSG_REQUIRE(get_encode() != nullptr, MSG_ERR_CUDA, "down_ring: cuTensorMapEncodeTiled unavailable");
  const int G = d->Cout / 64, Ho = d->H / 2, Wo = d->W / 2;

  DnParams p;
  p.N = d->N; p.H = d->H; p.W = d->W; p.Co_total = d->Co_total;
  p.stats = (d->flags & MSG_CONV_STATS) ? stats : nullptr;
  p.in_stats = in_stats; p.Cs_total = d->Cs_total; p.cs_off = d->cs_off;
  p.segs = (Wo + BM - 1) / BM;
  p.total_rows = (long long)d->N * p.segs * Ho;
  MSG_REQUIRE(p.total_rows < (1LL << 40), MSG_ERR_SHAPE, "down_ring: too many rows");

  CUtensorMap mapA, mapB, mapY;
  {
    // the input row as [W/2][2] pixels: coordinate 1 selects the even or the odd pixels, coordinate 2 the pixel pair
    const cuuint64_t dims[5] = {64, 2, (cuuint64_t)Wo, (cuuint64_t)d->H, (cuuint64_t)d->N};
    const cuuint64_t strides[4] = {(cuuint64_t)d->Ci_total * 2, (cuuint64_t)2 * d->Ci_total * 2, (cuuint64_t)d->W * d->Ci_total * 2,
                                   (cuuint64_t)d->H * d->W * d->Ci_total * 2};
    const cuuint32_t box[5] = {64, 1, (cuuint32_t)SLAB_PX, 1, 1};
    const CUresult r = encode(&mapA, 5, (const __nv_bfloat16*)x + d->ci_off, dims, strides, box, true);
    MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "down_ring: cuTensorMapEncodeTiled(x) failed with %d", (int)r);
  }
  CUresult r = encode_weights(&mapB, w_stacks, (long long)G * W_ROWS);
  MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "down_ring: cuTensorMapEncodeTiled(w) failed with %d", (int)r);
  r = encode_store(&mapY, y, d->Co_total, Wo, Ho, d->N, 32, 1);
  MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "down_ring: cuTensorMapEncodeTiled(y) failed with %d", (int)r);
  for (int g = 0; g < G; ++g) {
    p.co_off = d->co_off + 64 * g;
    p.bias = bias ? bias + 64 * g : nullptr;
    p.w_row0 = g * W_ROWS;
    const int rc = launch<down_ring_kernel>("down_ring_kernel", dn_shape(), NTHREADS, p.total_rows, 4, p, mapA, mapB, mapY, st);
    if (rc) return rc;
  }
  return MSG_OK;
}
