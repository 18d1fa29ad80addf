// Persistent, warp-specialised tcgen05 implicit-GEMM convolution fed by TMA (sm_100a, bf16).
//
// The A operand of an implicit-GEMM conv on NHWC data needs no im2col buffer and no per-thread
// address math when the output plane width is a power of two: a 128-pixel M tile is R = 128/Wt full
// (or partial, Wt = 128) output rows of Wt pixels, and for one filter tap its input pixels form a
// regular 4-D box [64 channels x Wt pixels (step = conv stride) x R rows (step = stride) x 1 image]
// of the activation tensor.  ONE cp.async.bulk.tensor.4d (tile mode, 128B swizzle, hardware
// zero-fill outside the image = the conv's zero padding, negative start coordinates allowed) lands it
// in shared memory in exactly the K-major SWIZZLE_128B layout tcgen05.mma reads.  The weight slab of
// the same K block is one 2-D TMA box.  So the producer is a single thread issuing two TMA
// instructions per K block; the SM's issue slots are free for the epilogue.
//
//   warp 0 : TMA producer (one elected lane), ring of kStages smem stages, full/empty mbarriers
//   warp 1 : TMEM allocator + MMA issuer (one lane): tcgen05.mma.cta_group::1.kind::f16, M=128,
//            N=BN<=256, K=16, accumulators DOUBLE-BUFFERED in TMEM (2 x BN columns)
//   warps 2-5 : epilogue.  tcgen05.ld -> +bias -> (IN statistics) -> activation -> bf16 -> smem
//            staging -> coalesced 128-byte row stores; releases the accumulator buffer as soon as it
//            has been read, so the next tile's MMAs overlap this tile's stores.
// One CTA per SM, looping over (m tile, n tile) work items.
//
// Geometry requirement (checked by conv2d_tma_supported): Cin % 64 == 0, and either Wg % 128 == 0 or
// (128 % Wg == 0 and Hg % (128/Wg) == 0).  Everything else takes the gather kernel (conv_tc.cu) or
// the SIMT engine.  Same descriptor semantics as include/msg_b200.h.
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdlib.h>

#include "common.cuh"
#include "tcgen05.cuh"

namespace msg {
namespace {
using namespace tc;

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int A_BYTES = BM * BK * 2;
constexpr int NTHREADS = 320;          // producer + MMA warp + up to two epilogue groups of four warps
constexpr int NTHREADS_XF = 448;       // ... + four transform warps (fused input InstanceNorm)
constexpr int EPI_FIXED = 16384 + 4 * 1088 * 4;  // per epilogue group: fp64 column sums [4][2][256] + transpose scratch [4][32][34]
constexpr int STAGE_PITCH = 128 + 16;   // manual flush: 64 bf16 columns per row + 16 B skew
constexpr int STAGE_BYTES = 2 * BM * 128;   // two [128 rows x 64 cols] bf16 TMA-store buffers (SW128)


struct TmaParams {
  msg_conv_desc d;
  const float* bias;
  void* y;
  double* stats;
  int BN, n_tiles, m_tiles, stages, tmem_cols;
  const double* in_stats;   // MSG_CONV_IN_NORM: raw plane sums [N][Ci_total][2] of the INPUT tensor
  const float* in_gamma;    // MSG_CONV_IN_NORM: optional affine of the input norm (common.cuh: in_affine), or null
  const float* in_beta;
  int in_img_stride;
  int xform;          // 1: four transform warps apply InstanceNorm + activation to every A tile in smem (1x1 convs)
  int b_resident;     // 1: all nkb weight tiles of the (single) N tile stay in smem for the whole kernel
  int epi_groups;     // 1: warps 2-5 drain both accumulator buffers; 2: warps 2-5 own buffer 0, warps 6-9 buffer 1
  int Wt, R;            // M tile = R rows x Wt pixels
  int cblocks;          // Cin / 64
  int nkb;              // KH*KW*cblocks
  int tstore;           // output rows of a tile are 128 consecutive pixels: full 64-column groups go out by TMA
};

template <bool XFORM>
__global__ void __launch_bounds__(XFORM ? NTHREADS_XF : NTHREADS, 1)
conv_tma_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                const __grid_constant__ CUtensorMap mapC, const TmaParams p) {
  extern __shared__ uint8_t smem_raw[];
  const msg_conv_desc& d = p.d;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int BN = p.BN, S = p.stages;
  const int b_bytes = BN * BK * 2;
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sA = base;
  const uint32_t sB = sA + S * A_BYTES;
  const uint32_t sStage = sB + (p.b_resident ? p.nkb : S) * b_bytes;   // epilogue staging, 1024-byte aligned
  const uint32_t sRed = sStage + p.epi_groups * STAGE_BYTES;              // per-warp column sums / transpose scratch
  const uint32_t sBias = sRed + p.epi_groups * EPI_FIXED;                 // bias staged once per CTA (<= 1024 floats)
  const uint32_t sXfTab = sBias + 4096;                     // fused input norm: scale[512], shift[512] of the current image
  const uint32_t sBar = sXfTab + 4096;                      // full[S], empty[S], xf[S], tfull[2], tempty[2], wres, tmem slot
  uint8_t* stage_gen = gen + (sStage - base);
  float* red = reinterpret_cast<float*>(gen + (sRed - base));
  float* sbias = reinterpret_cast<float*>(gen + (sBias - base));
  float* xf_tab = reinterpret_cast<float*>(gen + (sXfTab - base));
  const bool bias_in_smem = p.bias != nullptr && d.Cout <= 1024;
  if (bias_in_smem)
    for (int i = tid; i < d.Cout; i += (int)blockDim.x) sbias[i] = p.bias[i];
  const uint32_t wres_bar = sBar + 8u * (3 * S + 4);        // "resident weights have landed"
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gen + (sBar - base) + 8 * (3 * S + 5));
  auto full_bar = [&](int s) { return sBar + 8u * s; };
  auto empty_bar = [&](int s) { return sBar + 8u * (S + s); };
  auto xf_bar = [&](int s) { return sBar + 8u * (2 * S + s); };          // "A tile of stage s has been normalised"
  auto tfull_bar = [&](int b) { return sBar + 8u * (3 * S + b); };
  auto tempty_bar = [&](int b) { return sBar + 8u * (3 * S + 2 + b); };

  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < S; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); mbar_init(xf_bar(s), 4); }
      for (int b = 0; b < 2; ++b) { mbar_init(tfull_bar(b), 1); mbar_init(tempty_bar(b), 4); }
      mbar_init(wres_bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  } else if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapA)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapB)) : "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int total_tiles = p.m_tiles * p.n_tiles;
  // each CTA owns a CONTIGUOUS range of tiles (same image, neighbouring rows: L2 locality, and the
  // epilogue can keep per-channel statistics on chip across its tiles)
  const int t_begin = (int)((long long)blockIdx.x * total_tiles / gridDim.x);
  const int t_end = (int)((long long)(blockIdx.x + 1) * total_tiles / gridDim.x);
  const int tiles_per_row = d.Wg / p.Wt;        // >= 1
  const int tile_rows = d.Hg / p.R;             // row groups per image

  if (warp == 0) {
    // ===================================== TMA producer =====================================
    if (lane == 0) {
      if (p.b_resident) {      // one N tile and few K blocks: the weights are loaded once and never re-streamed
        mbar_expect_tx(wres_bar, (uint32_t)(p.nkb * b_bytes));
        for (int kb = 0; kb < p.nkb; ++kb) tma_load_2d(sB + kb * b_bytes, &mapB, wres_bar, kb * BK, 0);
      }
      int s = 0;
      uint32_t ph = 0;
      bool wrapped = false;
      for (int t = t_begin; t < t_end; ++t) {
        const int nt = t % p.n_tiles, mt = t / p.n_tiles;
        const int img = mt / (tile_rows * tiles_per_row);
        const int rem = mt - img * (tile_rows * tiles_per_row);
        const int rg = rem / tiles_per_row, cg = rem - rg * tiles_per_row;
        const int i0 = rg * p.R, j0 = cg * p.Wt;
        const int w_base = j0 * d.in_stride - d.pad_w, h_base = i0 * d.in_stride - d.pad_h;
        const int w_row0 = (d.flags & MSG_CONV_PER_IMAGE_W) ? img * d.Cout : 0;   // per-image weights: row block of this image
        int kb = 0;
        for (int th = 0; th < d.KH; ++th)
          for (int tw = 0; tw < d.KW; ++tw)
            for (int cb = 0; cb < p.cblocks; ++cb, ++kb) {
              if (wrapped) mbar_wait(empty_bar(s), ph ^ 1u);
              mbar_expect_tx(full_bar(s), A_BYTES + (p.b_resident ? 0 : b_bytes));
              tma_load_4d(sA + s * A_BYTES, &mapA, full_bar(s), cb * BK, w_base + tw * d.dil, h_base + th * d.dil, img);
              if (!p.b_resident) tma_load_2d(sB + s * b_bytes, &mapB, full_bar(s), kb * BK, nt * BN + w_row0);
              if (++s == S) { s = 0; ph ^= 1u; wrapped = true; }   // no per-K-block div/mod by the runtime stage count
            }
      }
    }
  } else if (warp == 1) {
    // ===================================== MMA issuer =====================================
    // The issue loop is a single warp's serial instruction stream (~6 cycles per dependent instruction), and a K
    // block of four N<=128 MMAs is only 128-256 tensor cycles: every instruction here is on the critical path.
    // So: the whole warp runs the loop (warp-uniform values stay in uniform registers), stage / phase are counted
    // incrementally (no div/mod by the runtime stage count), descriptors are one multiply-add from the stage
    // index, and one elected lane issues the four MMAs and the commit of a K block.
    {
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      const uint32_t hi = (uint32_t)(make_sw128_desc(0) >> 32);     // constant high descriptor word (SBO, version, swizzle)
      const uint32_t a_base = sA >> 4, b_base = sB >> 4;
      const uint32_t a_step = A_BYTES >> 4, b_step = (uint32_t)b_bytes >> 4;
      const bool leader = elect_one();        // one election for the whole kernel: no ELECT / reconvergence per K block
      const bool bres = p.b_resident != 0;
      int s = 0;
      uint32_t ph = 0, lt = 0;
      if (bres) mbar_wait(wres_bar, 0);
      for (int t = t_begin; t < t_end; ++t, ++lt) {
        const int buf = lt & 1;
        if (lt >= 2) mbar_wait(tempty_bar(buf), ((lt >> 1) - 1) & 1);
        tc_fence_after();
        const uint32_t tacc = tmem_base + (uint32_t)(buf * BN);
        for (int kb = 0; kb < p.nkb; ++kb) {
          mbar_wait(XFORM ? xf_bar(s) : full_bar(s), ph);
          tc_fence_after();
          // descriptors as {32-bit start-address word, constant high word}: the K-step advance is a 32-bit add
          const uint32_t a_lo = a_base + (uint32_t)s * a_step;
          const uint32_t b_lo = b_base + (uint32_t)(bres ? kb : s) * b_step;
          if (leader) {
            umma_bf16_lo(tacc, a_lo, b_lo, hi, idesc, kb != 0);
            umma_bf16_lo(tacc, a_lo + 2, b_lo + 2, hi, idesc, true);
            umma_bf16_lo(tacc, a_lo + 4, b_lo + 4, hi, idesc, true);
            umma_bf16_lo(tacc, a_lo + 6, b_lo + 6, hi, idesc, true);
            umma_commit(empty_bar(s));
          }
          __syncwarp();
          if (++s == S) { s = 0; ph ^= 1u; }
        }
        if (leader) umma_commit(tfull_bar(buf));
        __syncwarp();
      }
    }
  } else if (XFORM && warp >= 2 + 4 * p.epi_groups) {
    // ===================================== fused input InstanceNorm (four transform warps) ==========
    // 1x1 convs only: the A tile is 128 consecutive pixels of ONE image x 64 channels, 128B-swizzled by TMA.
    // Each landed stage is rewritten in place as act((x - mean) * rstd) with the apply kernel's exact arithmetic
    // (fmaf(x, scale, shift), bf16 round-to-nearest), so the fused conv is bit-identical to IN-apply + conv while
    // the normalised tensor never exists in HBM.  Thread t owns physical 16-byte chunk (t & 7) of rows (t >> 3) + 16 i:
    // a warp touches 512 contiguous bytes per access (conflict-free) and, because the swizzle only uses row & 7, the
    // LOGICAL channel chunk of a thread is the same for all its rows -- its 8 scales / shifts live in registers.
    const int xt = tid - 32 * (2 + 4 * p.epi_groups);           // 0..127
    const int pchunk = xt & 7, rbase = xt >> 3;
    const int lchunk = pchunk ^ (rbase & 7);
    const int hw = d.Hg * d.Wg;
    const double inv_hw = 1.0 / (double)hw;
    int cur_img = -1, cur_cb = -1;
    float sc[8], sh[8];
    int s = 0;
    uint32_t ph = 0;
    for (int t = t_begin; t < t_end; ++t) {
      const int mt = t / p.n_tiles;
      const int img = (int)(((long long)mt * BM) / hw);
      if (img != cur_img) {                                      // new image: rebuild the per-channel table
        asm volatile("bar.sync 2, 128;" ::: "memory");           // everyone is done reading the old table
        for (int ci = xt; ci < d.Cin; ci += 128) {
          const int c = d.ci_off + ci;
          float g, b, mean, rstd;
          in_affine(p.in_gamma, p.in_beta, (size_t)img * p.in_img_stride + c, g, b);
          in_scale_shift(p.in_stats + ((size_t)img * d.Ci_total + c) * 2, inv_hw, g, b, mean, rstd, xf_tab[ci], xf_tab[512 + ci]);
        }
        asm volatile("bar.sync 2, 128;" ::: "memory");
        cur_img = img; cur_cb = -1;
      }
      for (int kb = 0; kb < p.nkb; ++kb) {                       // 1x1 conv: K block kb = channel block kb
        if (kb != cur_cb) {
#pragma unroll
          for (int e = 0; e < 8; ++e) { sc[e] = xf_tab[kb * 64 + lchunk * 8 + e]; sh[e] = xf_tab[512 + kb * 64 + lchunk * 8 + e]; }
          cur_cb = kb;
        }
        mbar_wait(full_bar(s), ph);
        uint8_t* tile = gen + (sA - base) + s * A_BYTES + rbase * 128 + pchunk * 16;
        if (d.in_act == MSG_ACT_RELU || d.in_act == MSG_ACT_NONE) {
          // packed path: two fmaf per FFMA2 (same roundings as the apply kernel's fmaf), bf16 RN pack, ReLU as a packed bf16
          // max AFTER rounding (rounding is monotone and keeps 0, so max(rn(o), 0) == rn(max(o, 0)) up to the sign of zero)
          const bool relu = d.in_act == MSG_ACT_RELU;
          const __nv_bfloat162 zero2 = __floats2bfloat162_rn(0.f, 0.f);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            uint4* ptr = reinterpret_cast<uint4*>(tile + i * (16 * 128));
            uint4 raw = *ptr;
            uint32_t w4[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float2 x2 = make_float2(__uint_as_float(w4[j] << 16), __uint_as_float(w4[j] & 0xffff0000u));
              const float2 o2 = __ffma2_rn(x2, make_float2(sc[2 * j], sc[2 * j + 1]), make_float2(sh[2 * j], sh[2 * j + 1]));
              __nv_bfloat162 pk = __floats2bfloat162_rn(o2.x, o2.y);
              if (relu) pk = __hmax2(pk, zero2);
              w4[j] = *reinterpret_cast<uint32_t*>(&pk);
            }
            *ptr = make_uint4(w4[0], w4[1], w4[2], w4[3]);
          }
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            uint4* ptr = reinterpret_cast<uint4*>(tile + i * (16 * 128));
            float v[8];
            unpack8(*ptr, v);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              float o = fmaf(v[e], sc[e], sh[e]);
              o = o > 0.f ? o : 0.2f * o;
              v[e] = o;
            }
            *ptr = pack8(v);
          }
        }
        fence_proxy_async();                                     // generic-proxy writes -> visible to the tensor core
        __syncwarp();
        if (lane == 0) mbar_arrive(xf_bar(s));
        if (++s == S) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp >= 2 && ((warp - 2) >> 2) < p.epi_groups) {
    // ===================================== epilogue (warps 2-5, and 6-9 with two groups) ===========
    // The epilogue of a 128 x BN tile is a single warp's instruction stream per 32 rows (~550 instructions per 64
    // columns with bias + statistics): with one warp per scheduler it is latency-bound and, for the 1x1 convs
    // (one K block per tile), the whole kernel's bottleneck.  With two groups, group g drains accumulator buffer g,
    // i.e. every other tile, so two epilogues are in flight per scheduler.
    const int q = warp & 3;                       // TMEM lane quarter this warp may access
    const int grp = (warp - 2) >> 2;              // epilogue group
    const int G = p.epi_groups;
    const int row = q * 32 + lane;                // row of the M tile
    const bool do_stats = d.flags & MSG_CONV_STATS;
    const bool nchw = d.flags & MSG_CONV_OUT_NCHW_F32;
    const bool accum = d.flags & MSG_CONV_ACCUM;
    const int hw = d.Hg * d.Wg;
    // this warp's staging slice: 8 KB = two [32 rows x 128 B] TMA-store buffers (1024-byte aligned), also
    // used as the skewed [32 x 144 B] tile of the manual flush
    uint8_t* stage_w = stage_gen + (grp * 4 + q) * 8192;
    const uint32_t stage_w_s = sStage + (grp * 4 + q) * 8192;
    // running column sums of this warp, [2][256], in fp64: the 32-row partial sums are formed in fp32 in a fixed
    // order, everything above that is fp64, so an image's statistics do not depend on how tiles were grouped per CTA
    // (batch size, epilogue groups) beyond fp64 rounding
    float2* wsum = reinterpret_cast<float2*>(red + grp * (EPI_FIXED / 4)) + q * 512;
    float* tr = red + grp * (EPI_FIXED / 4) + 4096 + q * 1088;            // [32][34] transpose scratch of this warp
    for (int i = lane; i < 512; i += 32) wsum[i] = make_float2(0.f, 0.f);
    __syncwarp();
    int stat_img = -1, stat_nt = -1, stat_cmax = 0;
    auto flush_stats = [&]() {
      if (stat_img >= 0) {
        for (int c = lane; c < stat_cmax; c += 32) {
          double* st = p.stats + ((size_t)stat_img * d.Co_total + d.co_off + stat_nt * BN + c) * 2;
          atomicAdd(st, f2sum_value(wsum[c]));
          atomicAdd(st + 1, f2sum_value(wsum[256 + c]));
          wsum[c] = make_float2(0.f, 0.f); wsum[256 + c] = make_float2(0.f, 0.f);
        }
      }
      __syncwarp();
    };
    uint32_t lt = 0, sgrp = 0;                    // tiles done, TMA-store groups issued by this warp
    bool tma_pending = false;                     // (lane 0) bulk groups possibly still reading smem
    for (int t = t_begin + (G == 2 ? grp : 0); t < t_end; t += G, ++lt) {
      const int nt = t % p.n_tiles, mt = t / p.n_tiles;
      const int buf = G == 2 ? grp : (int)(lt & 1);                      // accumulator buffer of this tile
      const uint32_t tf_parity = G == 2 ? (lt & 1) : ((lt >> 1) & 1);    // its (lt or lt/2)-th use
      const long long m0 = (long long)mt * BM;
      const int co0 = nt * BN;
      const int cmax = (d.Cout - co0) < BN ? (d.Cout - co0) : BN;
      const bool vec = !nchw && ((d.Co_total | d.co_off | cmax) & 7) == 0;
      int opix;
      {
        const long long m = m0 + row;
        const int n = (int)(m / hw);
        const int rem = (int)(m - (long long)n * hw);
        const int gi = rem / d.Wg, gj = rem - gi * d.Wg;
        opix = (n * d.Ho + gi * d.out_stride + d.out_off_h) * d.Wo + gj * d.out_stride + d.out_off_w;
      }
      const int opix_w = __shfl_sync(0xffffffffu, opix, 0);   // tstore: this warp's 32 rows are consecutive pixels
      const int n_img = (int)(m0 / hw);
      if (do_stats && (n_img != stat_img || nt != stat_nt)) {
        flush_stats();
        stat_img = n_img; stat_nt = nt; stat_cmax = cmax;
      }
      mbar_wait(tfull_bar(buf), tf_parity);
      tc_fence_after();
      const uint32_t tacc = tmem_base + (uint32_t)(buf * BN) + ((uint32_t)(q * 32) << 16);
      for (int cg = 0; cg < cmax; cg += 64) {
        const int ncol = (cmax - cg) < 64 ? (cmax - cg) : 64;
        __syncwarp();
        float v[64];
        tmem_ld32(tacc + (uint32_t)cg, *reinterpret_cast<float(*)[32]>(&v[0]));
        if (ncol > 32) tmem_ld32(tacc + (uint32_t)(cg + 32), *reinterpret_cast<float(*)[32]>(&v[32]));
        tmem_ld_wait();
        if (cg + 64 >= cmax) {                    // last read of this accumulator: hand it back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(tempty_bar(buf));
        }
        if (p.bias != nullptr) {
          if (bias_in_smem) {
            // packed f32x2 adds on 128-bit shared loads: 16 LDS.128 + 32 FADD2 instead of 64 LDS + 64 FADD (the epilogue's
            // instruction stream, not HBM, set the pace of the 1x1 convs).  Columns >= ncol are never stored.
            const float4* b4 = reinterpret_cast<const float4*>(sbias + co0 + cg);
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) {
              const float4 b = b4[jj];
              const float2 lo = __fadd2_rn(make_float2(v[4 * jj], v[4 * jj + 1]), make_float2(b.x, b.y));
              const float2 hi2 = __fadd2_rn(make_float2(v[4 * jj + 2], v[4 * jj + 3]), make_float2(b.z, b.w));
              v[4 * jj] = lo.x; v[4 * jj + 1] = lo.y; v[4 * jj + 2] = hi2.x; v[4 * jj + 3] = hi2.y;
            }
          } else {
#pragma unroll
            for (int jj = 0; jj < 64; ++jj)
              if (jj < ncol) v[jj] += __ldg(p.bias + co0 + cg + jj);
          }
        }
        if (do_stats) {
          // column sums of this warp's 32 rows, accumulated ON CHIP across the CTA's tiles (lane l owns
          // column 32h+l of the group); flushed with fp64 atomics only when the image changes / at the end
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            if (h * 32 < ncol) {
              // transpose this warp's 32 x 32 block through smem ([col][34]: conflict-free both ways); lane l
              // then owns column l and sums its 32 rows (x and x^2) -- ~2x fewer instructions than shuffles
#pragma unroll
              for (int jj = 0; jj < 32; ++jj) tr[jj * 34 + lane] = v[h * 32 + jj];
              __syncwarp();
              // packed f32x2: rows (2r, 2r+1) of this lane's column per LDS.64 (pitch 34: conflict-free both ways)
              float2 s2 = make_float2(0.f, 0.f), q2 = make_float2(0.f, 0.f);
#pragma unroll
              for (int r = 0; r < 16; ++r) {
                const float2 xv = *reinterpret_cast<const float2*>(&tr[lane * 34 + 2 * r]);
                s2 = __fadd2_rn(s2, xv);
                q2 = __ffma2_rn(xv, xv, q2);
              }
              const float cs = s2.x + s2.y, css = q2.x + q2.y;
              __syncwarp();
              f2sum_add(wsum[cg + h * 32 + lane], cs);
              f2sum_add(wsum[256 + cg + h * 32 + lane], css);
            }
          }
        }
        if (d.act != MSG_ACT_NONE) {              // activation, switch hoisted out of the element loop
          if (d.act == MSG_ACT_RELU) {
#pragma unroll
            for (int jj = 0; jj < 64; ++jj) v[jj] = fmaxf(v[jj], 0.f);
          } else if (d.act == MSG_ACT_LRELU) {
#pragma unroll
            for (int jj = 0; jj < 64; ++jj) v[jj] = v[jj] > 0.f ? v[jj] : 0.2f * v[jj];
          } else {
#pragma unroll
            for (int jj = 0; jj < 64; ++jj)
              if (jj < ncol) v[jj] = tanhf(v[jj]);
          }
        }
        if (nchw) {
          float* y = reinterpret_cast<float*>(p.y);
          const int plane = d.Ho * d.Wo;
          const int n = opix / plane, pp = opix - n * plane;
#pragma unroll
          for (int jj = 0; jj < 64; ++jj)
            if (jj < ncol)
              y[((size_t)n * d.Co_total + d.co_off + co0 + cg + jj) * plane + pp] = v[jj];
        } else if (p.tstore && vec && !accum && ncol == 64) {
          // ---- per-warp TMA store of [32 rows x 64 cols] through a 128B-swizzled staging buffer: no
          //      cross-warp barrier anywhere on the store path
          const uint32_t sb = sgrp & 1;
          if (lane == 0 && tma_pending) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
          __syncwarp();
          uint8_t* dstrow = stage_w + sb * 4096 + lane * 128;
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            float o[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) o[e] = v[g * 8 + e];
            *reinterpret_cast<uint4*>(dstrow + ((g ^ (lane & 7)) << 4)) = pack8(o);
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&mapC, stage_w_s + sb * 4096, d.co_off + co0 + cg, opix_w);
            tma_pending = true;
          }
          ++sgrp;
        } else if (vec && (ncol == 64 || ncol == 32 || ncol == 16)) {
          // ---- manual flush: per-warp skewed staging, then 16-byte chunks, consecutive lanes along a row
          if (p.tstore) {                         // the TMA buffers alias this region: drain them first
            if (lane == 0 && tma_pending) { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); tma_pending = false; }
            __syncwarp();
          }
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            if (g * 8 < ncol) {
              float o[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) o[e] = v[g * 8 + e];
              *reinterpret_cast<uint4*>(stage_w + lane * STAGE_PITCH + g * 16) = pack8(o);
            }
          }
          __syncwarp();
          const int lg = ncol == 64 ? 3 : (ncol == 32 ? 2 : 1);       // log2(chunks per row)
          __nv_bfloat16* ybase = reinterpret_cast<__nv_bfloat16*>(p.y) + d.co_off + co0 + cg;
#pragma unroll
          for (int itn = 0; itn < 8; ++itn) {
            const int idx = itn * 32 + lane;
            if (idx < (32 << lg)) {               // uniform per warp
              const int r = idx >> lg, ch = idx & ((1 << lg) - 1);
              uint4 val = *reinterpret_cast<const uint4*>(stage_w + r * STAGE_PITCH + ch * 16);
              const int op = __shfl_sync(0xffffffffu, opix, r);
              __nv_bfloat16* dst = ybase + (size_t)op * d.Co_total + ch * 8;
              if (accum) {
                float a[8], b[8];
                unpack8(val, a);
                unpack8(*reinterpret_cast<const uint4*>(dst), b);
#pragma unroll
                for (int e = 0; e < 8; ++e) a[e] += b[e];
                val = pack8(a);
              }
              *reinterpret_cast<uint4*>(dst) = val;
            }
          }
          __syncwarp();
        } else {
          __nv_bfloat16* y = reinterpret_cast<__nv_bfloat16*>(p.y) + (size_t)opix * d.Co_total + d.co_off + co0 + cg;
#pragma unroll
          for (int e = 0; e < 64; ++e)
            if (e < ncol) {
              float val = v[e];
              if (accum) val += __bfloat162float(y[e]);
              y[e] = __float2bfloat16_rn(val);
            }
        }
      }
    }
    if (do_stats) flush_stats();
    if (lane == 0 && tma_pending) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
  }
}

// ---- host side -------------------------------------------------------------------------------

struct Tiling { int Wt, R; };
bool pick_tiling(const msg_conv_desc* d, Tiling* t) {
  if (d->Wg >= 128) {
    if (d->Wg % 128) return false;
    t->Wt = 128; t->R = 1;
    return true;
  }
  if (128 % d->Wg) return false;
  t->Wt = d->Wg; t->R = 128 / d->Wg;
  return d->Hg % t->R == 0;
}
int pick_bn(int Cout) {
  int tiles = (Cout + 255) / 256;
  int per = (Cout + tiles - 1) / tiles;
  int bn = (per + 15) / 16 * 16;
  if (bn > 64 && bn % 64 && (bn + 63) / 64 * 64 <= 256) bn = (bn + 63) / 64 * 64;   // whole 64-column store groups
  return bn < 16 ? 16 : bn;
}

}  // namespace

bool conv2d_tma_supported(const msg_conv_desc* d, const void* x, const void* w, const void* y) {
  if (d->dtype != MSG_BF16) return false;
  if (d->flags & MSG_CONV_IN_NORM) {     // fused input InstanceNorm: 1x1 stride-1 convs whose tile lies in one image
    if (d->KH != 1 || d->KW != 1 || d->in_stride != 1 || d->pad_h || d->pad_w || d->Cin > 512) return false;
    if (((long long)d->Hg * d->Wg) % BM) return false;
    if (d->in_act != MSG_ACT_NONE && d->in_act != MSG_ACT_RELU && d->in_act != MSG_ACT_LRELU) return false;
  }
  if (d->Cin % 64 || (d->Ci_total & 7) || (d->ci_off & 7)) return false;
  if (((uintptr_t)x | (uintptr_t)w) & 15) return false;
  if (!(d->flags & MSG_CONV_OUT_NCHW_F32) && ((uintptr_t)y & 15)) return false;
  if (d->in_stride != 1 && d->in_stride != 2) return false;
  if ((d->flags & MSG_CONV_PER_IMAGE_W) && ((long long)d->Hg * d->Wg) % BM) return false;   // tiles inside one image
  Tiling t;
  if (!pick_tiling(d, &t)) return false;
  if (t.Wt * d->in_stride > 256 || t.R * d->in_stride > 256) return false;
  if ((long long)d->N * d->Hg * d->Wg / BM > 0x7fffffffLL / 8) return false;
  return get_encode() != nullptr;
}

int conv2d_tma(const msg_conv_desc* d, const void* x, const void* w, const float* bias, void* y,
               double* stats, const double* in_stats, const float* in_gamma, const float* in_beta, int in_img_stride, cudaStream_t st) {
  EncodeTiledFn enc = get_encode();
  MSG_REQUIRE(enc != nullptr, MSG_ERR_CUDA, "conv_tma: cuTensorMapEncodeTiled unavailable");
  Tiling tl;
  MSG_REQUIRE(pick_tiling(d, &tl), MSG_ERR_UNSUPPORTED, "conv_tma: unsupported plane geometry");
  TmaParams p;
  p.d = *d; p.bias = bias; p.y = y; p.stats = stats; p.in_stats = in_stats;
  p.in_gamma = in_gamma; p.in_beta = in_beta; p.in_img_stride = in_img_stride;
  p.xform = (d->flags & MSG_CONV_IN_NORM) ? 1 : 0;
  p.BN = pick_bn(d->Cout);
  p.n_tiles = (d->Cout + p.BN - 1) / p.BN;
  p.m_tiles = (int)((long long)d->N * d->Hg * d->Wg / BM);
  p.Wt = tl.Wt; p.R = tl.R;
  p.cblocks = d->Cin / 64;
  p.nkb = d->KH * d->KW * p.cblocks;
  p.tmem_cols = 32;
  while (p.tmem_cols < 2 * p.BN) p.tmem_cols <<= 1;
  const int K = d->KH * d->KW * d->Cin;
  static const bool env_bres = [] { const char* e = getenv("MSG_TMA_BRESIDENT"); return !(e && e[0] == '0'); }();
  p.b_resident = (env_bres && p.n_tiles == 1 && p.nkb * p.BN * BK * 2 <= 64 * 1024 && !(d->flags & MSG_CONV_PER_IMAGE_W)) ? 1 : 0;
  const int bres_bytes = p.b_resident ? p.nkb * p.BN * BK * 2 : 0;
  const int stage_bytes = A_BYTES + (p.b_resident ? 0 : p.BN * BK * 2);
  // two epilogue groups when the extra staging / scratch (57 KB) still leaves >= 3 pipeline stages
  static const int env_groups = [] { const char* e = getenv("MSG_TMA_EPI_GROUPS"); return e ? atoi(e) : 0; }();
  {
    const int st2 = (220 * 1024 - bres_bytes - (2 * (STAGE_BYTES + EPI_FIXED) + 4096 + 4096 + 320 + 1024)) / stage_bytes;
    // K-heavy tiles (many K blocks per tile) are L2->SM-bound and want the deep ring; the 1x1 convs (<= 4 K blocks
    // per tile) are epilogue-bound and fine with 2 stages
    p.epi_groups = (st2 >= 5 || (st2 >= 2 && p.nkb <= 4)) ? 2 : 1;
  }
  if (env_groups == 1 || env_groups == 2) p.epi_groups = env_groups;
  const int fixed = p.epi_groups * (STAGE_BYTES + EPI_FIXED) + 4096 + 4096 + 320 + 1024 + bres_bytes;
  static const bool env_tstore = [] { const char* e = getenv("MSG_TMA_STORE"); return !(e && e[0] == '0'); }();
  p.tstore = (env_tstore && !(d->flags & (MSG_CONV_OUT_NCHW_F32 | MSG_CONV_ACCUM)) && d->out_stride == 1 && d->out_off_h == 0 &&
              d->out_off_w == 0 && d->Ho == d->Hg && d->Wo == d->Wg && ((d->Co_total | d->co_off) & 7) == 0 &&
              (((uintptr_t)y) & 15) == 0) ? 1 : 0;
  int stages = (220 * 1024 - fixed) / stage_bytes;
  if (stages > (p.b_resident ? 8 : 6)) stages = p.b_resident ? 8 : 6;
  if (stages < 2) stages = 2;
  p.stages = stages;
  const size_t smem = (size_t)stages * stage_bytes + fixed;

  CUtensorMap mapA, mapB;
  {
    cuuint64_t dims[4] = {(cuuint64_t)d->Cin, (cuuint64_t)d->Wi, (cuuint64_t)d->Hi, (cuuint64_t)d->N};
    cuuint64_t strides[3] = {(cuuint64_t)d->Ci_total * 2, (cuuint64_t)d->Wi * d->Ci_total * 2,
                             (cuuint64_t)d->Hi * d->Wi * d->Ci_total * 2};
    cuuint32_t box[4] = {(cuuint32_t)BK, (cuuint32_t)(tl.Wt * d->in_stride), (cuuint32_t)(tl.R * d->in_stride), 1};
    cuuint32_t es[4] = {1, (cuuint32_t)d->in_stride, (cuuint32_t)d->in_stride, 1};
    void* base = (void*)((const __nv_bfloat16*)x + d->ci_off);
    CUresult r = enc(&mapA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, base, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "conv_tma: cuTensorMapEncodeTiled(A) failed with %d", (int)r);
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)d->Cout * ((d->flags & MSG_CONV_PER_IMAGE_W) ? d->N : 1)};
    cuuint64_t strides[1] = {(cuuint64_t)K * 2};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)p.BN};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(&mapB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)w, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "conv_tma: cuTensorMapEncodeTiled(B) failed with %d", (int)r);
  }
  CUtensorMap mapC = mapB;   // unused unless tstore
  if (p.tstore) {
    cuuint64_t dims[2] = {(cuuint64_t)d->Co_total, (cuuint64_t)d->N * d->Ho * d->Wo};
    cuuint64_t strides[1] = {(cuuint64_t)d->Co_total * 2};
    cuuint32_t box[2] = {64, 32};   // one epilogue warp's rows
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(&mapC, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, y, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "conv_tma: cuTensorMapEncodeTiled(C) failed with %d", (int)r);
  }
  static DeviceOnce attr_set;     // cudaFuncSetAttribute is per device
  if (attr_set.needed()) {
    cudaError_t e = cudaFuncSetAttribute(conv_tma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    MSG_REQUIRE(e == cudaSuccess, MSG_ERR_CUDA, "conv_tma: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    attr_set.done();
  }
  int grid = sm_count();
  const int total = p.m_tiles * p.n_tiles;
  if (grid > total) grid = total;
  if (p.xform) conv_tma_kernel<true><<<grid, 64 + 128 * p.epi_groups + 128, smem, st>>>(mapA, mapB, mapC, p);
  else conv_tma_kernel<false><<<grid, 64 + 128 * p.epi_groups, smem, st>>>(mapA, mapB, mapC, p);
  return check_launch("conv_tma_kernel");
}

}  // namespace msg
