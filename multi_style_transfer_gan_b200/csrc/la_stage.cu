// Fused LocalAttention stage (enhanced_generator.py:13-47), ONE tcgen05 kernel per stage (sm_100a, bf16):
//
//     [InstanceNorm + ReLU of the producing conv, applied to the landed tile]  ->  qkv 1x1 conv  ->  per 4x4 window:
//     S = normalize(q) normalize(k)^T  [C x C]  ->  softmax over the last dim  ->  P v  ->  proj 1x1 conv
//
// The reference materialises qkv ([.., 3C]), the window-permuted copies, the logits ([nW, C, C], larger than the
// activation), the attention output and the projected output in global memory; round 1 ran three launches with a 3C
// channel HBM round trip.  Here the only HBM traffic is the C-channel input tile and the C-channel output tile.
//
// Tile = 128 pixels = 8 windows (4 rows x 32 columns of one image), brought in by a 5-D TMA box ordered
// (channel, x-in-window, y-in-window, window column) so that tile row r = 16 * window + pixel-in-window.
//
//   warp 0      TMA producer: x tiles; at C=128 also the streamed weight K blocks (C=64: weights resident in smem)
//   warp 1      issuer G: the 1x1-conv GEMMs on tcgen05 -- qkv as three N=C chunks (q | k | v) of M=128 pixels into a
//               two-slot TMEM accumulator ring, and the projection of the PREVIOUS tile (A operand = attention output,
//               MN-major in smem)
//   warp 2      issuer A: per window (C=128) / window pair (C=64, block-diagonal) S = Qh^T Kh as ONE tcgen05.mma with both
//               operands MN-major (K = the 16 pixels), then P.V with the A operand read FROM TENSOR MEMORY (P is written
//               back over S by the softmax warps, FA4 style) and V (+ a group of all-ones rows that yields the softmax row
//               sums in fp32 for free) K-major from smem; S/P/O double-buffered in TMEM
//   warp 3      issuer PV (see issuer A)
//   warps 4-11  drain: tcgen05.ld of the q / k / v accumulators (thread = pixel and one half of the channels; the two halves of
//               a pixel exchange their partial sums of squares through shared memory), normalise, -> bf16 (q, k, k
//               pre-multiplied by log2 e) / fp16 (v) operand tiles.  A single warp per 32 pixels was the pace-setter of the
//               kernel (one serial instruction stream, ~5 cycles per instruction)
//   next 12 / 16  softmax + O drain: one group per S buffer; tcgen05.ld S (thread = row i; at C=128 two warps per row, each half
//               of the columns), exp2 (half MUFU, half packed fp16 polynomial on the FMA pipe; |S| <= 1 so no running max),
//               tcgen05.st P (fp16) over consumed S columns; then O / rowsum -> bf16 -> the projection's A operand
//   last 4      InstanceNorm + ReLU of the landed x tile in shared memory, exactly the arithmetic of the stand-alone apply
//               kernel (as conv_tma.cu), alternating with the epilogue of the previous tile: projection accumulators -> bf16
//               -> 128B-swizzled staging -> per-warp 5-D TMA store
//
// Biases ride on the tensor pipe: the q / k / proj GEMMs get one extra K=16 step whose A operand is a constant [1, 1, 0, ...]
// row and whose B rows are [hi(b_n), lo(b_n), 0, ...] (bf16 split: 16 mantissa bits), and the v bias is two extra rows of the
// P.V product's B operand beside the all-ones row that yields the softmax row sums -- no bias arithmetic on the CUDA cores.
//
// TMEM (512 columns): [0, 2C) accumulator ring (slot 0: q, v; slot 1: k, proj), then the 128-column S buffers; inside an
// S buffer P occupies columns [0, 32) (+ [64, 96) at C=128) and O columns [32, 32 + N_pv).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdlib.h>

#include "common.cuh"
#include "la_mma.cuh"
#include "tcgen05.cuh"

namespace msg {
namespace {
using namespace tc;

// every MSG_LA_MUFU_EVERY-th pair of exponentials on the MUFU (one MUFU.EX2.F16 per HALF: 8 XU cycles per warp instruction and
// value pair), the others as a packed degree-4 polynomial on the FMA pipe (4 HFMA2 per pair); 0 = polynomial only
#ifndef MSG_LA_MUFU_EVERY
#define MSG_LA_MUFU_EVERY 2
#endif
#ifndef MSG_LA_SLEEP_NS
#define MSG_LA_SLEEP_NS 40
#endif
#if MSG_LA_SLEEP_NS > 0
#define MBW(b, ph) mbar_wait_sleep<MSG_LA_SLEEP_NS>(b, ph)
#else
#define MBW(b, ph) mbar_wait(b, ph)
#endif

template <int C>
struct Cfg {
  static constexpr int KB = C / 64;                    // 64-channel blocks
  static constexpr int UNITS = C == 64 ? 4 : 8;        // attention units per tile: window pairs (C=64) / windows (C=128)
  static constexpr int NPV = C == 64 ? 48 : 32;        // N of the P.V MMA: [16 px | 8 ones] per window (+ 8 don't-care at C=128)
  static constexpr int NBUF = C == 64 ? 3 : 2;         // S / P / O buffers in tensor memory (units in flight)
  static constexpr int NSET = C == 64 ? 2 : 1;         // q / k / v operand sets in shared memory (tiles in flight)
  static constexpr int XS = C == 64 ? 2 : 1;           // x-tile stages (a consumed stage doubles as the output staging)
  static constexpr int WS = 2;                         // streamed-weight stages (C=128)
  static constexpr int X_TILE = 128 * 128;             // one K block of an x tile: 128 pixel rows x 128 B
  static constexpr int X_BYTES = KB * X_TILE;
  static constexpr int OFF_X = 0;
  static constexpr int W_BYTES = C == 64 ? (192 + 64) * 128 : WS * 128 * 128;
  static constexpr int OFF_W = OFF_X + XS * X_BYTES;
  static constexpr int QK_BYTES = KB * 8 * 2048;       // [mn block][window][16 pixel rows x 128 B]
  static constexpr int V_KB = 8 * 3072;                // per K block: [window][16 pixel rows + 8 ones rows][128 B]
  static constexpr int V_BYTES = KB * V_KB;
  static constexpr int SET_BYTES = 2 * QK_BYTES + V_BYTES;     // q | k | v of one tile
  static constexpr int OFF_SET = OFF_W + W_BYTES;
  static constexpr int OFF_A = OFF_SET + NSET * SET_BYTES + 1024;   // (+ the don't-care 4th row group of the last window at C=128)
  static constexpr int A_BYTES = KB * 128 * 128;       // attention output = A operand of the projection
  // output staging of the epilogue: at C=128 (one x stage, no spare smem) it aliases the x stage, which the qkv GEMMs of
  // the NEXT tile have consumed by the time the projection completes; at C=64 it is its own region
  static constexpr bool STG_ALIAS_X = C == 128;
  static constexpr int OFF_STG = STG_ALIAS_X ? OFF_X : OFF_A + A_BYTES;
  // bias operands (no-swizzle K-major core matrices, 16 B per row): the constant ones rows, a zero block that serves as the
  // second K chunk of every bias descriptor, and the [hi, lo] rows of the q | k | proj biases
  static constexpr int OFF_ONES = OFF_A + A_BYTES + (STG_ALIAS_X ? 0 : A_BYTES);
  static constexpr int OFF_BIASB = OFF_ONES + 2048;
  static constexpr int OFF_ZERO = OFF_BIASB + 3 * C * 16;       // (after both: the descriptors' chunk distance is unsigned)
  static constexpr int OFF_EX = OFF_ZERO + 2048;                // [tile parity][channel half][pixel] partial (sum q^2, sum k^2)
  static constexpr int OFF_XF = OFF_EX + 2 * 2 * 128 * 8;       // fused input norm: scale[C], shift[C]
  static constexpr int OFF_BAR = OFF_XF + 2 * C * 4;
  static constexpr int SMEM = OFF_BAR + 512 + 1024;    // + alignment slack
  static constexpr int SCOL0 = 2 * C;                  // first S buffer column
  static constexpr int OOFF = 32;                      // O columns inside an S buffer
  static constexpr int SMH = C == 64 ? 1 : 2;          // softmax warps per S row (column halves)
  static constexpr int NSMW = 4 * NBUF * SMH;          // softmax warps
  static constexpr int NWARPS = 12 + NSMW + 4;
  static_assert(OFF_A % 1024 == 0 && OFF_SET % 1024 == 0 && SET_BYTES % 1024 == 0, "operand tiles must be 1024-byte aligned");
  static_assert(SMEM <= 227 * 1024, "shared memory budget");
  static_assert(SCOL0 + NBUF * 128 <= 512, "tensor memory budget");
};

struct LaParams {
  int N, H, W;
  int tiles_w, tiles_per_img, total_tiles;
  const float* bqkv;
  const float* bproj;
  const double* in_stats;     // XF: raw plane sums [N][C][2] of the input tensor
  const float* in_gamma;      // XF: optional affine of the input norm (common.cuh: in_affine), or null
  const float* in_beta;
  int in_img_stride;
  int in_act;
  unsigned long long* trace;  // MSG_LA_TRACE builds only: [role][event] = (tag, clock) pairs of CTA 0
};

#ifdef MSG_LA_TRACE
// timeline instrumentation (development builds: MSG_LA_TRACE=1 python -m multi_style_transfer_gan_b200.build):
// lane 0 of each role of CTA 0 appends (event, tile, unit, clock64) -- read back with tools/la_trace.py
#define TR_DECL_IF(role, cond) unsigned long long* tr_ = (p.trace && blockIdx.x == 0 && lane == 0 && (cond)) ? p.trace + (role) * 4096 : nullptr; int tr_n = 0
#define TR_DECL(role) TR_DECL_IF(role, true)
#define TR(ev, lt_, u_) do { if (tr_ && tr_n < 2047) { tr_[2 * tr_n] = ((unsigned long long)(ev) << 32) | ((unsigned long long)(lt_) << 8) | (unsigned long long)(u_); tr_[2 * tr_n + 1] = clock64(); ++tr_n; tr_[4094] = tr_n; } } while (0)
#else
#define TR_DECL(role) do {} while (0)
#define TR_DECL_IF(role, cond) do {} while (0)
#define TR(ev, lt_, u_) do {} while (0)
#endif

enum Bar {
  B_XFULL = 0, B_XEMPTY = 2, B_XFDONE = 4, B_WFULL = 6, B_WEMPTY = 8, B_WRES = 10,
  B_ACCFULL = 11, B_ACCEMPTY = 13,      // accumulator ring: slot 0 = q, v (in that order, one consumer); slot 1 = k
  B_PFULL = 15, B_PEMPTY = 16,          // projection accumulators (TMEM slot 1, shared with k): their own barriers, because a parity wait
                                        // only separates ADJACENT phases and slot 1 has two consumers (drain warps: k; epilogue warps: proj)
  B_STFREE = 17,                        // the output staging (= a consumed x stage) has been read by the TMA stores
  B_ASREADY = 18,                       // attention output of a tile complete in smem (8 softmax / O-drain warps)
  B_VREADY = 19,                        // [set]
  B_QKREADY = 21,                       // [set][drain warp]: q and k rows of that warp's two windows written
  B_WINFREE = 29,                       // [set][drain warp]: the MMAs reading that warp's windows (S and P.V) have completed
  B_SFULL = 37, B_PREADY = 40, B_OFULL = 43, B_OEMPTY = 46,      // [S buffer]
  B_COUNT = 49
};

__device__ __forceinline__ uint32_t pack_f16x2_rn(float lo, float hi) {
  __half2 t = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ uint32_t pack_bf16x2_rn(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
// after tcgen05.wait::ld: pins every later use of the loaded registers behind the wait (the load's asm statement names them as
// outputs, so without this the compiler may schedule a use between the load and the wait)
template <int N>
__device__ __forceinline__ void reg_fence(float (&v)[N]) {
#pragma unroll
  for (int i = 0; i < N; ++i) asm volatile("" : "+f"(v[i])::"memory");
}
// sum of squares of N values on four independent chains (two packed accumulators)
template <int N>
__device__ __forceinline__ void sumsq(const float (&v)[N], float2& a0, float2& a1) {
#pragma unroll
  for (int j = 0; j < N; j += 4) {
    const float2 x0 = make_float2(v[j], v[j + 1]), x1 = make_float2(v[j + 2], v[j + 3]);
    a0 = __ffma2_rn(x0, x0, a0);
    a1 = __ffma2_rn(x1, x1, a1);
  }
}
template <int N>
__device__ __forceinline__ void tmem_ldN(uint32_t taddr, float (&v)[N]) {
  if constexpr (N == 32) tmem_ld32(taddr, v); else tmem_ld16(taddr, v);
}
// One pass over COLS columns of an accumulator slot in CH-column chunks, the tcgen05.ld of chunk i + 1 in flight while chunk i
// is processed (a load + wait per chunk cost ~300 cycles of exposed latency each: the drain warps were the pace-setter of the
// kernel).  released() runs once the LAST load has completed: the slot may be handed back to the MMA issuer.
template <int COLS, int CH, class F, class R>
__device__ __forceinline__ void acc_pass(uint32_t taddr, F&& f, R&& released) {
  constexpr int NCH = COLS / CH;
  float va[CH], vb[CH];
  tmem_ldN<CH>(taddr, va);
#pragma unroll
  for (int i = 0; i < NCH; ++i) {
    float(&cur)[CH] = (i & 1) ? vb : va;
    float(&nxt)[CH] = (i & 1) ? va : vb;
    tmem_ld_wait();
    reg_fence(cur);
    if (i + 1 < NCH) tmem_ldN<CH>(taddr + CH * (i + 1), nxt);
    else released();
    f(CH * i, cur);
  }
}

// AFF (with XF): the input norm has a per-image affine.  A template parameter so that the affine-free kernel keeps its register
// allocation (C = 128 spills in its transform warps).
template <int C, bool XF, bool AFF = false>
__global__ void __launch_bounds__(32 * Cfg<C>::NWARPS, 1)
la_stage_kernel(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapWqkv,
                const __grid_constant__ CUtensorMap mapWproj, const __grid_constant__ CUtensorMap mapOut, const LaParams p) {
  using K = Cfg<C>;
  constexpr int KB = K::KB, UNITS = K::UNITS, NBUF = K::NBUF, NSET = K::NSET, XS = K::XS;
  constexpr int SM0 = 12;                    // first softmax warp
  constexpr int CH = C == 64 ? 32 : 16;      // accumulator drain chunk (columns): 1024 threads at C=128 leave 64 registers each
  constexpr int EP0 = SM0 + K::NSMW;         // first transform / epilogue warp
  extern __shared__ uint8_t smem_raw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sX = base + K::OFF_X, sW = base + K::OFF_W, sSet = base + K::OFF_SET, sA = base + K::OFF_A, sBar = base + K::OFF_BAR;
  const uint32_t sOnes = base + K::OFF_ONES, sZero = base + K::OFF_ZERO, sBiasB = base + K::OFF_BIASB;
  float2* ex = reinterpret_cast<float2*>(gen + K::OFF_EX);
  float* xf_tab = reinterpret_cast<float*>(gen + K::OFF_XF);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gen + K::OFF_BAR + 8 * B_COUNT);
  auto bar = [&](int i) { return sBar + 8u * (uint32_t)i; };

  // ---- one-time setup
  // bias operands: ones rows [1, 1, 0 ...], the zero chunk, [hi, lo, 0 ...] rows of the q | k | proj biases (bf16 split)
  for (int i = tid; i < 128; i += (int)blockDim.x) {
    *reinterpret_cast<uint4*>(gen + K::OFF_ONES + i * 16) = make_uint4(0x3F803F80u, 0u, 0u, 0u);
    *reinterpret_cast<uint4*>(gen + K::OFF_ZERO + i * 16) = make_uint4(0u, 0u, 0u, 0u);
  }
  for (int i = tid; i < 3 * C; i += (int)blockDim.x) {
    const float b = i < 2 * C ? p.bqkv[i] : p.bproj[i - 2 * C];
    const __nv_bfloat16 bh = __float2bfloat16_rn(b);
    const __nv_bfloat16 bl = __float2bfloat16_rn(b - __bfloat162float(bh));
    *reinterpret_cast<uint4*>(gen + K::OFF_BIASB + i * 16) =
        make_uint4((uint32_t)__bfloat16_as_ushort(bh) | ((uint32_t)__bfloat16_as_ushort(bl) << 16), 0u, 0u, 0u);
  }
  // the extra row group of every window of V (fp16): row 0 all ones (P.[ones] = softmax row sums, accumulated in fp32 by the
  // MMA), rows 1, 2 = hi / lo of the v bias (P.[b] / rowsum = the bias term of the attention output), rows 3-7 zero
  for (int i = tid; i < NSET * KB * 8 * 64; i += (int)blockDim.x) {
    const int set = i / (KB * 8 * 64), r = i - set * (KB * 8 * 64);
    const int kb = r / (8 * 64), w = (r / 64) & 7, rr = (r >> 3) & 7, ch = r & 7;
    uint4 val = make_uint4(0u, 0u, 0u, 0u);
    if (rr == 0) val = make_uint4(0x3C003C00u, 0x3C003C00u, 0x3C003C00u, 0x3C003C00u);
    else if (rr <= 2) {
      uint32_t o[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        __half h2[2];
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          const float b = p.bqkv[2 * C + kb * 64 + ch * 8 + 2 * e + t];
          const __half bh = __float2half_rn(b);
          h2[t] = rr == 1 ? bh : __float2half_rn(b - __half2float(bh));
        }
        o[e] = (uint32_t)__half_as_ushort(h2[0]) | ((uint32_t)__half_as_ushort(h2[1]) << 16);
      }
      val = make_uint4(o[0], o[1], o[2], o[3]);
    }
    *reinterpret_cast<uint4*>(gen + K::OFF_SET + set * K::SET_BYTES + 2 * K::QK_BYTES + kb * K::V_KB + w * 3072 + 2048 + rr * 128 +
                              ((ch ^ rr) << 4)) = val;
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < 2; ++s) {
        mbar_init(bar(B_XFULL + s), 1); mbar_init(bar(B_XEMPTY + s), 1); mbar_init(bar(B_XFDONE + s), 4);
        mbar_init(bar(B_WFULL + s), 1); mbar_init(bar(B_WEMPTY + s), 1);
        mbar_init(bar(B_ACCFULL + s), 1); mbar_init(bar(B_ACCEMPTY + s), 8);
        mbar_init(bar(B_VREADY + s), 8);
      }
      for (int s = 0; s < 8; ++s) { mbar_init(bar(B_QKREADY + s), 2); mbar_init(bar(B_WINFREE + s), 1); }
      for (int s = 0; s < 3; ++s) {
        mbar_init(bar(B_SFULL + s), 1); mbar_init(bar(B_PREADY + s), 4 * K::SMH); mbar_init(bar(B_OFULL + s), 1); mbar_init(bar(B_OEMPTY + s), 4 * K::SMH);
      }
      mbar_init(bar(B_WRES), 1); mbar_init(bar(B_PFULL), 1); mbar_init(bar(B_PEMPTY), 4); mbar_init(bar(B_STFREE), 4);
      mbar_init(bar(B_ASREADY), K::NSMW);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  } else if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapX)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapWqkv)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapWproj)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapOut)) : "memory");
  }
  fence_proxy_async();        // the generic-proxy ones rows above are read by tcgen05.mma
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  // contiguous tile range of this CTA (same image, neighbouring tiles; the norm table is rebuilt per image)
  const int t_begin = (int)((long long)blockIdx.x * p.total_tiles / gridDim.x);
  const int t_end = (int)((long long)(blockIdx.x + 1) * p.total_tiles / gridDim.x);
  const int T = t_end - t_begin;
  auto tile_coords = [&](int t, int& img, int& h0, int& wc0) {
    img = t / p.tiles_per_img;
    const int rem = t - img * p.tiles_per_img;
    const int th = rem / p.tiles_w;
    h0 = th * 4;
    wc0 = (rem - th * p.tiles_w) * 8;
  };
  const uint32_t hi = (uint32_t)(make_sw128_desc(0) >> 32);     // SBO = 1024, version, SWIZZLE_128B: shared by every descriptor here

  if (warp == 0) {
    // =========================================== TMA producer ===========================================
    if (lane == 0) {
      TR_DECL(0);
      if (C == 64) {
        mbar_expect_tx(bar(B_WRES), (192 + 64) * 128);
        tma_load_2d(sW, &mapWqkv, bar(B_WRES), 0, 0);
        tma_load_2d(sW + 192 * 128, &mapWproj, bar(B_WRES), 0, 0);
      }
      int ws = 0;
      uint32_t wn = 0;                                   // weight loads issued
      auto wload = [&](const CUtensorMap* m, int col, int row) {
        if (wn >= (uint32_t)K::WS) MBW(bar(B_WEMPTY + ws), ((wn / K::WS) - 1) & 1);
        mbar_expect_tx(bar(B_WFULL + ws), 128 * 128);
        tma_load_2d(sW + ws * (128 * 128), m, bar(B_WFULL + ws), col, row);
        ws ^= 1; ++wn;
      };
      for (int lt = 0; lt < T; ++lt) {
        int img, h0, wc0;
        tile_coords(t_begin + lt, img, h0, wc0);
        const int xs = lt % XS;
        if (lt >= XS) MBW(bar(B_XEMPTY + xs), ((lt / XS) - 1) & 1);
        // C=128: the stage was the output staging of tile lt - 2, whose TMA stores must have finished reading it (the epilogue of
        // tile lt - 1 cannot have completed yet -- its projection is issued after the qkv GEMMs of THIS tile -- so the parity
        // wait is on an adjacent phase)
        if (K::STG_ALIAS_X && lt >= 2) MBW(bar(B_STFREE), (lt - 2) & 1);
        TR(1, lt, 0);
        mbar_expect_tx(bar(B_XFULL + xs), K::X_BYTES);
        for (int kb = 0; kb < KB; ++kb)
          tma_load_5d(sX + xs * K::X_BYTES + kb * K::X_TILE, &mapX, bar(B_XFULL + xs), kb * 64, 0, h0, wc0, img);
        if (C == 128) {
          for (int ch = 0; ch < 3; ++ch)
            for (int kb = 0; kb < KB; ++kb) wload(&mapWqkv, kb * 64, ch * 128);
          if (lt > 0)
            for (int kb = 0; kb < KB; ++kb) wload(&mapWproj, kb * 64, 0);
        }
      }
      if (C == 128 && T > 0)
        for (int kb = 0; kb < KB; ++kb) wload(&mapWproj, kb * 64, 0);
    }
  } else if (warp == 1) {
    // =========================================== issuer G: qkv chunks + projection of the previous tile =================
    const bool leader = elect_one();
    TR_DECL(1);
    const uint32_t idesc_qkv = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(C >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    const uint32_t idesc_proj = idesc_qkv | (1u << 15);          // A = attention output, MN-major
    // bias step: A = the ones rows, B = [hi, lo] bias rows n0 .. n0 + C (both no-swizzle K-major, second K chunk = the zero block)
    const uint32_t hi_ns = (uint32_t)(128 >> 4) | (1u << 14);
    const uint32_t ones_lo = (sOnes >> 4) | (((sZero - sOnes) >> 4) << 16);
    auto bias_mma = [&](uint32_t tacc, int n0) {
      const uint32_t b0 = sBiasB + (uint32_t)n0 * 16u;
      umma_bf16_lo(tacc, ones_lo, (b0 >> 4) | (((sZero - b0) >> 4) << 16), hi_ns, idesc_qkv, true);
    };
    int ws = 0;
    uint32_t wn = 0;
    if (C == 64) MBW(bar(B_WRES), 0);
    auto wwait = [&]() {                                          // next streamed weight stage -> its descriptor word
      MBW(bar(B_WFULL + ws), (wn / K::WS) & 1);
      const uint32_t lo = (sW + ws * (128 * 128)) >> 4;
      return lo;
    };
    auto wdone = [&]() {
      if (leader) umma_commit(bar(B_WEMPTY + ws));
      ws ^= 1; ++wn;
    };
    auto proj = [&](int lt) {
      // TMEM slot 1 is used in the order k(0), k(1), proj(0), k(2), proj(1), ..., proj(T-1): its previous user is k(lt+1)
      // (drained by the drain warps: ACCEMPTY[1] phase lt+1), or for the last tile proj(T-2) / k(0)
      if (lt < T - 1) MBW(bar(B_ACCEMPTY + 1), (lt + 1) & 1);
      else if (T == 1) MBW(bar(B_ACCEMPTY + 1), 0);
      else MBW(bar(B_PEMPTY), (T - 2) & 1);
      MBW(bar(B_ASREADY), lt & 1);
      tc_fence_after();
      TR(10, lt, 0);
      const uint32_t tacc = tmem + C;
      const uint32_t a_lo0 = (sA >> 4) | ((uint32_t)((C * 128) >> 4) << 16);       // LBO = next 64-pixel block
      for (int kb = 0; kb < KB; ++kb) {
        uint32_t b_lo;
        if (C == 128) { b_lo = wwait(); tc_fence_after(); } else b_lo = (sW + 192 * 128) >> 4;
        if (leader) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16_lo2(tacc, a_lo0 + (uint32_t)((kb * 4 + k) * 128), hi, b_lo + 2 * k, hi, idesc_proj, (kb | k) != 0);
        }
        __syncwarp();
        if (C == 128) wdone();
      }
      if (leader) {
        bias_mma(tacc, 2 * C);
        umma_commit(bar(B_PFULL));
      }
      __syncwarp();
      TR(11, lt, 0);
    };
    for (int lt = 0; lt < T; ++lt) {
      const int xs = lt % XS;
      MBW(bar((XF ? B_XFDONE : B_XFULL) + xs), (lt / XS) & 1);
      tc_fence_after();
      TR(1, lt, 0);
      for (int ch = 0; ch < 3; ++ch) {
        const int slot = ch & 1;
        if (slot == 0) {                 // slot 0: q(lt) = use 2 lt, v(lt) = use 2 lt + 1, one consumer (the drain warps)
          const int n = 2 * lt + (ch >> 1);
          if (n >= 1) MBW(bar(B_ACCEMPTY + 0), (n - 1) & 1);
        } else if (lt == 1) {            // slot 1 before k(1): k(0) drained
          MBW(bar(B_ACCEMPTY + 1), 0);
        } else if (lt >= 2) {            // slot 1 before k(lt): proj(lt-2) drained by the epilogue warps
          MBW(bar(B_PEMPTY), (lt - 2) & 1);
        }
        tc_fence_after();
        TR(2, lt, ch);
        const uint32_t tacc = tmem + slot * C;
        for (int kb = 0; kb < KB; ++kb) {
          uint32_t b_lo;
          if (C == 128) { b_lo = wwait(); tc_fence_after(); } else b_lo = (sW + ch * 64 * 128) >> 4;
          const uint32_t a_lo = (sX + xs * K::X_BYTES + kb * K::X_TILE) >> 4;
          if (leader) {
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16_lo(tacc, a_lo + 2 * k, b_lo + 2 * k, hi, idesc_qkv, (kb | k) != 0);
          }
          __syncwarp();
          if (C == 128) wdone();
        }
        if (leader) {
          if (ch < 2) bias_mma(tacc, ch * C);          // (the v bias rides in the P.V product)
          umma_commit(bar(B_ACCFULL + slot));
        }
        __syncwarp();
        TR(3, lt, ch);
      }
      if (leader) umma_commit(bar(B_XEMPTY + xs));
      __syncwarp();
      if (lt > 0) proj(lt - 1);
    }
    if (T > 0) proj(T - 1);
  } else if (warp == 2 || warp == 3) {
    // =========================================== issuers A: S = Qh^T Kh (warp 2) and O = P V (warp 3) per unit =====================
    // Two issuing warps, each an in-order stream with blocking (hardware-suspended) barrier waits: S(g) goes out as soon as
    // buffer g % NBUF is free and the unit's q / k rows are written; P.V(g) as soon as its softmax is done -- neither stream can
    // hold back the other (one in-order issuer stalled the P.V products of a tile behind the S of the next one; a polling issuer
    // burns the issue slots of the scheduler it shares with a quarter of the softmax warps).
    const bool leader = elect_one();
    const uint32_t idesc_s = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    const uint32_t idesc_pv = (1u << 4) | ((uint32_t)(K::NPV >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);   // fp16 x fp16
    constexpr uint32_t QK_LBO = C == 64 ? 2048 : 8 * 2048;       // next 64 rows of M / N: the pair's other window / the next channel block
    constexpr uint32_t UNIT_Q = C == 64 ? 2 * 2048 : 2048;       // bytes of q / k per unit
    constexpr uint32_t UNIT_V = C == 64 ? 2 * 3072 : 3072;
    TR_DECL(warp == 2 ? 2 : 23);
    const int total = T * UNITS;
    if (warp == 2) {
      for (int g = 0; g < total; ++g) {
        const int lt = g / UNITS, u = g - lt * UNITS;
        const int set = lt % NSET, b = g % NBUF;
        if (g >= NBUF) MBW(bar(B_OEMPTY + b), ((g / NBUF) - 1) & 1);            // unit g - NBUF drained: the buffer is free
        if (C == 64 || !(u & 1)) MBW(bar(B_QKREADY + set * 4 + (C == 64 ? u : (u >> 1))), (lt / NSET) & 1);
        tc_fence_after();
        TR(2, lt, u);
        if (leader) {
          const uint32_t q0 = sSet + set * K::SET_BYTES + u * UNIT_Q;
          const uint32_t a_lo = (q0 >> 4) | ((QK_LBO >> 4) << 16);
          const uint32_t b_lo = ((q0 + K::QK_BYTES) >> 4) | ((QK_LBO >> 4) << 16);
          umma_bf16_lo(tmem + K::SCOL0 + b * 128, a_lo, b_lo, hi, idesc_s, false);
          umma_commit(bar(B_SFULL + b));
        }
        __syncwarp();
      }
    } else {
      for (int g = 0; g < total; ++g) {
        const int lt = g / UNITS, u = g - lt * UNITS;
        const int set = lt % NSET, b = g % NBUF;
        if (u == 0) MBW(bar(B_VREADY + set), (lt / NSET) & 1);
        MBW(bar(B_PREADY + b), (g / NBUF) & 1);
        tc_fence_after();
        TR(4, lt, u);
        if (leader) {
          const uint32_t scol = tmem + K::SCOL0 + b * 128;
          const uint32_t v0 = sSet + set * K::SET_BYTES + 2 * K::QK_BYTES + u * UNIT_V;
#pragma unroll
          for (int ks = 0; ks < C / 16; ++ks) {
            const uint32_t b_lo = (v0 + (ks >> 2) * K::V_KB + (ks & 3) * 32) >> 4;
            // P of channels [64 h, 64 h + 64) sits in columns [64 h, 64 h + 32): written over S columns its own warps consumed
            const uint32_t pcol = C == 64 ? (uint32_t)(ks * 8) : (uint32_t)((ks >> 2) * 64 + (ks & 3) * 8);
            umma_ts_lo(scol + K::OOFF, scol + pcol, b_lo, hi, idesc_pv, ks != 0);
          }
          umma_commit(bar(B_OFULL + b));
          // The windows of drain warp w = (C == 64 ? u : u / 2) are free once this P.V has completed: its S product finished
          // before the softmax that produced P (so before this instruction was issued), although another warp issued it.
          if (C == 64 || (u & 1)) umma_commit(bar(B_WINFREE + set * 4 + (C == 64 ? u : (u >> 1))));
        }
        __syncwarp();
      }
    }
  } else if (warp >= 4 && warp < 12) {
    // =========================================== drain: q / k / v accumulators -> operand tiles ==========================
    // S only needs the PRODUCT 1 / (|q_p| |k_p|) per pixel p (the contraction index), so q is stored raw and k carries both norms
    // (and log2 e).  Thread = (pixel, channel half); the sums of squares of q and k are taken as soon as the accumulators are
    // full and exchanged between the two halves of a pixel; the (short) write passes wait until the MMAs of the previous tile of
    // this set have finished reading this warp's two windows.
    const int q = warp & 3, h = (warp - 4) >> 2;
    const int r = q * 32 + lane;               // tile row = pixel: window r >> 4, pixel-in-window r & 15
    const int w = r >> 4, px = r & 15;
    constexpr int CW = C / 2;                  // channels per thread
    const int cb = h * CW;
    const uint32_t lane_addr = ((uint32_t)(q * 32) << 16) + (uint32_t)cb;
    const uint32_t row_off = (uint32_t)(w * 2048 + (px >> 3) * 1024 + (px & 7) * 128);       // inside a q / k mn-block
    const uint32_t vrow_off = (uint32_t)(w * 3072 + (px >> 3) * 1024 + (px & 7) * 128);      // inside a v K block
    const int sw = px & 7;
    TR_DECL_IF(3 + q, h == 0);
    for (int lt = 0; lt < T; ++lt) {
      const int set = lt % NSET;
      uint8_t* set_base = gen + K::OFF_SET + set * K::SET_BYTES;
      float2 sq0 = make_float2(0.f, 0.f), sq1 = sq0, sk0 = sq0, sk1 = sq0;
      auto release = [&](int slot) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(B_ACCEMPTY + slot));
      };
      auto store = [&](uint8_t* dst0, int c0, const uint32_t (&o)[CH / 2], int kb_stride) {       // c0: absolute first channel
        uint8_t* dst = dst0 + (c0 >> 6) * kb_stride;
        const int cc0 = (c0 & 63) >> 3;
#pragma unroll
        for (int g = 0; g < CH / 8; ++g)
          *reinterpret_cast<uint4*>(dst + (((cc0 + g) ^ sw) << 4)) = make_uint4(o[4 * g], o[4 * g + 1], o[4 * g + 2], o[4 * g + 3]);
      };
      // ---- k, pass 1 (slot 1, phase lt): sum of squares only -- no smem write, so it runs ahead of the window release
      MBW(bar(B_ACCFULL + 1), lt & 1);
      tc_fence_after();
      TR(1, lt, 1);
      acc_pass<CW, CH>(tmem + C + lane_addr, [&](int c0, float (&v)[CH]) { (void)c0; sumsq<CH>(v, sk0, sk1); }, [] {});
      TR(2, lt, 1);
      if (lt >= NSET) MBW(bar(B_WINFREE + set * 4 + q), ((lt / NSET) - 1) & 1);
      TR(3, lt, 1);
      // ---- q (slot 0, phase 2 lt), single pass: sum of squares and the raw bf16 operand
      MBW(bar(B_ACCFULL + 0), 0);
      tc_fence_after();
      TR(1, lt, 0);
      acc_pass<CW, CH>(tmem + lane_addr, [&](int c0, float (&v)[CH]) {
        sumsq<CH>(v, sq0, sq1);
        uint32_t o[CH / 2];
#pragma unroll
        for (int e = 0; e < CH / 2; ++e) o[e] = pack_bf16x2_rn(v[2 * e], v[2 * e + 1]);
        store(set_base + row_off, cb + c0, o, 8 * 2048);
      }, [&] { release(0); });
      // the other half's partial sums (double-buffered by tile parity: a slot is rewritten two barriers later)
      float2* exs = ex + (lt & 1) * 256;
      exs[h * 128 + r] = make_float2((sq0.x + sq0.y) + (sq1.x + sq1.y), (sk0.x + sk0.y) + (sk1.x + sk1.y));
      asm volatile("bar.sync %0, 64;" ::"r"(3 + q) : "memory");
      const float2 mine = exs[h * 128 + r], other = exs[(h ^ 1) * 128 + r];
      // F.normalize: x / max(|x|, 1e-12) on each of q and k; log2(e) so the softmax exponential is a bare ex2.  (lower half +
      // upper half in both threads: the same value bit for bit)
      const float ssq = h ? other.x + mine.x : mine.x + other.x, ssk = h ? other.y + mine.y : mine.y + other.y;
      const float rn = rsqrtf(fmaxf(ssq, 1e-24f)) * rsqrtf(fmaxf(ssk, 1e-24f)) * 1.4426950408889634f;
      const float2 rn2 = make_float2(rn, rn);
      // ---- k, pass 2: k / (|q_p| |k_p|) * log2 e
      acc_pass<CW, CH>(tmem + C + lane_addr, [&](int c0, float (&v)[CH]) {
        uint32_t o[CH / 2];
#pragma unroll
        for (int e = 0; e < CH / 2; ++e) {
          const float2 t = __fmul2_rn(make_float2(v[2 * e], v[2 * e + 1]), rn2);
          o[e] = pack_bf16x2_rn(t.x, t.y);
        }
        store(set_base + K::QK_BYTES + row_off, cb + c0, o, 8 * 2048);
      }, [&] { release(1); });
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(B_QKREADY + set * 4 + q));
      TR(4, lt, 1);
      // ---- v (slot 0, phase 2 lt + 1): -> fp16
      MBW(bar(B_ACCFULL + 0), 1);
      tc_fence_after();
      TR(1, lt, 2);
      acc_pass<CW, CH>(tmem + lane_addr, [&](int c0, float (&v)[CH]) {
        uint32_t o[CH / 2];
#pragma unroll
        for (int e = 0; e < CH / 2; ++e) o[e] = pack_f16x2_rn(v[2 * e], v[2 * e + 1]);
        store(set_base + 2 * K::QK_BYTES + vrow_off, cb + c0, o, K::V_KB);
      }, [&] { release(0); });
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(B_VREADY + set));
      TR(4, lt, 2);
    }
  } else if (warp >= SM0 && warp < EP0) {
    // =========================================== softmax + O drain: one group of warps per S buffer ======================
    // group b owns buffer b (units b, b + NBUF, ...): S -> P = exp2(S) (fp16, over consumed S columns) -> [issuer PV: P.V] ->
    // (O + P.b_v) / rowsum -> bf16 -> the projection's MN-major A tile.  The NBUF lifecycles run staggered, so the tensor pipe
    // always has a unit to work on.  C=128: two warps per 32 rows, each with 64 of the 128 S columns and 8 of the 16 pixels of O.
    const int q = warp & 3;
    const int grp = (warp - SM0) / (4 * K::SMH);
    const int half = K::SMH == 2 ? ((warp - SM0) >> 2) & 1 : 0;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const int total = T * UNITS;
    const uint32_t sbuf = tmem + K::SCOL0 + grp * 128 + lane_addr;
    // C=64: lanes 64-127 hold the pair's second window in columns 64-127, P of every lane in [0, 32).  C=128: half h reads S
    // columns [64 h, 64 h + 64) and writes P to [64 h, 64 h + 32)
    const uint32_t scol = sbuf + (C == 64 ? 64 * (q >> 1) : 64 * half);
    const uint32_t pcol = sbuf + (C == 64 ? 0 : 64 * half);
    const uint32_t ocol = sbuf + K::OOFF + (C == 64 ? 24 * (q >> 1) : 0);
    const int i_ch = C == 64 ? 32 * (q & 1) + lane : q * 32 + lane;   // channel of this thread's row
    TR_DECL_IF(7 + grp * 4 + q, half == 0);
    uint32_t ph = 0;
    for (int g = grp; g < total; g += NBUF, ph ^= 1u) {
      const int lt = g / UNITS, u = g - lt * UNITS;
      MBW(bar(B_SFULL + grp), ph);
      tc_fence_after();
      TR(1, lt, u);
      {
        // 16-column chunks, the load of chunk i + 1 in flight while chunk i is exponentiated
        constexpr int NCK = 64 / 16;
        float va[16], vb[16];
        tmem_ld16(scol, va);
#pragma unroll
        for (int i = 0; i < NCK; ++i) {
          float(&cur)[16] = (i & 1) ? vb : va;
          float(&nxt)[16] = (i & 1) ? va : vb;
          tmem_ld_wait();
          reg_fence(cur);
          if (i + 1 < NCK) tmem_ld16(scol + 16 * (i + 1), nxt);
          uint32_t pk[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint32_t x = pack_f16x2_rn(cur[2 * j], cur[2 * j + 1]);
            pk[j] = (MSG_LA_MUFU_EVERY > 0 && j % (MSG_LA_MUFU_EVERY > 0 ? MSG_LA_MUFU_EVERY : 1) == 0) ? la::ex2_f16x2(x) : la::exp2_poly_f16x2(x);
          }
          tmem_st8(pcol + 8 * i, pk);
        }
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(B_PREADY + grp));
      TR(2, lt, u);
      // ---- O of the same unit: this thread's pixels (all 16 at C=64, 8 at C=128) + [row sum, P.b_hi, P.b_lo, -]
      MBW(bar(B_OFULL + grp), ph);
      tc_fence_after();
      TR(3, lt, u);
      constexpr int NPX = 16 / K::SMH;
      float v[NPX], x4[4];
      if constexpr (NPX == 16) tmem_ld16(ocol, v); else tmem_ld8(ocol + 8 * half, v);
      tmem_ld4(ocol + 16, x4);
      tmem_ld_wait();
      reg_fence(v);
      reg_fence(x4);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(B_OEMPTY + grp));
      // first unit of this group in tile lt: the projection of tile lt - 1 must have finished reading the A tile
      if (g - NBUF < lt * UNITS && lt >= 1) MBW(bar(B_PFULL), (lt - 1) & 1);
      const float inv = __fdividef(1.f, x4[0]);               // row sum of P (in [C/e^1.5, C e^1.5]) from the ones row
      const float bsum = x4[1] + x4[2];
      const int win = C == 64 ? 2 * u + (q >> 1) : u;         // window of this thread's row
      uint8_t* dst = gen + K::OFF_A + (win >> 2) * (C * 128) + i_ch * 128;
#pragma unroll
      for (int e = 0; e < NPX / 8; ++e) {
        uint32_t o[4];
#pragma unroll
        for (int k2 = 0; k2 < 4; ++k2) o[k2] = pack_bf16x2_rn((v[e * 8 + 2 * k2] + bsum) * inv, (v[e * 8 + 2 * k2 + 1] + bsum) * inv);
        const int ee = K::SMH == 2 ? half : e;
        *reinterpret_cast<uint4*>(dst + (((2 * (win & 3) + ee) ^ (i_ch & 7)) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
      }
      if (g + NBUF >= (lt + 1) * UNITS) {       // last unit of this group in the tile
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(B_ASREADY));
      }
      TR(4, lt, u);
    }
  } else if (warp >= EP0) {
    // ============ fused input InstanceNorm + activation of tile lt (as conv_tma.cu), then the projection epilogue of tile lt - 1 =======
    // (one group of four warps for both: each is a short burst per tile, and the order x(lt) -> qkv GEMMs(lt) -> proj(lt - 1) ->
    // epilogue(lt - 1) is the order the issuer works in anyway)
    // epilogue staging at C=128 = the x stage, whose tile (lt + 1) the qkv GEMMs have consumed: PFULL(lt) is committed by issuer G
    // after those GEMMs, so its completion implies they are done; the producer reloads the stage only after STFREE
    const int q = warp & 3;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const int r = q * 32 + lane;
    const int xt = tid - 32 * EP0;         // 0..127
    const int pchunk = xt & 7, rbase = xt >> 3;
    const int lchunk = pchunk ^ (rbase & 7);
    const double inv_hw = 1.0 / ((double)p.H * (double)p.W);
    const bool relu = p.in_act == MSG_ACT_RELU;
    const __nv_bfloat162 zero2 = __floats2bfloat162_rn(0.f, 0.f);
    int cur_img = -1;
    TR_DECL(19 + q);
    auto epilogue = [&](int lt) {
      MBW(bar(B_PFULL), lt & 1);
      tc_fence_after();
      TR(3, lt, 0);
      acc_pass<C, CH>(tmem + C + lane_addr, [&](int c0, float (&v)[CH]) {
        uint8_t* dst = gen + K::OFF_STG + (c0 >> 6) * K::X_TILE + r * 128;
        const int cc0 = (c0 & 63) >> 3;
#pragma unroll
        for (int g = 0; g < CH / 8; ++g) {
          uint32_t o[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) o[e] = pack_bf16x2_rn(v[g * 8 + 2 * e], v[g * 8 + 2 * e + 1]);
          *reinterpret_cast<uint4*>(dst + (((cc0 + g) ^ (r & 7)) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
        }
      }, [&] {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(B_PEMPTY));
      });
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        int img, h0, wc0;
        tile_coords(t_begin + lt, img, h0, wc0);
        for (int kb = 0; kb < KB; ++kb)
          tma_store_5d(&mapOut, base + K::OFF_STG + kb * K::X_TILE + q * 4096, kb * 64, 0, h0, wc0 + 2 * q, img);
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        mbar_arrive(bar(B_STFREE));
      }
      __syncwarp();
      TR(4, lt, 0);
    };
    auto xform = [&](int lt) {
      const int img = (t_begin + lt) / p.tiles_per_img;
      if (img != cur_img) {
        asm volatile("bar.sync 2, 128;" ::: "memory");
        for (int ci = xt; ci < C; ci += 128) {
          float g = 1.f, b = 0.f, mean, rstd;
          if constexpr (AFF) in_affine(p.in_gamma, p.in_beta, (size_t)img * p.in_img_stride + ci, g, b);
          in_scale_shift(p.in_stats + ((size_t)img * C + ci) * 2, inv_hw, g, b, mean, rstd, xf_tab[ci], xf_tab[C + ci]);
        }
        asm volatile("bar.sync 2, 128;" ::: "memory");
        cur_img = img;
      }
      const int xs = lt % XS;
      MBW(bar(B_XFULL + xs), (lt / XS) & 1);
#pragma unroll 1
      for (int kb = 0; kb < KB; ++kb) {
        float sc[8], sh[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) { sc[e] = xf_tab[kb * 64 + lchunk * 8 + e]; sh[e] = xf_tab[C + kb * 64 + lchunk * 8 + e]; }
        uint8_t* tile = gen + K::OFF_X + xs * K::X_BYTES + kb * K::X_TILE + rbase * 128 + pchunk * 16;
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
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(B_XFDONE + xs));
    };
    // The transform runs one tile ahead of the GEMMs.  With two x stages (C=64) tile lt + 1 is transformed BEFORE the epilogue of
    // tile lt - 1 (whose projection is only issued after the qkv GEMMs of tile lt: waiting for it first would serialise
    // GEMMs(lt) -> proj(lt - 1) -> epilogue(lt - 1) -> transform(lt + 1) -> GEMMs(lt + 1)); with one stage (C=128) the load of
    // tile lt + 1 needs the staging of epilogue(lt - 1) back, so the epilogue comes first.
    if (XF && T > 0) xform(0);
    for (int lt = 0; lt < T; ++lt) {
      if (XS == 2) {
        if (XF && lt + 1 < T) xform(lt + 1);
        if (lt >= 1) epilogue(lt - 1);
      } else {
        if (lt >= 1) epilogue(lt - 1);
        if (XF && lt + 1 < T) xform(lt + 1);
      }
    }
    if (T > 0) epilogue(T - 1);
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
  }
}

unsigned long long* g_trace = nullptr;

template <int C, bool XF, bool AFF = false>
int launch(const CUtensorMap& mX, const CUtensorMap& mQ, const CUtensorMap& mP, const CUtensorMap& mO, const LaParams& p, cudaStream_t st) {
  static DeviceOnce attr_set;
  if (attr_set.needed()) {
    cudaError_t e = cudaFuncSetAttribute(la_stage_kernel<C, XF, AFF>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<C>::SMEM);
    MSG_REQUIRE(e == cudaSuccess, MSG_ERR_CUDA, "la_stage: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    attr_set.done();
  }
  int grid = sm_count();
  if (grid > p.total_tiles) grid = p.total_tiles;
  la_stage_kernel<C, XF, AFF><<<grid, 32 * Cfg<C>::NWARPS, Cfg<C>::SMEM, st>>>(mX, mQ, mP, mO, p);
  return check_launch("la_stage_kernel");
}

}  // namespace

bool la_stage_supported(int dtype, int N, int H, int W, int C, const void* x, const void* wqkv, const void* wproj, const void* out) {
  if (dtype != MSG_BF16) return false;
  if (C != 64 && C != 128) return false;
  if (N <= 0 || H <= 0 || W <= 0 || (H & 3) || (W & 3)) return false;
  if (((uintptr_t)x | (uintptr_t)wqkv | (uintptr_t)wproj | (uintptr_t)out) & 15) return false;
  const long long tiles = (long long)N * (H / 4) * ((W + 31) / 32);
  if (tiles > 0x3fffffffLL) return false;
  return get_encode() != nullptr;
}

int la_stage_fwd(const void* x, const double* in_stats, const float* in_gamma, const float* in_beta, int in_img_stride, int in_act,
                 const void* wqkv, const float* bqkv, const void* wproj, const float* bproj, int N, int H, int W, int C, void* out,
                 cudaStream_t st) {
  EncodeTiledFn enc = get_encode();
  MSG_REQUIRE(enc != nullptr, MSG_ERR_CUDA, "la_stage: cuTensorMapEncodeTiled unavailable");
  LaParams p;
  p.N = N; p.H = H; p.W = W;
  p.tiles_w = (W + 31) / 32;
  p.tiles_per_img = (H / 4) * p.tiles_w;
  p.total_tiles = N * p.tiles_per_img;
  p.bqkv = bqkv; p.bproj = bproj; p.in_stats = in_stats; p.in_act = in_act;
  p.in_gamma = in_gamma; p.in_beta = in_beta; p.in_img_stride = in_img_stride;
  p.trace = g_trace;
  CUtensorMap mX, mO, mQ, mP;
  for (int which = 0; which < 2; ++which) {
    // (channel, x in window, y, window column, image): a box lands as [window][y in window][x in window][64 ch]
    cuuint64_t dims[5] = {(cuuint64_t)C, 4, (cuuint64_t)H, (cuuint64_t)(W / 4), (cuuint64_t)N};
    cuuint64_t strides[4] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)4 * C * 2, (cuuint64_t)H * W * C * 2};
    cuuint32_t box[5] = {64, 4, 4, which == 0 ? 8u : 2u, 1};
    cuuint32_t es[5] = {1, 1, 1, 1, 1};
    CUresult r = enc(which == 0 ? &mX : &mO, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, which == 0 ? (void*)x : out, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     which == 0 ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B : CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "la_stage: cuTensorMapEncodeTiled(%s) failed with %d", which == 0 ? "x" : "out", (int)r);
  }
  for (int which = 0; which < 2; ++which) {
    const int rows = which == 0 ? 3 * C : C;
    cuuint64_t dims[2] = {(cuuint64_t)C, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)C * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)(C == 64 ? rows : 128)};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(which == 0 ? &mQ : &mP, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, which == 0 ? (void*)wqkv : (void*)wproj, dims, strides, box,
                     es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "la_stage: cuTensorMapEncodeTiled(w) failed with %d", (int)r);
  }
  const bool xf = in_stats != nullptr;
  const bool aff = in_gamma != nullptr;
  if (C == 64) {
    if (!xf) return launch<64, false>(mX, mQ, mP, mO, p, st);
    return aff ? launch<64, true, true>(mX, mQ, mP, mO, p, st) : launch<64, true>(mX, mQ, mP, mO, p, st);
  }
  if (!xf) return launch<128, false>(mX, mQ, mP, mO, p, st);
  return aff ? launch<128, true, true>(mX, mQ, mP, mO, p, st) : launch<128, true>(mX, mQ, mP, mO, p, st);
}

}  // namespace msg

using namespace msg;

/* development hook (MSG_LA_TRACE builds): device buffer of 24 x 4096 u64 receiving CTA 0's role timelines; NULL = off */
extern "C" int msg_la_stage_set_trace(void* buf) {
  g_trace = reinterpret_cast<unsigned long long*>(buf);
  return MSG_OK;
}

extern "C" int msg_la_stage_supported(int dtype, int N, int H, int W, int C, const void* x, const void* wqkv, const void* wproj,
                                      const void* out) {
  return la_stage_supported(dtype, N, H, W, C, x, wqkv, wproj, out) ? 1 : 0;
}

extern "C" int msg_la_stage_fwd_affine(int dtype, const void* x, const double* in_stats, const float* in_gamma, const float* in_beta,
                                       int in_img_stride, int in_act, const void* wqkv, const float* bqkv, const void* wproj,
                                       const float* bproj, int N, int H, int W, int C, void* out, void* stream) {
  MSG_REQUIRE(x && wqkv && bqkv && wproj && bproj && out, MSG_ERR_SHAPE, "la_stage: null pointer");
  MSG_REQUIRE(la_stage_supported(dtype, N, H, W, C, x, wqkv, wproj, out), MSG_ERR_UNSUPPORTED,
              "la_stage: needs bf16, C in {64, 128}, H and W multiples of 4, 16-byte aligned pointers (got C=%d, %dx%d)", C, H, W);
  MSG_REQUIRE(in_stats == nullptr || in_act == MSG_ACT_NONE || in_act == MSG_ACT_RELU, MSG_ERR_UNSUPPORTED,
              "la_stage: fused input norm supports ReLU / no activation");
  MSG_REQUIRE((in_gamma == nullptr) == (in_beta == nullptr) && (in_gamma == nullptr || in_stats != nullptr) && in_img_stride >= 0,
              MSG_ERR_SHAPE, "la_stage: an input affine needs gamma, beta and in_stats");
  return la_stage_fwd(x, in_stats, in_gamma, in_beta, in_img_stride, in_act, wqkv, bqkv, wproj, bproj, N, H, W, C, out, as_stream(stream));
}

extern "C" int msg_la_stage_fwd(int dtype, const void* x, const double* in_stats, int in_act, const void* wqkv, const float* bqkv,
                                const void* wproj, const float* bproj, int N, int H, int W, int C, void* out, void* stream) {
  return msg_la_stage_fwd_affine(dtype, x, in_stats, nullptr, nullptr, 0, in_act, wqkv, bqkv, wproj, bproj, N, H, W, C, out, stream);
}
