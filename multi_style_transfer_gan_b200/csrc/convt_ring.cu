// ConvTranspose2d(k = 4, stride 2, pad 1) of the decoder (enhanced_generator.py:116-123, up2: 128 -> 64 channels) as a ROW RING of
// tensor-memory accumulators (sm_100a, bf16 operands, fp32 accumulate) -- the transposed-conv sibling of msb_ring.cu; the shared
// mechanics are in ring.cuh.
//
// out[o, u] = sum in[i, j] w[ky, kx] with o = 2 i - 1 + ky, u = 2 j - 1 + kx.  The four sub-pixel phase launches of the row-slab
// path (conv_slab.cu) each re-read two input rows per output row and issue one N = 64 MMA per tap; here a CTA walks DOWN a
// 128-pixel column strip of the INPUT, one launch per horizontal phase px = u mod 2:
//   * every input row slab [136 pixels x Cin] is loaded ONCE per launch (TMA, zero fill = the implicit padding); the launch's weights
//     (2 horizontal taps x 4 vertical taps x Cin x 64 output channels = 128 KB at Cin = 128) stay resident in shared memory;
//   * input row r feeds the output rows 2r-1, 2r, 2r+1, 2r+2 (ky = 0..3), whose accumulators are ADJACENT 64-column slots of an
//     eight-slot ring (slot = output row mod 8): for each of the two horizontal taps of the phase (a shifted view of the slab) ALL
//     FOUR vertical taps are one tcgen05.mma of N = 256 over the weight stack [ky = 0 | 1 | 2 | 3] -- 2 to 4 MMAs per K step and
//     input row instead of 16 (the ring wraps once every four rows: two N = 128 MMAs there);
//   * input row r completes output rows 2r-1 and 2r: eight epilogue warps (lane quarter x channel half) drain both and hand their
//     [32 px x 32 ch] pieces to the TMA store through a tensor map whose pixel stride is 2 (the other phase's pixels lie in between).
// A slot is touched again three input rows after its row completed, so the issuer may run LEAD = 3 rows ahead of the epilogue.
// A piece [y0, y1) of input rows owns the output rows [2 y0, 2 y1) and reads the input rows y0 - 1 .. y1.
// The schedule is stated and run on tensors in slab.py (convt_ring_row_mmas) / tests/test_convt_ring_cpu.py.
//
//   warp 0      TMA producer: the phase's weight stacks once, then one slab per input row
//   warp 1      MMA issuer (also allocates TMEM)
//   warps 4-11  epilogue
#include "ring.cuh"

namespace msg {
namespace {
using namespace ring;

constexpr int NEW = 8;                  // epilogue warps
constexpr int NC = 64;                  // output channels per launch = columns per row accumulator
constexpr uint32_t LEAD = 3;
constexpr int W_ROWS = 2 * 4 * NC;      // weight rows per 64-channel block of the input: [2 horizontal taps][4 ky][64 co]
constexpr int OUT_B = 2048;             // per-warp scratch: [16 ch][32 px] fp32 for the statistics, then the [32 px][32 ch] bf16 piece

template <int KB>
__host__ __device__ constexpr Shape ct_shape() { return Shape{KB * W_ROWS * 128, KB * SLAB_BYTES, NC, NEW * OUT_B, 2}; }

struct CtParams {
  int N, H, W, Co_total, co_off;        // input plane H x W; output 2H x 2W
  int segs;
  long long total_rows;                 // N * segs * H input rows
  int stages;
  int px;                               // horizontal phase of this launch
  int w_row0;                           // first row of this launch's stacks in the weight array
  const float* bias;                    // [64] (of this launch's channels) or null
  double* stats;
};

template <int KB>
__global__ void __launch_bounds__(32 * (EPI0 + NEW), 1)
convt_ring_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                  const __grid_constant__ CUtensorMap mapY, const CtParams p) {
  constexpr Shape SH = ct_shape<KB>();
  using Walk = Pieces<1, 1>;
  extern __shared__ uint8_t smem_raw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const Smem sm(smem_raw, SH, p.stages);
  const Bars& bars = sm.b;
  float* sbias = sm.bias();

  if (tid < NC) sbias[tid] = p.bias ? p.bias[tid] : 0.f;
  const uint32_t tmem_base = prologue(sm, warp, lane, 1, NEW, 0, &mapA, &mapB, &mapY);
  const Walk pieces(p.total_rows, p.H, p.segs);

  if (warp == 0) {
    if (lane == 0)
      producer(sm, pieces, p.H, &mapB, SH.w_bytes, p.w_row0, SH.stage_bytes, [&](const Walk& pc, int r, uint32_t dst, uint32_t bar) {
#pragma unroll
        for (int kb = 0; kb < KB; ++kb) tma_load_4d(dst + kb * SLAB_BYTES, &mapA, bar, kb * 64, pc.seg * BM - HALO, r, pc.img);
      });
  } else if (warp == 1) {
    const bool leader = elect_one();
    const uint32_t hi = (uint32_t)(make_sw128_desc(0) >> 32);
    const uint32_t b_base = sm.sB() >> 4;
    const int dx1 = p.px == 0 ? -1 : 1;    // the phase's second horizontal tap reads the neighbour pixel on this side
    issuer<LEAD, false>(bars, pieces, p.H, leader, [&](const Walk& pc, int r, int s) {
      const uint32_t a0 = sm.sA(s, SH.stage_bytes) >> 4;
      // entries e = ky = 0..3 = output rows 2r-1 .. 2r+2; those of this piece are an interval of adjacent ring slots
      const int o_lo = 2 * r - 1 > 2 * pc.y0 ? 2 * r - 1 : 2 * pc.y0, o_hi = 2 * r + 2 < 2 * pc.y1 - 1 ? 2 * r + 2 : 2 * pc.y1 - 1;   // inclusive
      if (o_lo <= o_hi)
        runs(o_hi - o_lo + 1, o_lo & 7, 8, [&](int e, int nrun, int slot) {
          const uint32_t idesc = idesc_bf16(NC * nrun);
          const uint32_t dcol = tmem_base + (uint32_t)(slot * NC);
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            const uint32_t wrow = (uint32_t)(t * 4 * NC + NC * (o_lo - (2 * r - 1) + e));
            const uint32_t av = a0 + (uint32_t)((HALO + (t == 0 ? 0 : dx1)) * 8);
#pragma unroll
            for (int kb = 0; kb < KB; ++kb)
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)
                umma_bf16_lo(dcol, av + (uint32_t)(kb * (SLAB_BYTES >> 4) + 2 * ks),
                             b_base + (uint32_t)(kb * W_ROWS * 8) + wrow * 8u + (uint32_t)(2 * ks), hi, idesc, true);
          }
        });
    });
  } else if (warp >= EPI0) {
    // ===================================== epilogue: warp = (lane quarter q, channel half h) =====================================
    const int q = warp & 3;
    const int ew = warp - EPI0;
    const int h = ew >> 2;                            // channels [32 h, 32 h + 32) of the launch's 64
    const int row = q * 32 + lane;                    // strip pixel = TMEM lane
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    uint8_t* buf = sm.scratch(ew, OUT_B);
    Stats stats;                                      // lane l: channel 32 h + l
    const bool do_stats = p.stats != nullptr;
    uint32_t k = 0;
    bool stored = false;                   // a TMA store of this warp may still be reading buf
    for (Walk pc = pieces; pc.next();) {
      const bool valid = pc.seg * BM + row < p.W;
      if (do_stats && pc.img != stats.img) { stats.flush<32>(p.stats, p.Co_total, p.co_off + 32 * h, lane); stats.img = pc.img; }
      for (int r = pc.r0; r < pc.r1; ++r, ++k) {
        bars.wait_rowdone(k);
        // input row r completed the output rows 2r - 1 and 2r (those of this piece)
        const int oA = 2 * r - 1, oB = 2 * r;
        const bool okA = oA >= 2 * pc.y0 && oA < 2 * pc.y1, okB = oB >= 2 * pc.y0 && oB < 2 * pc.y1;        // (warp-uniform)
        float vA[32], vB[32];
        if (okA | okB) {
          tc_fence_after();
          const uint32_t tA = tmem_base + lane_addr + (uint32_t)((oA & 7) * NC + 32 * h);
          const uint32_t tB = tmem_base + lane_addr + (uint32_t)((oB & 7) * NC + 32 * h);
          if (okA) tmem_ld32(tA, vA);
          if (okB) tmem_ld32(tB, vB);
          tmem_ld_wait();
          if (okA) tmem_zero<32>(tA);
          if (okB) tmem_zero<32>(tB);
          tmem_st_wait();
          tc_fence_before();
        }
        arrive_drained(bars, k, lane);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          if (!(half == 0 ? okA : okB)) continue;
          float (&v)[32] = half == 0 ? vA : vB;
#pragma unroll
          for (int c = 0; c < 32; ++c) v[c] += sbias[32 * h + c];
          if (stored) wait_store_read<0>(lane);      // the previous piece's store has read buf
          if (do_stats) piece_stats<32>(reinterpret_cast<float*>(buf), v, valid, lane, stats);
          // this phase's pixels of the output row: the tensor map's pixel stride is 2
          store_piece_bf16<32>(buf, v, lane, &mapY, p.co_off + 32 * h, pc.seg * BM + q * 32, half == 0 ? oA : oB, pc.img);
          stored = true;
        }
      }
    }
    if (do_stats) stats.flush<32>(p.stats, p.Co_total, p.co_off + 32 * h, lane);
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  teardown(warp, tmem_base);
}

}  // namespace
}  // namespace msg

using namespace msg;

extern "C" int msg_convt_ring(const msg_convt_ring_desc* d, const void* x, const void* w_stacks, const float* bias, void* y,
                              double* stats, void* stream) {
  cudaStream_t st = as_stream(stream);
  MSG_REQUIRE(d != nullptr && x && w_stacks && y, MSG_ERR_SHAPE, "convt_ring: null argument");
  MSG_REQUIRE(d->dtype == MSG_BF16, MSG_ERR_UNSUPPORTED, "convt_ring: bf16 only");
  MSG_REQUIRE(d->Cin == 64 || d->Cin == 128, MSG_ERR_UNSUPPORTED, "convt_ring: Cin must be 64 or 128 (got %d): the phase's weights stay resident", d->Cin);
  MSG_REQUIRE(d->Cout > 0 && d->Cout % 64 == 0, MSG_ERR_UNSUPPORTED, "convt_ring: Cout must be a multiple of 64 (got %d)", d->Cout);
  MSG_REQUIRE(d->N > 0 && d->H > 0 && d->W > 0, MSG_ERR_SHAPE, "convt_ring: bad plane");
  MSG_REQUIRE((d->Ci_total & 7) == 0 && (d->ci_off & 7) == 0 && d->ci_off + d->Cin <= d->Ci_total, MSG_ERR_SHAPE, "convt_ring: input channel layout");
  MSG_REQUIRE((d->Co_total & 7) == 0 && (d->co_off & 7) == 0 && d->co_off + d->Cout <= d->Co_total, MSG_ERR_SHAPE, "convt_ring: output channel layout");
  MSG_REQUIRE((((uintptr_t)x | (uintptr_t)w_stacks | (uintptr_t)y) & 15) == 0, MSG_ERR_ALIGN, "convt_ring: operands must be 16-byte aligned");
  MSG_REQUIRE(!(d->flags & MSG_CONV_STATS) || stats != nullptr, MSG_ERR_SHAPE, "convt_ring: stats buffer missing");
  MSG_REQUIRE(get_encode() != nullptr, MSG_ERR_CUDA, "convt_ring: cuTensorMapEncodeTiled unavailable");
  const int KB = d->Cin / 64, G = d->Cout / 64;

  CtParams p;
  p.N = d->N; p.H = d->H; p.W = d->W; p.Co_total = d->Co_total;
  p.stats = (d->flags & MSG_CONV_STATS) ? stats : nullptr;
  p.segs = (d->W + BM - 1) / BM;
  p.total_rows = (long long)d->N * p.segs * d->H;
  MSG_REQUIRE(p.total_rows < (1LL << 40), MSG_ERR_SHAPE, "convt_ring: too many rows");

  CUtensorMap mapA, mapB;
  CUresult r = encode_slab(&mapA, (const __nv_bfloat16*)x + d->ci_off, d->Cin, d->Ci_total, d->W, d->H, d->N);
  MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "convt_ring: cuTensorMapEncodeTiled(x) failed with %d", (int)r);
  r = encode_weights(&mapB, w_stacks, (long long)G * 2 * KB * W_ROWS);
  MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "convt_ring: cuTensorMapEncodeTiled(w) failed with %d", (int)r);
  for (int g = 0; g < G; ++g)
    for (int px = 0; px < 2; ++px) {
      CUtensorMap mapY;
      // this phase's pixels of the output: pixel stride 2, starting at pixel px
      r = encode_store(&mapY, (__nv_bfloat16*)y + (size_t)px * d->Co_total, d->Co_total, d->W, 2 * d->H, d->N, 32, 2);
      MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "convt_ring: cuTensorMapEncodeTiled(y) failed with %d", (int)r);
      p.px = px;
      p.co_off = d->co_off + 64 * g;
      p.bias = bias ? bias + 64 * g : nullptr;
      p.w_row0 = (g * 2 + px) * KB * W_ROWS;
      // at least 4 input rows per CTA (each piece re-reads 2 halo rows)
      const int rc = KB == 1 ? launch<convt_ring_kernel<1>>("convt_ring_kernel", ct_shape<1>(), 32 * (EPI0 + NEW), p.total_rows, 4, p,
                                                            mapA, mapB, mapY, st)
                             : launch<convt_ring_kernel<2>>("convt_ring_kernel", ct_shape<2>(), 32 * (EPI0 + NEW), p.total_rows, 4, p,
                                                            mapA, mapB, mapY, st);
      if (rc) return rc;
    }
  return MSG_OK;
}
