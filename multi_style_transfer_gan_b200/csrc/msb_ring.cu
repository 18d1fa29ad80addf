// MultiScaleBlock branches (enhanced_generator.py:52-71: 1x1 | 3x3 dil 1 | 3x3 dil 2 | 3x3 dil 4, C -> 4 x C/4 channels) as a ROW
// RING of tensor-memory accumulators (sm_100a, bf16 operands, fp32 accumulate), C = 64 (one pass) and C = 128 (three passes).
// The mechanics shared with the other ring kernels are in ring.cuh.
//
// The per-tap row-slab kernel (conv_slab.cu) issues 25 MMAs of N = C/4 per K step and output row; a tcgen05.mma with M = 128
// costs ~45 cycles however small N is, so that kernel runs at 15-25 % of the tensor pipe, and it loads seven input row slabs per
// output row (plus, at C = 128, the streamed weights).  Here a CTA walks DOWN a 128-pixel column strip of one image:
//   * every input row slab [136 pixels x C ch] is loaded ONCE (TMA boxes, zero fill = the convs' padding); weights stay resident;
//   * for a horizontal shift sx the three vertical taps of a dilated 3x3 branch send input row r to output rows r - d, r, r + d,
//     whose accumulators sit in ADJACENT tensor-memory columns -- every branch keeps one ring of C/4-column row accumulators per
//     residue class (row mod d) -- so they are ONE MMA of N = 3C/4 over a weight stack [ky = 2 | ky = 1 | ky = 0];
//   * the row finished by input row r (branch 1: r, branch 2: r - 1, branch 3: r - 2, branch 4: r - 4) is drained by that
//     branch's epilogue group (bias, IN statistics, bf16, per-warp TMA store of its channel slice of its own output row).
// C = 128 (32 columns per row accumulator) does not fit 512 tensor-memory columns in one go: branches 1 + 2, branch 3 and
// branch 4 run as three launches (passes), each with its own resident weight stacks.
// The schedule is stated (and run on tensors) in slab.py: RING_PASSES / ring_col / ring_row_mmas; this file restates it.
//
//   warp 0      TMA producer: the pass's weight stacks once, then one slab per input row
//   warps 1-3   MMA issuers (warp 1 also allocates TMEM), at most two rows ahead of the epilogue.  An issuing thread pays ~13
//               cycles per instruction (profiles/r1_mma_rate_microbench.md) and this schedule needs ~6 per MMA (ring slots and
//               runs change every row), so ONE issuer ran the MMAs at ~85 cycles each; the branches of a pass are spread over up
//               to three issuers (disjoint column ranges: the streams need no ordering)
//   warps 4-    epilogue: one group of four warps per branch of the pass (thread = strip pixel = TMEM lane)
#include "ring.cuh"

#include <type_traits>

namespace msg {
namespace {
using namespace ring;

// ---- pass tables (slab.py: RING_PASSES): branch ids and ring lengths of pass PS at width C
__host__ __device__ constexpr int ring_nb(int C, int ps) { return C == 64 ? 4 : (ps == 0 ? 2 : 1); }
__host__ __device__ constexpr int ring_branch(int C, int ps, int i) { return C == 64 ? i : (ps == 0 ? i : ps + 1); }
// ring length R per residue class (slab.py: RING_PASSES).  The issuers may run LEAD steps ahead of the epilogue: the slot of the row
// a 3x3 branch of dilation d finishes at step k is touched again at step k + (R - 2) d (the 1x1 branch: k + R), so
// LEAD <= min over the pass of that distance.
__host__ __device__ constexpr int ring_slots(int C, int ps, int i) {
  const int b = ring_branch(C, ps, i);
  if (C == 64) return b == 0 ? 3 : (b == 1 ? 5 : 4);            // 48 + 80 + 128 + 256 = 512 columns, LEAD 3
  return b == 0 ? 4 : (b == 1 ? 6 : (b == 2 ? 8 : 4));          // pass 0: 128 + 2 x 192 (two sets) | pass 1: 512 | pass 2: 512
}
__host__ __device__ constexpr int ring_lead(int C, int ps) { return C == 64 ? 3 : (ps == 0 ? 4 : 8); }
__host__ __device__ constexpr int ring_dil(int b) { return b == 0 ? 1 : (1 << (b - 1)); }
// a branch whose accumulators are DUPLICATED by input-row parity (C = 128 pass 0, the dilation-1 3x3): even and odd input rows
// accumulate into two separate rings, so two issuers share the branch without touching the same columns; the epilogue adds them
__host__ __device__ constexpr int ring_dup(int C, int ps, int i) { return (C == 128 && ps == 0 && ring_branch(C, ps, i) == 1) ? 2 : 1; }
__host__ __device__ constexpr int ring_width(int C, int ps, int i) { return ring_dil(ring_branch(C, ps, i)) * ring_slots(C, ps, i) * (C / 4); }
__host__ __device__ constexpr int ring_base(int C, int ps, int i) {
  int col = 0;
  for (int j = 0; j < i; ++j) col += ring_width(C, ps, j) * ring_dup(C, ps, j);
  return col;
}
__host__ __device__ constexpr int ring_wrow0(int C, int ps, int i) {          // first weight row of branch i inside a 64-channel block
  int row = 0;
  for (int j = 0; j < i; ++j) row += (ring_branch(C, ps, j) == 0 ? 1 : 9) * (C / 4);
  return row;
}
__host__ __device__ constexpr int ring_halo(int C, int ps) { return ring_dil(ring_branch(C, ps, ring_nb(C, ps) - 1)); }   // rows above / below a piece
__host__ __device__ constexpr int ring_rows(int C, int ps) { return ring_wrow0(C, ps, ring_nb(C, ps)); }
// (first) issuer of branch i of the pass, and over how many issuers the branch is split BY INPUT ROW PARITY (one issuer alone is
// instruction-bound at 60-85 cycles per MMA, see the header).  A branch of dilation d >= 2 sends input row r only to output rows of
// its own residue class (r mod d), so the issuers of even and of odd rows write disjoint accumulators; the dilation-1 branch at
// C = 128 gets a second set of accumulators instead (ring_dup).
__host__ __device__ constexpr int ring_issuer(int C, int ps, int i) { return C == 64 ? (i <= 1 ? 0 : i - 1) : (ps == 0 ? i : 0); }
__host__ __device__ constexpr int ring_split(int C, int ps, int i) { return (C == 128 && (ps >= 1 || i == 1)) ? 2 : 1; }
__host__ __device__ constexpr int ring_nissue(int C, int ps) { return C == 64 ? 3 : (ps == 0 ? 3 : 2); }

// shared memory of pass PS: weight stacks [KB][rows][128 B], slabs of KB 64-channel blocks, bias [C], and per epilogue warp
// [16 ch][32 px] fp32 for the statistics and the staging of its piece, 32 pixels x C/4 channels (bf16).  C = 128: one 2 KB buffer
// serves both in turn (it buys a slab stage); C = 64: statistics + two 1 KB staging buffers
template <int C, int PS>
__host__ __device__ constexpr Shape ring_shape() {
  return Shape{C / 64 * ring_rows(C, PS) * 128, C / 64 * SLAB_BYTES, C, 4 * ring_nb(C, PS) * (C == 64 ? 4096 : 2048), 2};
}

struct RingParams {
  int N, H, W, Co_total, co_off;
  int segs;
  long long total_rows;           // N * segs * H
  int stages;
  int w_row0;                     // first row of this pass's stacks in the weight array
  const float* bias;
  double* stats;
};

template <int C, int PS, int I>
__device__ __forceinline__ uint32_t ring_col(int y) {       // TMEM column of the accumulator of output row y (>= 0) of branch I of the pass
  constexpr int d = ring_dil(ring_branch(C, PS, I)), R = ring_slots(C, PS, I), base = ring_base(C, PS, I), Q = C / 4;
  return (uint32_t)(base + ((y % d) * R + (y / d) % R) * Q);   // (second set of a duplicated branch: + ring_width)
}

template <int C, int PS>
__global__ void __launch_bounds__(32 * (EPI0 + 4 * ring_nb(C, PS)), 1)
msb_ring_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                const __grid_constant__ CUtensorMap mapY, const RingParams p) {
  constexpr int Q = C / 4, KB = C / 64, NB = ring_nb(C, PS), NISSUE = ring_nissue(C, PS);
  constexpr int ROWS = ring_rows(C, PS);                  // weight rows per 64-channel block
  constexpr Shape SH = ring_shape<C, PS>();
  constexpr int NEW = 4 * NB;                             // epilogue warps
  constexpr int NBUF = C == 64 ? 2 : 1;
  constexpr int OUT_B = C == 64 ? 4096 : 2048;
  constexpr int HV = ring_halo(C, PS);                    // input rows above / below a piece = the largest dilation of the pass
  constexpr uint32_t LEAD = (uint32_t)ring_lead(C, PS);
  using Walk = Pieces<1, HV>;
  extern __shared__ uint8_t smem_raw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const Smem sm(smem_raw, SH, p.stages);
  const Bars& bars = sm.b;
  float* sbias = sm.bias();

  if (tid < C) sbias[tid] = p.bias ? p.bias[tid] : 0.f;
  const uint32_t tmem_base = prologue(sm, warp, lane, NISSUE, NEW, 0, &mapA, &mapB, &mapY);
  const Walk pieces(p.total_rows, p.H, p.segs);

  if (warp == 0) {
    if (lane == 0)
      producer(sm, pieces, p.H, &mapB, SH.w_bytes, p.w_row0, SH.stage_bytes, [&](const Walk& pc, int r, uint32_t dst, uint32_t bar) {
#pragma unroll
        for (int kb = 0; kb < KB; ++kb) tma_load_4d(dst + kb * SLAB_BYTES, &mapA, bar, kb * 64, pc.seg * BM - HALO, r, pc.img);
      });
  } else if (warp < EPI0) {
    const int me = warp - 1;
    if (me < NISSUE) {
      const bool leader = elect_one();
      const uint32_t hi = (uint32_t)(make_sw128_desc(0) >> 32);
      const uint32_t b_base = sm.sB() >> 4;
      issuer<LEAD, false>(bars, pieces, p.H, leader, [&](const Walk& pc, int r, int s) {
        const uint32_t a0 = sm.sA(s, SH.stage_bytes) >> 4;
        // the branches of this issuer: compile-time loop, the others fold away
        auto branch = [&](auto IC) {
          constexpr int I = decltype(IC)::value;
          constexpr int b = ring_branch(C, PS, I);
          constexpr uint32_t wr0 = (uint32_t)ring_wrow0(C, PS, I);
          if constexpr (b == 0) {
            if (r >= pc.y0 && r < pc.y1) {     // the 1x1 conv, output row r
              const uint32_t dcol = tmem_base + ring_col<C, PS, I>(r);
#pragma unroll
              for (int kb = 0; kb < KB; ++kb)
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)
                  umma_bf16_lo(dcol, a0 + (uint32_t)(kb * (SLAB_BYTES >> 4) + HALO * 8 + 2 * ks),
                               b_base + (uint32_t)((kb * ROWS + (int)wr0) * 8 + 2 * ks), hi, idesc_bf16(Q), true);
            }
          } else {
            // entries e = 0, 1, 2 = output rows r - d, r, r + d (vertical taps ky = 2, 1, 0); those of this piece are an interval
            // of entries whose slots in the residue class's ring are adjacent except where the ring wraps
            constexpr int d = ring_dil(b);
            constexpr int R = ring_slots(C, PS, I);
            const uint32_t set = ring_dup(C, PS, I) > 1 ? (uint32_t)((r & 1) * ring_width(C, PS, I)) : 0u;
            const int e_lo = r - d >= pc.y0 ? 0 : (r >= pc.y0 ? 1 : 2);          // r + d >= y0 holds for every row of the piece's halo
            const int e_hi = r + d < pc.y1 ? 2 : (r < pc.y1 ? 1 : 0);            // r - d < y1 likewise
            if (e_lo <= e_hi && r + d >= pc.y0 && r - d < pc.y1) {
              const int ylo = r + (e_lo - 1) * d;                                // first output row (>= y0 >= 0)
              const int cls = ylo % d;
              runs(e_hi - e_lo + 1, (ylo / d) % R, R, [&](int e, int nrun, int idx) {
                const uint32_t idesc = idesc_bf16(Q * nrun);
                const uint32_t dcol = tmem_base + (uint32_t)(ring_base(C, PS, I) + (cls * R + idx) * Q) + set;
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
                  const uint32_t wrow = wr0 + (uint32_t)(kx * 3 * Q + Q * (e_lo + e));
                  const uint32_t av = a0 + (uint32_t)((HALO + (kx - 1) * d) * 8);
#pragma unroll
                  for (int kb = 0; kb < KB; ++kb)
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)
                      umma_bf16_lo(dcol, av + (uint32_t)(kb * (SLAB_BYTES >> 4) + 2 * ks),
                                   b_base + (uint32_t)(kb * ROWS * 8) + wrow * 8u + (uint32_t)(2 * ks), hi, idesc, true);
                }
              });
            }
          }
        };
        auto mine = [&](int i) { return ring_issuer(C, PS, i) + (r & (ring_split(C, PS, i) - 1)) == me; };
        if (mine(0)) branch(std::integral_constant<int, 0>{});
        if constexpr (NB > 1) { if (mine(1)) branch(std::integral_constant<int, 1>{}); }
        if constexpr (NB > 2) { if (mine(2)) branch(std::integral_constant<int, 2>{}); }
        if constexpr (NB > 3) { if (mine(3)) branch(std::integral_constant<int, 3>{}); }
      });
    }
  } else {
    // ===================================== epilogue: four warps per branch =====================================
    const int q = warp & 3;
    const int ew = warp - EPI0;                       // epilogue warp index
    const int bi = ew >> 2;                           // branch index inside the pass
    const int b = ring_branch(C, PS, bi);
    const int lag = b == 0 ? 0 : (1 << (b - 1));      // input row r completes output row r - lag of branch b
    const int row = q * 32 + lane;                    // strip pixel = TMEM lane
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    uint8_t* buf = sm.scratch(ew, OUT_B);
    Stats stats;                                      // lane l < Q: channel l of the branch
    const bool do_stats = p.stats != nullptr;
    uint32_t col_dup = 0;                             // column distance to the second accumulator set of a duplicated branch
    auto col_of = [&](int y) -> uint32_t {            // (bi is warp-uniform; the table folds per case)
      switch (bi) {
        case 0: return ring_col<C, PS, 0>(y);
        case 1: if constexpr (NB > 1) return ring_col<C, PS, 1>(y);
        case 2: if constexpr (NB > 2) return ring_col<C, PS, 2>(y);
        default: if constexpr (NB > 3) return ring_col<C, PS, 3>(y);
      }
      return 0u;
    };
    if constexpr (NB > 1) { if (bi == 1 && ring_dup(C, PS, 1) > 1) col_dup = (uint32_t)ring_width(C, PS, 1); }
    if (bi == 0 && ring_dup(C, PS, 0) > 1) col_dup = (uint32_t)ring_width(C, PS, 0);
    uint32_t k = 0;                        // steps
    uint32_t nst = 0;                      // pieces stored by this warp
    for (Walk pc = pieces; pc.next();) {
      const bool valid = pc.seg * BM + row < p.W;
      if (do_stats && pc.img != stats.img) { stats.flush<Q>(p.stats, p.Co_total, p.co_off + Q * b, lane); stats.img = pc.img; }
      for (int r = pc.r0; r < pc.r1; ++r, ++k) {
        const int y = r - lag;                                       // the row this input row completed for this branch
        // every warp follows every step (also those that finish nothing for it): a warp that ran ahead would arrive on a
        // drained barrier whose previous phase is still open
        bars.wait_rowdone(k);
        if (y >= pc.y0 && y < pc.y1) {                               // (warp-uniform)
          tc_fence_after();
          const uint32_t taddr = tmem_base + lane_addr + col_of(y);
          float v[Q];
          tmem_ld_n(taddr, v);
          if (col_dup) {                                             // (warp-uniform) even-row set + odd-row set
            float v2[Q];
            tmem_ld_n(taddr + col_dup, v2);
            tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < Q; ++c) v[c] += v2[c];
            tmem_zero<Q>(taddr + col_dup);
          } else {
            tmem_ld_wait();
          }
          tmem_zero<Q>(taddr);
          tmem_st_wait();
          tc_fence_before();
          arrive_drained(bars, k, lane);
#pragma unroll
          for (int c = 0; c < Q; ++c) v[c] += sbias[Q * b + c];
          uint8_t* stg = NBUF == 2 ? buf + 2048 + (nst & 1) * 1024 : buf;
          if (nst >= (uint32_t)NBUF) wait_store_read<NBUF - 1>(lane);   // the store issued NBUF pieces ago has read its buffer
          if (do_stats) piece_stats<Q>(reinterpret_cast<float*>(buf), v, valid, lane, stats);
          store_piece_bf16<Q>(stg, v, lane, &mapY, p.co_off + Q * b, pc.seg * BM + q * 32, y, pc.img);
          ++nst;
        } else {
          if (lane == 0) mbar_arrive(bars.drained(k));           // nothing for this group at this step
        }
      }
    }
    if (do_stats) stats.flush<Q>(p.stats, p.Co_total, p.co_off + Q * b, lane);
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  teardown(warp, tmem_base);
}

template <int C, int PS>
int launch_pass(const CUtensorMap& mapA, const CUtensorMap& mapB, const CUtensorMap& mapY, RingParams p, int w_row0, cudaStream_t st) {
  static_assert(ring_shape<C, PS>().stages() >= 2, "msb_ring: the slab ring of this pass does not fit shared memory");
  p.w_row0 = w_row0;
  // at least 8 rows per CTA (each piece re-reads 8 halo rows)
  return launch<msb_ring_kernel<C, PS>>("msb_ring_kernel", ring_shape<C, PS>(), 32 * (EPI0 + 4 * ring_nb(C, PS)), p.total_rows, 8, p,
                                        mapA, mapB, mapY, st);
}

int msb_ring_impl(const msg_msb_ring_desc* d, int C, const void* x, const void* w_stacks, const float* bias, void* y, double* stats,
                  cudaStream_t st) {
  MSG_REQUIRE(d != nullptr && x && w_stacks && y, MSG_ERR_SHAPE, "msb_ring: null argument");
  MSG_REQUIRE(C == 64 || C == 128, MSG_ERR_UNSUPPORTED, "msb_ring: C must be 64 or 128 (got %d)", C);
  MSG_REQUIRE(d->dtype == MSG_BF16, MSG_ERR_UNSUPPORTED, "msb_ring: bf16 only");
  MSG_REQUIRE(d->N > 0 && d->H > 0 && d->W > 0, MSG_ERR_SHAPE, "msb_ring: bad plane");
  MSG_REQUIRE((d->Ci_total & 7) == 0 && (d->ci_off & 7) == 0 && d->ci_off + C <= d->Ci_total, MSG_ERR_SHAPE, "msb_ring: input channel layout");
  MSG_REQUIRE((d->Co_total & 7) == 0 && (d->co_off & 7) == 0 && d->co_off + C <= d->Co_total, MSG_ERR_SHAPE, "msb_ring: output channel layout");
  MSG_REQUIRE((((uintptr_t)x | (uintptr_t)w_stacks | (uintptr_t)y) & 15) == 0, MSG_ERR_ALIGN, "msb_ring: operands must be 16-byte aligned");
  MSG_REQUIRE(!(d->flags & MSG_CONV_STATS) || stats != nullptr, MSG_ERR_SHAPE, "msb_ring: stats buffer missing");
  MSG_REQUIRE(get_encode() != nullptr, MSG_ERR_CUDA, "msb_ring: cuTensorMapEncodeTiled unavailable");

  RingParams p;
  p.N = d->N; p.H = d->H; p.W = d->W; p.Co_total = d->Co_total; p.co_off = d->co_off;
  p.bias = bias; p.stats = (d->flags & MSG_CONV_STATS) ? stats : nullptr;
  p.segs = (d->W + BM - 1) / BM;
  p.total_rows = (long long)d->N * p.segs * d->H;
  MSG_REQUIRE(p.total_rows < (1LL << 40), MSG_ERR_SHAPE, "msb_ring: too many rows");
  const int KB = C / 64;
  int total_w_rows = 0;
  for (int ps = 0; ps < (C == 64 ? 1 : 3); ++ps) total_w_rows += KB * ring_rows(C, ps);

  CUtensorMap mapA, mapB, mapY;
  CUresult r = encode_store(&mapY, y, d->Co_total, d->W, d->H, d->N, C / 4, 1);
  MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "msb_ring: cuTensorMapEncodeTiled(y) failed with %d", (int)r);
  r = encode_slab(&mapA, (const __nv_bfloat16*)x + d->ci_off, C, d->Ci_total, d->W, d->H, d->N);
  MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "msb_ring: cuTensorMapEncodeTiled(x) failed with %d", (int)r);
  r = encode_weights(&mapB, w_stacks, total_w_rows);
  MSG_REQUIRE(r == CUDA_SUCCESS, MSG_ERR_CUDA, "msb_ring: cuTensorMapEncodeTiled(w) failed with %d", (int)r);
  if (C == 64) return launch_pass<64, 0>(mapA, mapB, mapY, p, 0, st);
  int row0 = 0;
  int rc = launch_pass<128, 0>(mapA, mapB, mapY, p, row0, st);
  if (rc) return rc;
  row0 += KB * ring_rows(128, 0);
  rc = launch_pass<128, 1>(mapA, mapB, mapY, p, row0, st);
  if (rc) return rc;
  row0 += KB * ring_rows(128, 1);
  return launch_pass<128, 2>(mapA, mapB, mapY, p, row0, st);
}

}  // namespace
}  // namespace msg

using namespace msg;

extern "C" int msg_msb_ring(const msg_msb_ring_desc* d, int C, const void* x, const void* w_stacks, const float* bias, void* y,
                            double* stats, void* stream) {
  return msb_ring_impl(d, C, x, w_stacks, bias, y, stats, as_stream(stream));
}

extern "C" int msg_msb64_ring(const msg_msb_ring_desc* d, const void* x, const void* w_stacks, const float* bias, void* y,
                              double* stats, void* stream) {
  return msb_ring_impl(d, 64, x, w_stacks, bias, y, stats, as_stream(stream));
}
