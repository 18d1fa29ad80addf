// Mechanics shared by the row-ring kernels (msb_ring.cu, convt_ring.cu, out7_ring.cu, down_ring.cu; DESIGN §3.7).  Each kernel
// keeps its schedule (which output rows an input row feeds, slots, weight-stack offsets), its transform and its epilogue; this
// header holds what they all do the same way:
//   * shared memory: [weight stacks | slab stages | bias | per-warp scratch | mbarriers | TMEM slot] from a 1024-aligned base, one
//     layout function for the host's byte count and the kernel's carve-up;
//   * mbarriers: slab full / empty (/ transformed) per stage, the resident weights, and rings of NBAR `rowdone[k]`
//     (tcgen05.commit after the MMAs of step k) and `drained[k]` (epilogue arrivals);
//   * prologue: barrier init, 512-column TMEM alloc, every accumulator zeroed (each MMA of a ring kernel accumulates), and teardown;
//   * work = the rows of all column strips (image, 128-pixel segment) laid end to end, CTA i takes the i-th equal share: at most a
//     few pieces of consecutive strips, every SM the same number of rows (whole-strip segments left 20 of 148 SMs idle at
//     16 x 512 x 512), a piece re-reads only its halo rows;
//   * warp 0 = TMA producer (weights once, then one stage per input row), warp 1 = MMA issuer (and TMEM owner): it may run LEAD
//     steps ahead of the epilogue and waits for a FULL drain at a piece boundary, where the rows of a new strip map onto the slots
//     afresh;
//   * epilogue: drain a slot (tcgen05.ld, zero it with tcgen05.st so that the row wrapping onto it needs no special case, arrive
//     on drained[k] before anything else), fixed-order IN statistics, bf16 staging and one TMA store per warp and piece.
#pragma once
#include <cuda.h>

#include "common.cuh"
#include "tcgen05.cuh"

namespace msg {
namespace ring {
using namespace tc;

constexpr int BM = 128;                 // strip width (pixels = TMEM lanes)
constexpr int HALO = 4;                 // slab pixels left of the strip (4 keeps a 64-channel block a 1024-byte multiple)
constexpr int SLAB_PX = BM + 2 * HALO;  // 136
constexpr int SLAB_BYTES = SLAB_PX * 128;  // one 64-channel block of a row slab, SW128: 17408 = 17 * 1024
constexpr int EPI0 = 4;                 // first epilogue warp (warp & 3 = TMEM lane quarter)
constexpr int NBAR = 8;                 // rowdone / drained barrier rings (>= every LEAD)
constexpr int MAX_STAGES = 8;
constexpr int SMEM_BYTES = 227 * 1024;

// ---------------------------------------------------------------- shared memory
struct Layout {                         // byte offsets from the 1024-aligned base
  int w, a, bias, scratch, bar, tmem_slot;
  int bytes;                            // dynamic shared memory to request (with the alignment slack)
};
struct Shape {
  int w_bytes, stage_bytes, bias_floats, scratch_bytes;
  int stage_bars;                       // 2: full, empty; 3: + transformed
  __host__ __device__ constexpr Layout layout(int stages) const {
    Layout L{};
    L.w = 0;
    L.a = w_bytes;
    L.bias = L.a + stages * stage_bytes;
    L.scratch = (L.bias + bias_floats * 4 + 127) & ~127;
    L.bar = (L.scratch + scratch_bytes + 7) & ~7;
    L.tmem_slot = L.bar + 8 * (stage_bars * stages + 1 + 2 * NBAR);
    L.bytes = 1024 + L.tmem_slot + 4;
    return L;
  }
  // the deepest slab ring (at most MAX_STAGES) that fits next to everything else; < 2 = does not fit
  __host__ __device__ constexpr int stages() const {
    int s = MAX_STAGES;
    while (s > 0 && layout(s).bytes > SMEM_BYTES) --s;
    return s;
  }
};

struct Bars {
  uint32_t bar;
  int S, stage_bars;
  __device__ __forceinline__ uint32_t full(int s) const { return bar + 8u * s; }
  __device__ __forceinline__ uint32_t empty(int s) const { return bar + 8u * (S + s); }
  __device__ __forceinline__ uint32_t xf(int s) const { return bar + 8u * (2 * S + s); }   // slab transformed in place
  __device__ __forceinline__ uint32_t wres() const { return bar + 8u * (stage_bars * S); }
  __device__ __forceinline__ uint32_t rowdone(uint32_t k) const { return bar + 8u * (stage_bars * S + 1 + (k & (NBAR - 1))); }
  __device__ __forceinline__ uint32_t drained(uint32_t k) const { return bar + 8u * (stage_bars * S + 1 + NBAR + (k & (NBAR - 1))); }
  __device__ __forceinline__ void wait_rowdone(uint32_t k) const { mbar_wait(rowdone(k), (k / NBAR) & 1); }
  __device__ __forceinline__ void wait_drained(uint32_t k) const { mbar_wait(drained(k), (k / NBAR) & 1); }
};

// The kernel's view of its shared memory: generic pointer and shared-window address of the aligned base, the layout, the barriers.
struct Smem {
  uint8_t* gen;
  uint32_t base;
  Layout L;
  Bars b;
  __device__ __forceinline__ Smem(uint8_t* raw, const Shape& sh, int stages) {
    base = (smem_u32(raw) + 1023u) & ~1023u;
    gen = raw + (base - smem_u32(raw));
    L = sh.layout(stages);
    b = Bars{base + (uint32_t)L.bar, stages, sh.stage_bars};
  }
  __device__ __forceinline__ uint32_t sB() const { return base + (uint32_t)L.w; }
  __device__ __forceinline__ uint32_t sA(int s, int stage_bytes) const { return base + (uint32_t)(L.a + s * stage_bytes); }
  __device__ __forceinline__ float* bias() const { return reinterpret_cast<float*>(gen + L.bias); }
  __device__ __forceinline__ uint8_t* scratch(int i, int bytes) const { return gen + L.scratch + i * bytes; }
  __device__ __forceinline__ uint8_t* stage_ptr(int s, int stage_bytes) const { return gen + L.a + s * stage_bytes; }
  __device__ __forceinline__ uint32_t* tmem_slot() const { return reinterpret_cast<uint32_t*>(gen + L.tmem_slot); }
};

// Barrier init (warp 1; arrival counts per kernel), TMEM alloc, tensor-map prefetch, all 512 columns zeroed by the first four
// epilogue warps.  Returns the TMEM base address.
__device__ __forceinline__ uint32_t prologue(const Smem& sm, int warp, int lane, uint32_t issuers, uint32_t drainers, uint32_t xformers,
                                             const CUtensorMap* m0, const CUtensorMap* m1, const CUtensorMap* m2) {
  const Bars& b = sm.b;
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < b.S; ++s) {
        mbar_init(b.full(s), 1);
        mbar_init(b.empty(s), issuers);
        if (b.stage_bars == 3) mbar_init(b.xf(s), xformers);
      }
      mbar_init(b.wres(), 1);
      for (int k = 0; k < NBAR; ++k) { mbar_init(b.rowdone(k), issuers); mbar_init(b.drained(k), drainers); }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(sm.tmem_slot())), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  } else if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m0)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m1)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m2)) : "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *sm.tmem_slot();
  if (warp >= EPI0 && warp < EPI0 + 4) {
    const uint32_t lane_addr = (uint32_t)((warp & 3) * 32) << 16;
    uint32_t z[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) z[i] = 0u;
    for (int c = 0; c < 512; c += 32) tmem_st32(tmem_base + lane_addr + (uint32_t)c, z);
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  return tmem_base;
}

__device__ __forceinline__ void teardown(int warp, uint32_t tmem_base) {
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// ---------------------------------------------------------------- work
// This CTA's pieces (img, seg, [y0, y1) of the ROWS rows of a strip), in order.  A piece reads the input rows [r0, r1) =
// [A y0 - HV, A y1 + HV), one step each (rows outside the plane included: they keep every role's step count k in lockstep).
template <int A, int HV>
struct Pieces {
  long long g, hi;
  int rows, segs;
  int img, seg, y0, y1, r0, r1;
  __device__ __forceinline__ Pieces(long long total_rows, int rows_per_strip, int segs_)
      : g((long long)blockIdx.x * total_rows / gridDim.x), hi((long long)(blockIdx.x + 1) * total_rows / gridDim.x),
        rows(rows_per_strip), segs(segs_) {}
  __device__ __forceinline__ bool next() {
    if (g >= hi) return false;
    const int strip = (int)(g / rows);
    y0 = (int)(g - (long long)strip * rows);
    const long long left = hi - g;
    y1 = (long long)(rows - y0) < left ? rows : y0 + (int)left;
    img = strip / segs;
    seg = strip - img * segs;
    g += y1 - y0;
    r0 = A * y0 - HV;
    r1 = A * y1 + HV;
    return true;
  }
};

// Position in the slab ring: stage s of the n-th slab.
struct SlabRing {
  int S, s = 0;
  uint32_t n = 0;
  __device__ __forceinline__ explicit SlabRing(int stages) : S(stages) {}
  __device__ __forceinline__ uint32_t parity() const { return (n / S) & 1; }
  __device__ __forceinline__ void acquire(const Bars& b) const {          // producer: the stage's previous slab has been consumed
    if (n >= (uint32_t)S) mbar_wait(b.empty(s), ((n / S) - 1) & 1);
  }
  __device__ __forceinline__ void advance() {
    if (++s == S) s = 0;
    ++n;
  }
};

// Warp 0, lane 0: the resident weight stacks (w_bytes from weight row w_row0 of mapB), then one stage per input row inside
// the plane [0, H_in) of every piece: load(pc, r, stage address, full barrier) issues its TMA loads of stage_bytes.
template <class P, class Load>
__device__ __forceinline__ void producer(const Smem& sm, P pc, int H_in, const CUtensorMap* mapB, int w_bytes, int w_row0, int stage_bytes,
                                         Load&& load) {
  const Bars& b = sm.b;
  mbar_expect_tx(b.wres(), (uint32_t)w_bytes);
  for (int r = 0; r < w_bytes / 128; r += 64) tma_load_2d(sm.sB() + r * 128, mapB, b.wres(), 0, w_row0 + r);
  SlabRing ring(b.S);
  while (pc.next()) {
    const int r_lo = pc.r0 < 0 ? 0 : pc.r0, r_hi = pc.r1 > H_in ? H_in : pc.r1;
    for (int r = r_lo; r < r_hi; ++r) {
      ring.acquire(b);
      mbar_expect_tx(b.full(ring.s), (uint32_t)stage_bytes);
      load(pc, r, sm.sA(ring.s, stage_bytes), b.full(ring.s));
      ring.advance();
    }
  }
}

// An issuing warp.  Step k: wait until the epilogue has drained step k - LEAD (the slots this row first touches belonged to rows
// finished no later than that) and, at a piece boundary, everything; for a row inside the plane wait for its slab (landed, or
// transformed when XF), let the leader (the warp's elected thread) issue mmas(pc, r, stage) and free the stage with a commit; then
// commit rowdone[k], which arrives when every MMA issued so far has completed.  The caller elects the leader before it computes its
// descriptor constants: elected after them, the C = 128 MultiScaleBlock passes spilled uniform registers between their MMAs.
template <uint32_t LEAD, bool XF, class P, class Mmas>
__device__ __forceinline__ void issuer(const Bars& b, P pc, int H_in, bool leader, Mmas&& mmas) {
  static_assert(LEAD <= NBAR, "barrier rings shorter than the lead");
  SlabRing ring(b.S);
  uint32_t k = 0;
  mbar_wait(b.wres(), 0);
  while (pc.next()) {
    for (int r = pc.r0; r < pc.r1; ++r, ++k) {
      if (k >= LEAD) b.wait_drained(k - LEAD);
      if (r == pc.r0 && k > 0) b.wait_drained(k - 1);
      if (r >= 0 && r < H_in) {
        mbar_wait(XF ? b.xf(ring.s) : b.full(ring.s), ring.parity());
        tc_fence_after();
        if (leader) {
          mmas(pc, r, ring.s);
          umma_commit(b.empty(ring.s));
        }
        __syncwarp();
        ring.advance();
      }
      if (leader) umma_commit(b.rowdone(k));
      __syncwarp();
    }
  }
}

// The entries [first, first + cnt) of a ring of LEN slots starting at slot `slot` are adjacent except where the ring wraps: one or
// two runs run(entry offset, length, slot), found by arithmetic (a run table in local memory cost the issuing thread ~1000 cycles
// per row).
template <class Run>
__device__ __forceinline__ void runs(int cnt, int slot, int len, Run&& run) {
  const int n1 = cnt < len - slot ? cnt : len - slot;
  run(0, n1, slot);
  if (cnt > n1) run(n1, cnt - n1, 0);
}

__device__ __forceinline__ uint32_t idesc_bf16(int n) {   // bf16 x bf16 -> fp32, K-major A and B, M = BM
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

// ---------------------------------------------------------------- epilogue
template <int N>
__device__ __forceinline__ void tmem_ld_n(uint32_t taddr, float (&v)[N]) {
  static_assert(N == 16 || N == 32, "");
  if constexpr (N == 16) tmem_ld16(taddr, v); else tmem_ld32(taddr, v);
}
template <int N>
__device__ __forceinline__ void tmem_zero(uint32_t taddr) {
  uint32_t z[N];
#pragma unroll
  for (int i = 0; i < N; ++i) z[i] = 0u;
  if constexpr (N == 16) tmem_st16(taddr, z); else tmem_st32(taddr, z);
}
// after the slots of step k are read and zeroed: hand them back before anything else (the issuer waits on this)
__device__ __forceinline__ void arrive_drained(const Bars& b, uint32_t k, int lane) {
  __syncwarp();
  if (lane == 0) mbar_arrive(b.drained(k));
}

// IN statistics: a running (sum, sum of squares) per lane = channel, two-float sums, fp64 atomics once per image.
struct Stats {
  float2 ws = make_float2(0.f, 0.f), wq = make_float2(0.f, 0.f);
  int img = -1;
  // flush the sums of the previous image of this warp's channels [ch0, ch0 + NCH) into stats[img][C_total][2]
  template <int NCH>
  __device__ __forceinline__ void flush(double* stats, int C_total, int ch0, int lane) {
    if (img >= 0 && lane < NCH) {
      double* st = stats + ((size_t)img * C_total + ch0 + lane) * 2;
      atomicAdd(st, f2sum_value(ws));
      atomicAdd(st + 1, f2sum_value(wq));
    }
    ws = make_float2(0.f, 0.f); wq = make_float2(0.f, 0.f);
  }
};

// Per-channel sums over the warp's 32 pixels of v[NCH] (pixels outside the plane count 0), 16 channels at a time through sc as
// [16 ch][32 px] fp32 (pixel index XOR channel: conflict-free both ways); lane (c, half) sums 16 pixels of channel c in a fixed
// order on two chains, one shuffle joins the halves (pixels 0-15 first on both: the same bits); lane l accumulates channel l.
template <int NCH>
__device__ __forceinline__ void piece_stats(float* sc, const float (&v)[NCH], bool valid, int lane, Stats& st) {
#pragma unroll
  for (int h = 0; h < NCH / 16; ++h) {
#pragma unroll
    for (int c = 0; c < 16; ++c) sc[c * 32 + (lane ^ c)] = valid ? v[16 * h + c] : 0.f;
    __syncwarp();
    const int c = lane & 15, r0 = lane & 16;
    float cs0 = 0.f, cs1 = 0.f, q0 = 0.f, q1 = 0.f;
#pragma unroll
    for (int j = 0; j < 16; j += 2) {
      const float x0 = sc[c * 32 + ((r0 + j) ^ c)], x1 = sc[c * 32 + ((r0 + j + 1) ^ c)];
      cs0 += x0; cs1 += x1;
      q0 = fmaf(x0, x0, q0); q1 = fmaf(x1, x1, q1);
    }
    float cs = cs0 + cs1, qs = q0 + q1;
    const float cs_o = __shfl_xor_sync(0xffffffffu, cs, 16), qs_o = __shfl_xor_sync(0xffffffffu, qs, 16);
    cs = r0 ? cs_o + cs : cs + cs_o;
    qs = r0 ? qs_o + qs : qs + qs_o;
    if ((lane >> 4) == h) { f2sum_add(st.ws, cs); f2sum_add(st.wq, qs); }
    __syncwarp();
  }
}

// lane 0 waits until at most N of the warp's TMA stores still read their staging buffers
template <int N>
__device__ __forceinline__ void wait_store_read(int lane) {
  if (lane == 0) asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
  __syncwarp();
}

// The warp's [32 pixels x Q channels] piece as bf16 into stg (rows of Q * 2 bytes, dense: the TMA store reads them un-swizzled),
// then ONE TMA store at (c0, c1, c2, c3); the tensor map clips pixels beyond the plane.  The 16-byte chunk a lane writes at step j
// is rotated by the lane, so the eight lanes of a store phase cover all 32 banks.  (Per-thread global stores -- 32 scattered sectors
// per warp instruction -- held the kernels back.)
template <int Q>
__device__ __forceinline__ void store_piece_bf16(uint8_t* stg, const float (&v)[Q], int lane, const CUtensorMap* map, int c0, int c1, int c2,
                                                 int c3) {
  uint4 pk[Q / 8];
#pragma unroll
  for (int c8 = 0; c8 < Q / 8; ++c8) {
    float o8[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) o8[c] = v[c8 * 8 + c];
    pk[c8] = pack8(o8);
  }
  const int rot = Q == 16 ? ((lane >> 2) & 1) : ((lane >> 1) & 3);
#pragma unroll
  for (int bit = 1; bit < Q / 8; bit <<= 1) {
    const bool sw = (rot & bit) != 0;
#pragma unroll
    for (int j = 0; j < Q / 8; ++j) {
      if (j & bit) continue;
      const uint4 a = pk[j], c2 = pk[j | bit];
      pk[j] = sw ? c2 : a;
      pk[j | bit] = sw ? a : c2;
    }
  }
#pragma unroll
  for (int j = 0; j < Q / 8; ++j) *reinterpret_cast<uint4*>(stg + lane * (Q * 2) + (j ^ rot) * 16) = pk[j];
  fence_proxy_async();
  __syncwarp();
  if (lane == 0) {
    tma_store_4d(map, smem_u32(stg), c0, c1, c2, c3);
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  }
}

// ---------------------------------------------------------------- transform warps
// Thread t of the four transform warps owns the physical 16-byte chunk (t & 7) of the slab rows (t >> 3) + 16 i: because the
// 128-byte swizzle only uses row & 7, the LOGICAL channel chunk is the same for all its rows and its 8 per-image scales / shifts
// (in_scale_shift: x * rstd * gamma + beta - mean * rstd * gamma, the affine optional) live in registers.
__device__ __forceinline__ void load_scale_shift(const double* in_stats, const float* in_gamma, const float* in_beta, int in_img_stride,
                                                 int img, int Cs_total, int cs_off, int lchunk, double inv_hw, float (&sc)[8], float (&sh)[8]) {
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = cs_off + lchunk * 8 + e;
    float g, b, mean, rstd;
    in_affine(in_gamma, in_beta, (size_t)img * in_img_stride + c, g, b);
    in_scale_shift(in_stats + ((size_t)img * Cs_total + c) * 2, inv_hw, g, b, mean, rstd, sc[e], sh[e]);
  }
}

// ---------------------------------------------------------------- host
// bf16 tensor maps: loads are 128-byte swizzled with 256-byte L2 promotion, stores plain.  strides: rank - 1 byte strides.
inline CUresult encode(CUtensorMap* m, int rank, const void* ptr, const cuuint64_t* dims, const cuuint64_t* strides, const cuuint32_t* box,
                       bool load) {
  const cuuint32_t es[5] = {1, 1, 1, 1, 1};
  return get_encode()(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(ptr), dims, strides, box, es,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, load ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                      load ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B : CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}
// row slabs of C channels of an NHWC tensor [N][H][W][C_total] (starting at the channel of ptr): 64-channel x 136-pixel boxes
inline CUresult encode_slab(CUtensorMap* m, const void* ptr, int C, int C_total, int W, int H, int N) {
  const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  const cuuint64_t strides[3] = {(cuuint64_t)C_total * 2, (cuuint64_t)W * C_total * 2, (cuuint64_t)H * W * C_total * 2};
  const cuuint32_t box[4] = {64, (cuuint32_t)SLAB_PX, 1, 1};
  return encode(m, 4, ptr, dims, strides, box, true);
}
// weight stacks: rows of 64 bf16, 64-row boxes
inline CUresult encode_weights(CUtensorMap* m, const void* ptr, long long rows) {
  const cuuint64_t dims[2] = {64, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {128};
  const cuuint32_t box[2] = {64, 64};
  return encode(m, 2, ptr, dims, strides, box, true);
}
// [32 px x box_c ch] pieces into an NHWC tensor [N][H][W][C_total] whose pixels lie px_stride apart (the map covers every px_stride-th)
inline CUresult encode_store(CUtensorMap* m, void* ptr, int C_total, int W, int H, int N, int box_c, int px_stride) {
  const cuuint64_t px = (cuuint64_t)px_stride * C_total * 2;
  const cuuint64_t dims[4] = {(cuuint64_t)C_total, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  const cuuint64_t strides[3] = {px, px * W, px * W * H};
  const cuuint32_t box[4] = {(cuuint32_t)box_c, 32, 1, 1};
  return encode(m, 4, ptr, dims, strides, box, false);
}

// One launch of a ring kernel: the stage count from the layout, the 227 KB opt-in once per device (the latch is per kernel:
// template <auto Kernel>), grid = min(SMs, rows / min_rows).
template <auto Kernel, class P>
int launch(const char* name, const Shape& sh, int threads, long long total_rows, int min_rows, P p, const CUtensorMap& m0,
           const CUtensorMap& m1, const CUtensorMap& m2, cudaStream_t st) {
  p.stages = sh.stages();
  MSG_REQUIRE(p.stages >= 2, MSG_ERR_UNSUPPORTED, "%s: the slab ring does not fit shared memory", name);
  static DeviceOnce attr_set;
  if (attr_set.needed()) {
    cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    MSG_REQUIRE(e == cudaSuccess, MSG_ERR_CUDA, "%s: cudaFuncSetAttribute: %s", name, cudaGetErrorString(e));
    attr_set.done();
  }
  const int sms = sm_count();
  const long long grid_ll = total_rows / min_rows;
  const int grid = grid_ll < 1 ? 1 : (grid_ll > sms ? sms : (int)grid_ll);
  Kernel<<<grid, threads, (size_t)sh.layout(p.stages).bytes, st>>>(m0, m1, m2, p);
  return check_launch(name);
}

}  // namespace ring
}  // namespace msg
