// tcgen05 / TMEM / TMA / mbarrier primitives (inline PTX) shared by the sm_100a convolution kernels
// (conv_tma.cu, conv_slab.cu, conv_shift.cu, conv_wgrad_tc.cu, conv_tc.cu).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace msg {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// try_wait with a suspend-time hint: without one a waiting warp comes back every ~30 cycles and the BRA / TRYWAIT / YIELD
// of its retry loop were 56 % of the instructions the fused LocalAttention kernel executed (ncu source page) -- issue slots
// taken from the warps doing the work.  With the hint the hardware parks the warp until the phase completes or the time is up.
#ifndef MSG_MBAR_SUSPEND_HINT
#define MSG_MBAR_SUSPEND_HINT 0x989680u
#endif
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity), "r"(MSG_MBAR_SUSPEND_HINT) : "memory");
  } while (!done);
}
// mbar_wait with back-off.  Measured on B200 (ncu source page of the fused LocalAttention kernel, 28 warps per CTA): try_wait
// comes back within ~30 cycles whatever the hint, so a waiting warp is an ELIGIBLE warp executing TRYWAIT / BRA / YIELD -- 56 % of
// all instructions executed -- and with ~5 waiting warps per scheduler the one warp with work to do got a fraction of the issue
// slots (9 cycles per instruction in the accumulator drain).  nanosleep takes the waiting warp out of the scheduler's rotation.
template <int NS>
__device__ __forceinline__ void mbar_wait_sleep(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done) : "r"(bar), "r"(parity) : "memory");
  while (!done) {
    asm volatile("nanosleep.u32 %0;" ::"r"((uint32_t)NS));
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
  }
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_bf16_acc(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 1;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc) : "memory");
}
// tcgen05.mma with descriptors given as {32-bit start-address word, constant high word}: the per-K-step advance is a
// 32-bit add on the low word (the 14-bit address field cannot carry), no 64-bit add-with-carry chains
__device__ __forceinline__ void umma_bf16_lo(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t hi, uint32_t idesc, bool acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 da, {%1, %3};\n\tmov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}"
      ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(hi), "r"(idesc), "r"((uint32_t)acc) : "memory");
}

// as umma_bf16_lo with separate high words for A and B (different layouts)
__device__ __forceinline__ void umma_bf16_lo2(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                              uint32_t idesc, bool acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"((uint32_t)acc) : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4) : "memory");
}
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3, int c4) {
  asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4) : "memory");
}
// tcgen05.mma with the A operand read from TENSOR MEMORY (lane = row, 16-bit elements packed two per 32-bit column,
// K-major only) and B from shared memory: the P.V product of the fused LocalAttention stage (P never leaves TMEM)
__device__ __forceinline__ void umma_ts_lo(uint32_t tmem_d, uint32_t tmem_a, uint32_t b_lo, uint32_t b_hi, uint32_t idesc, bool acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\tsetp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"((uint32_t)acc) : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
      "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
        "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
        "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31]) : "memory");
}
// non-blocking probe of an mbarrier phase (polling issuers that serve several queues)
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done) : "r"(bar), "r"(parity) : "memory");
  return done != 0;
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, float (&v)[4]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld1(uint32_t taddr, float (&v)[1]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r[0]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
                 "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// A operand: K-major, no swizzle: 8-row x 16-byte core matrices; SBO = 128 B between 8-row groups
// (rows are 16 B apart), LBO = byte distance between the two K chunks of one UMMA_K=16 step.
__device__ __forceinline__ uint64_t make_noswz_desc(uint32_t saddr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)(128 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}
// MN-major, 128-byte swizzle: atoms of [8 K-rows x 64 MN-elements] = 1024 B; SBO = 1024 (next 8 K rows),
// LBO = distance to the next 64-element MN block (here: the next 16 KB box).
__device__ __forceinline__ uint64_t make_mn_sw128_desc(uint32_t saddr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// column sums over the 32 lanes of a warp by recursive halving: on return v[0] of lane l holds the
// sum over all lanes of the original v[l].
__device__ __forceinline__ float warp_transpose_reduce32(float (&v)[32], int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool up = lane & off;
#pragma unroll
    for (int i = 0; i < off; ++i) {
      float send = up ? v[i] : v[i + off];
      float keep = up ? v[i + off] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

// tcgen05.ld of 32 columns followed by the wait (for epilogues that consume the values immediately)
__device__ __forceinline__ void tmem_ld32_sync(uint32_t taddr, float (&v)[32]) {
  tmem_ld32(taddr, v);
  tmem_ld_wait();
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

}  // namespace tc
}  // namespace msg
