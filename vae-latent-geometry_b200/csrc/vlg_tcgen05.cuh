// Thin inline-PTX wrappers for the Blackwell (sm_100a) primitives the tensor-core kernels
// use: mbarrier, 1-D bulk async copy (TMA engine, UBLKCP), TMEM allocation, tcgen05.ld/st,
// tcgen05.mma kind::tf32 with the A operand in TMEM, tcgen05.commit.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace vlg {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }

// ---- mbarrier ----------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// (a suspend-time hint on try_wait made no difference: polling only fills idle issue slots)
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ---- 1-D bulk copy global -> shared, completion on an mbarrier (TMA engine) ---------------
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ---- proxies / fences ----------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- TMEM allocation (one full warp) --------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// ---- TMEM <-> registers: lane = 32*(warp%4)+laneid, N consecutive 32-bit columns ----------
#define VLG_R8(v, o) "=r"(v[o + 0]), "=r"(v[o + 1]), "=r"(v[o + 2]), "=r"(v[o + 3]), "=r"(v[o + 4]), "=r"(v[o + 5]), "=r"(v[o + 6]), "=r"(v[o + 7])
#define VLG_W8(v, o) "r"(v[o + 0]), "r"(v[o + 1]), "r"(v[o + 2]), "r"(v[o + 3]), "r"(v[o + 4]), "r"(v[o + 5]), "r"(v[o + 6]), "r"(v[o + 7])

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : VLG_R8(v, 0), VLG_R8(v, 8)
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : VLG_R8(v, 0), VLG_R8(v, 8), VLG_R8(v, 16), VLG_R8(v, 24)
      : "r"(taddr)
      : "memory");
}
// Load + wait fused into ONE asm statement: the destination registers only become visible to
// the compiler after tcgen05.wait::ld, so it cannot schedule their consumers before the wait
// (separate asm statements do not order register uses -- that bit us once).
__device__ __forceinline__ void tmem_ld32_sync(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : VLG_R8(v, 0), VLG_R8(v, 8), VLG_R8(v, 16), VLG_R8(v, 24)
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32x2_sync(uint32_t taddr0, uint32_t taddr1, uint32_t (&a)[32], uint32_t (&b)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%64];\n\t"
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%32,%33,%34,%35,%36,%37,%38,%39,%40,%41,%42,%43,%44,%45,%46,%47,%48,%49,%50,%51,%52,%53,%54,%55,%56,%57,%58,%59,%60,%61,%62,%63}, [%65];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : VLG_R8(a, 0), VLG_R8(a, 8), VLG_R8(a, 16), VLG_R8(a, 24), VLG_R8(b, 0), VLG_R8(b, 8), VLG_R8(b, 16), VLG_R8(b, 24)
      : "r"(taddr0), "r"(taddr1)
      : "memory");
}
__device__ __forceinline__ void tmem_ld8_sync(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : VLG_R8(v, 0)
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&v)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]),
               "r"(v[3])
               : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), VLG_W8(v, 0)
               : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      VLG_W8(v, 0), VLG_W8(v, 8)
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
      VLG_W8(v, 0), VLG_W8(v, 8), VLG_W8(v, 16), VLG_W8(v, 24)
      : "memory");
}

// ---- UMMA descriptors ------------------------------------------------------------------------
// Shared-memory matrix descriptor, no swizzle ("interleaved" canonical layout of 8x16B core
// matrices), sm_100 version field = 1.  lbo/sbo in bytes (multiples of 16).
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= uint64_t((saddr >> 4) & 0x3FFF);
  d |= uint64_t((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= uint64_t((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= uint64_t(1) << 46;  // descriptor version (Blackwell)
  return d;                // base_offset = 0, lbo_mode = 0, layout_type = SWIZZLE_NONE
}

// Instruction descriptor for kind::tf32, fp32 accumulate, A K-major (TMEM), M = 128.
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int N, int b_mn_major) {
  return (1u << 4)                       // D format F32
         | (2u << 7) | (2u << 10)        // A, B format TF32
         | (uint32_t(b_mn_major) << 16)  // B major-ness
         | (uint32_t(N >> 3) << 17)      // N
         | (uint32_t(128 >> 4) << 24);   // M
}

// Instruction descriptor for kind::f16 with fp16 A and B (format code 0), fp32 accumulate, M = 128.
__host__ __device__ constexpr uint32_t umma_idesc_f16(int N) {
  return (1u << 4)                      // D format F32
         | (uint32_t(N >> 3) << 17)     // N
         | (uint32_t(128 >> 4) << 24);  // M
}

// D[tmem] (+)= A[tmem] * B[smem]; issued by ONE thread.
__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Warp-convergent forms: every lane of the issuing warp executes the statement, `leader` (0/1, from
// elect_one) selects the lane whose instruction takes effect.  Keeping the issue loop convergent
// lets ptxas emit a bare predicated UTCHMMA; inside an `if (lane == 0)` branch it wraps every MMA in
// an ELECT / BRA.U.ANY serialisation loop (~12 instructions, ~100 cycles per MMA -- more than the
// tensor core needs for the MMA itself).
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t leader;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(leader));
  return leader;
}
__device__ __forceinline__ void umma_tf32_ts_elect(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                                   uint32_t accumulate, uint32_t leader) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 q, %5, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(leader)
      : "memory");
}
// kind::f16: A holds two 16-bit values per TMEM column (K = 16 per instruction = 8 columns)
__device__ __forceinline__ void umma_f16_ts_elect(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                                  uint32_t accumulate, uint32_t leader) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 q, %5, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(leader)
      : "memory");
}
// Both operands in shared memory (descriptors): D[tmem] (+)= A[smem] * B[smem].
__device__ __forceinline__ void umma_f16_ss_elect(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                  uint32_t accumulate, uint32_t leader) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 q, %5, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void umma_tf32_ss_elect(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                   uint32_t accumulate, uint32_t leader) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 q, %5, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(leader)
      : "memory");
}
// generic-proxy writes (st.global / st.shared) made visible to the async proxy (TMA reads, tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void umma_commit_elect(uint64_t* bar, uint32_t leader) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "setp.ne.b32 q, %1, 0;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar)),
      "r"(leader)
      : "memory");
}

// Arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

}  // namespace tc
}  // namespace vlg
