// Thin inline-PTX wrappers for the sm_100a features the tensor-core kernels use:
// mbarrier, bulk async copy (TMA engine, 1-D), tcgen05 (alloc / mma / commit / ld / fences),
// the shared-memory matrix / instruction descriptors of tcgen05.mma, and the SW128 operand-tile format the kernels share.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t lane_id() { uint32_t l; asm volatile("mov.u32 %0, %%laneid;" : "=r"(l)); return l; }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n .reg .pred p;\n elect.sync _|p, 0xffffffff;\n selp.u32 %0, 1, 0, p;\n}" : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- programmatic dependent launch
// pdl_trigger(): lets the next kernel of the stream be scheduled early (its prologue overlaps this kernel's tail);
// pdl_wait(): blocks until the previous kernel of the stream has completed and its writes are visible.  Both are
// no-ops for a kernel launched without the programmatic-serialization attribute.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
               : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {}
}

// ---------------------------------------------------------------- bulk async copy global -> shared (TMA engine)
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// pull a global range into L2 ahead of the bulk copy that will need it (no shared-memory destination, no barrier)
__device__ __forceinline__ void bulk_prefetch_l2(const void *src_gmem, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src_gmem), "r"(bytes) : "memory");
}
// bulk async copy shared -> global (TMA engine), tracked by bulk groups
__device__ __forceinline__ void bulk_s2g(void *dst_gmem, const void *src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// named barrier over a subset of the CTA's warps
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t *dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]^T, kind::f16 (fp16/bf16 operands, fp32 accumulate), one CTA
__device__ __forceinline__ void mma_f16_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}"
               ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// mbarrier arrive once every tcgen05 op issued so far by this thread has completed (implies fence::before_thread_sync)
__device__ __forceinline__ void mma_commit(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets lane (base_lane + i), columns col..col+31
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- packed fp32x2 math (sm_100: FADD2 / FMUL2 / FFMA2)
__device__ __forceinline__ uint64_t pack2(float lo, float hi) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ uint64_t pack2u(uint32_t lo, uint32_t hi) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi)); return r; }
__device__ __forceinline__ void unpack2(uint64_t v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) { uint64_t r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
// volatile variant: keeps its program-order position among other volatile asm statements (MUFU streams, barriers)
__device__ __forceinline__ uint64_t add2v(uint64_t a, uint64_t b) { uint64_t r; asm volatile("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t sub2(uint64_t a, uint64_t b) { uint64_t r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) { uint64_t r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) { uint64_t r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }

template <int N> __device__ __forceinline__ void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

// ---------------------------------------------------------------- descriptors
// Shared-memory matrix descriptor, 128-byte swizzle (layout_type 2), descriptor version 1 (sm_100).
//   bits [0,14) start address >> 4, [16,30) leading byte offset >> 4, [32,46) stride byte offset >> 4,
//   [46,48) version, [61,64) layout type.
// K-major operand (rows = M/N index, 64 fp16 = 128 B per row, 8-row groups of 1024 B):
//   SBO = 1024 (next 8-row group), LBO unused (1).  Advancing K by 16 elements = +32 B on the start address.
// MN-major operand (rows = K index, 64 M/N elements = 128 B per row, 8-row groups of 1024 B):
//   SBO = byte distance between 8-row K groups, LBO = byte distance between 64-element M/N groups.
__host__ __device__ constexpr uint64_t smem_desc_sw128(uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) | ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46) |
         ((uint64_t)2 << 61);
}
__device__ __forceinline__ uint64_t smem_desc_at(uint64_t base_desc, uint32_t smem_addr) {
  return base_desc | (uint64_t)((smem_addr >> 4) & 0x3FFF);
}
// Instruction descriptor, kind::f16: fp16 A/B (format 0), fp32 accumulator (c_format 1 at bit 4),
// a_major bit 15, b_major bit 16 (0 = K-major, 1 = MN-major), N>>3 at [17,23), M>>4 at [24,29).
__host__ __device__ constexpr uint32_t idesc_f16(uint32_t M, uint32_t N, uint32_t a_mn_major, uint32_t b_mn_major) {
  return (1u << 4) | (a_mn_major << 15) | (b_mn_major << 16) | ((N >> 3) << 17) | ((M >> 4) << 24);
}
// same with bf16 A/B operands (format 1 at bits [7,10) and [10,13))
__host__ __device__ constexpr uint32_t idesc_bf16(uint32_t M, uint32_t N, uint32_t a_mn_major, uint32_t b_mn_major) {
  return idesc_f16(M, N, a_mn_major, b_mn_major) | (1u << 7) | (1u << 10);
}

// Byte offset of element (row, col) of a [rows x 64]-fp16 K-major SW128 sub-tile (16 KB for 128 rows):
// row r at r*128, 16-byte chunk j stored at position j ^ (r & 7).
__host__ __device__ constexpr uint32_t sw128_offset(uint32_t row, uint32_t col /* 0..63 */) {
  return row * 128u + ((((col >> 3) ^ (row & 7u)) << 4) | ((col & 7u) << 1));
}

// The 128 x 128 operand tile of the attention kernels (Kq, Kc, Vc^T, Uc): two 16 KB SW128 sub-tiles of 64 columns
constexpr int DD = 128;
constexpr uint32_t IMG_BYTES = 128 * DD * 2;
constexpr uint32_t SUB_BYTES = 128 * 64 * 2;

__device__ __forceinline__ uint32_t pack_half2(float lo, float hi) {
  __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t *>(&h);
}
__device__ __forceinline__ uint32_t pack_bf162(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t *>(&h);
}

}  // namespace ptx
