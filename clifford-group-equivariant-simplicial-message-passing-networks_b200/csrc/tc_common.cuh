// tcgen05 / TMEM / mbarrier helpers for the tensor-core kernels (sm_100a only; inline PTX, no CUTLASS).
//
// Operand layout used by every tensor-core kernel of this library ("plane" layout, no swizzle):
//   a plane holds a [R rows x Cc channels] fp32 matrix as 16-byte units of 4 consecutive channels,
//       byte offset of (r, c) = ((c / 4) * R + r) * 16 + (c % 4) * 4
//   i.e. [Cc/4][R][4].  Eight consecutive rows of one unit column are 128 contiguous bytes = one UMMA core matrix.
//   Used as a K-major operand (MMA rows = plane rows, K = channels): one K=8 step is two unit columns,
//   LBO (K direction) = R*16 bytes, SBO (8-row groups) = 128 bytes, start = base + 2*ks*R*16
//   (canonical SWIZZLE_NONE K-major layout ((8,n),2):((1,SBO),LBO) in 16-byte units).
// MN-major TF32 operands (K = plane rows, MMA rows = channels; the weight-gradient GEMMs) only exist in the
// SWIZZLE_128B_BASE32B layout: 32-channel groups of [rows][128 B], the 32-byte unit index of a row xor-ed with
// (row & 3); LBO = byte stride between 32-channel groups, SBO = 512 (groups of 4 rows), one K=8 step = 1024 bytes.
// Every encoding here was pinned on a B200 with tools/tc_probe_raw.py (profiles/r01_tc_probe.log).
// fp32 accuracy on the TF32 pipe comes from the usual error-compensated split  x = hi + lo  with hi = x with the low
// 13 mantissa bits cleared (exactly representable in TF32) and three MMAs per product: hi*hi + hi*lo + lo*hi.
// Single-pass TF32 mode (csmpn_block_desc.tf32, kernels instantiated with TERMS = 1) rounds each operand to nearest TF32
// once and issues one MMA per product.
#pragma once
#include "common.cuh"

namespace csmpn {
namespace tc {

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ------------------------------------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_addr(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// bulk async copy global -> shared, completion counted on an mbarrier (bytes % 16 == 0, 16-byte aligned both sides)
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_addr(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_addr(bar))
               : "memory");
}
// generic-proxy writes to shared memory -> visible to the async proxy (UMMA operand reads, bulk copies)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------ TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {  // one full warp; cols = 2^k >= 32
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr(dst_smem)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {  // the allocating warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// warp-collective loads: lane l of the warp reads TMEM lane (taddr.lane + l), N consecutive 32-bit columns
__device__ __forceinline__ void tmem_ld1(uint32_t taddr, float& v) {
  uint32_t r;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(taddr));
  v = __uint_as_float(r);
}
__device__ __forceinline__ void tmem_ld2(uint32_t taddr, float* v) {
  uint32_t r0, r1;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(taddr));
  v[0] = __uint_as_float(r0); v[1] = __uint_as_float(r1);
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, float* v) {
  uint32_t r0, r1, r2, r3;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(taddr));
  v[0] = __uint_as_float(r0); v[1] = __uint_as_float(r1); v[2] = __uint_as_float(r2); v[3] = __uint_as_float(r3);
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const float* v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(__float_as_uint(v[0])),
               "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3]))
               : "memory");
}
// TMEM address of (lane, column) relative to an allocation base
__device__ __forceinline__ uint32_t tmem_at(uint32_t base, uint32_t lane, uint32_t col) { return base + (lane << 16) + col; }

// ------------------------------------------------------------------------------------------------ UMMA descriptors
// shared-memory matrix descriptor, SWIZZLE_NONE, Blackwell version field = 1
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}
// K-major view of a plane with R rows: K step ks (8 channels)
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t plane_saddr, uint32_t R, uint32_t ks) {
  return smem_desc(plane_saddr + 2u * ks * R * 16u, R * 16u, 128u);
}
// MN-major TF32 operand: [rows][32 channels] groups in the SWIZZLE_128B_BASE32B layout (base 512-byte aligned),
// K step ks = rows 8*ks .. 8*ks+7; group_stride = bytes between consecutive 32-channel groups
__device__ __forceinline__ uint64_t desc_mn32b(uint32_t base_saddr, uint32_t group_stride, uint32_t ks) {
  return smem_desc(base_saddr + ks * 1024u, group_stride, 512u) | ((uint64_t)1 << 61);
}
// byte offset of (row r, channel c < 32) inside one 32-channel group of that layout
__host__ __device__ constexpr uint32_t mn32b_off(uint32_t r, uint32_t c) {
  return r * 128u + ((((c >> 3) ^ (r & 3u)) << 5) | ((c & 7u) << 2));
}
// instruction descriptor: kind::tf32, fp32 accumulate, dense; a_mn / b_mn = operand is MN-major
__host__ __device__ constexpr uint32_t idesc_tf32(int M, int N, bool a_mn, bool b_mn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// One elected lane of a fully converged warp.  The MMA-issuing code is executed by the WHOLE warp with only the
// tcgen05 instructions predicated on the elected lane: descriptors then live in uniform registers.  (Issuing from
// inside an `if (lane == 0)` region costs ~65 cycles per MMA: every operand goes through an R2UR waterfall loop.)
__device__ __forceinline__ uint32_t elect_one_sync() {
  uint32_t pred = 0, laneid = 0;
  asm volatile(
      "{\n\t.reg .b32 %%rx;\n\t.reg .pred %%px;\n\t"
      "elect.sync %%rx|%%px, %2;\n\t"
      "@%%px mov.s32 %1, 1;\n\t"
      "mov.s32 %0, %%rx;\n\t}"
      : "+r"(laneid), "+r"(pred)
      : "r"(0xFFFFFFFFu));
  return pred;
}
// warp index as a provably warp-uniform value
__device__ __forceinline__ int uniform_warp_idx() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread
__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// warp-collective forms: call from a converged warp, one elected lane issues
__device__ __forceinline__ void mma_tf32_w(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  if (elect_one_sync()) mma_tf32(d_tmem, adesc, bdesc, idesc, accumulate);
}
__device__ __forceinline__ void mma_commit(uint64_t* bar);
__device__ __forceinline__ void mma_commit_w(uint64_t* bar) {
  if (elect_one_sync()) mma_commit(bar);
}
// all MMAs issued so far by this thread -> one arrival on the mbarrier when they have completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_addr(bar)) : "memory");
}

// 256-bit global accesses (sm_100: LDG/STG.E.ENL2.256): one Cl(3,0) multivector in the reference layout is 32 bytes, so a
// (row, channel) element is one full sector per instruction instead of two half-sector float4 accesses.  32-byte aligned.
__device__ __forceinline__ void ld_global_v8(float* v, const float* p) {
  asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
               : "l"(p));
}
__device__ __forceinline__ void st_global_v8(float* p, const float* v) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
               "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
               : "memory");
}
__device__ __forceinline__ bool aligned32(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 31u) == 0; }

// ------------------------------------------------------------------------------------------------ split
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }
// single-pass TF32 operand: x rounded to the nearest TF32 value (ties away from zero), low 13 mantissa bits zero, so the
// truncating operand read of kind::tf32 takes it exactly
__device__ __forceinline__ float tf32_rna(float x) {
  uint32_t y;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(y) : "f"(x));
  return __uint_as_float(y);
}
__device__ __forceinline__ float4 tf32_rna4(const float4& x) { return make_float4(tf32_rna(x.x), tf32_rna(x.y), tf32_rna(x.z), tf32_rna(x.w)); }
__device__ __forceinline__ void split4(const float4& x, float4& hi, float4& lo) {
  hi.x = tf32_hi(x.x); hi.y = tf32_hi(x.y); hi.z = tf32_hi(x.z); hi.w = tf32_hi(x.w);
  lo.x = x.x - hi.x; lo.y = x.y - hi.y; lo.z = x.z - hi.z; lo.w = x.w - hi.w;
}
// byte offset of (row r, channel c) in a plane with R rows
__host__ __device__ constexpr uint32_t plane_off(uint32_t R, uint32_t r, uint32_t c) { return ((c >> 2) * R + r) * 16u + (c & 3u) * 4u; }

}  // namespace tc
}  // namespace csmpn
