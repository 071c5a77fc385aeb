// Blackwell (sm_100a) primitives used by the tcgen05 kernels: mbarrier, TMA
// (cp.async.bulk.tensor), TMEM allocation, tcgen05.mma / commit / ld, UMMA
// shared-memory and instruction descriptors.  Inline PTX only.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace stg {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Bounded wait: a protocol bug traps (kernel error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  const long long t0 = clock64();
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (ok) break;
    if (clock64() - t0 > 4000000000LL) __trap();
  }
}

__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// Elected forms for WARP-UNIFORM code (all 32 lanes converged, operands uniform): elect.sync picks one lane and only its
// instruction takes effect.  ptxas knows the elected predicate selects exactly one thread, so it emits the single-issuer
// instruction (UTMALDG / UTCHMMA / UTCBAR) directly with uniform-register operands - a `lane == 0` predicate makes it
// wrap every such instruction in a loop over the (possibly many) threads for which the predicate holds.
#define STG_EL_BEGIN "{\n\t.reg .pred P_el;\n\telect.sync _|P_el, 0xffffffff;\n\t"
__device__ __forceinline__ void mbar_expect_tx_el(uint32_t bar, uint32_t bytes) {
  asm volatile(STG_EL_BEGIN "@P_el mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_3d_el(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(STG_EL_BEGIN
      "@P_el cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n\t}"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_4d_el(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(STG_EL_BEGIN
      "@P_el cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n\t}"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void umma_bf16_el(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(STG_EL_BEGIN ".reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "@P_el tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
               ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit_el(uint32_t bar) {
  asm volatile(STG_EL_BEGIN "@P_el tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar) : "memory");
}

// elected TMA stores / bulk-group bookkeeping (bulk groups belong to the issuing THREAD: elect.sync with a full mask
// picks the same lane every time, so stores, commit and wait of the epilogue DMA warp all land on one thread)
__device__ __forceinline__ void tma_store_4d_el(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile(STG_EL_BEGIN "@P_el cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];\n\t}"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void bulk_commit_el() { asm volatile(STG_EL_BEGIN "@P_el cp.async.bulk.commit_group;\n\t}" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read_el() { asm volatile(STG_EL_BEGIN "@P_el cp.async.bulk.wait_group.read %0;\n\t}" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all_el() { asm volatile(STG_EL_BEGIN "@P_el cp.async.bulk.wait_group 0;\n\t}" ::: "memory"); }

// ---- programmatic dependent launch (PDL).  A kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may
// start while its predecessor in the stream is still running: its prologue (barrier init, TMEM allocation, tensor-map
// prefetch) overlaps the predecessor's tail.  pdl_wait() blocks until the predecessor grid has COMPLETED and its memory
// is visible - it must precede every global-memory access; pdl_trigger() lets the successor start its own prologue.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---- TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_slot), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]; bf16 inputs, fp32 accumulate, cta_group::1
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 lanes x 16 consecutive fp32 columns: thread i of the warp gets lane (base_lane + i)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// ---- descriptors
// K-major operand tile, rows of 128 B (64 bf16), 128-byte swizzle, 8-row groups 1024 B apart.
__device__ __forceinline__ uint64_t smem_desc_kmajor_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);  // start address
  d |= (uint64_t)1 << 16;                      // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;            // stride byte offset: next 8-row group
  d |= (uint64_t)1 << 46;                      // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                      // SWIZZLE_128B
  return d;
}
// K-major operand tile whose rows are only 32 or 64 bytes long (16 / 32 bf16: the per-group K extent of a grouped
// convolution), TMA-loaded with the matching 32- / 64-byte swizzle; 8-row groups are 8 * row_bytes apart.
__device__ __forceinline__ uint64_t smem_desc_kmajor_narrow(uint32_t smem_addr, int row_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)((8 * row_bytes) >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(row_bytes == 32 ? 6 : (row_bytes == 64 ? 4 : 2)) << 61;   // SWIZZLE_32B / _64B / _128B
  return d;
}
// MN-major operand tile: [k rows][64 mn elements] per 128 B row, 128-byte swizzle.
// lbo = byte distance between 64-element MN groups, sbo = byte distance between 8-row K groups.
__device__ __forceinline__ uint64_t smem_desc_mnmajor_sw128(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// kind::f16 instruction descriptor: bf16 x bf16 -> fp32, M=128, N=n
__device__ __forceinline__ uint32_t idesc_bf16_f32(int m, int n, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

}  // namespace tc

// host: cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda)
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiled get_encode_tiled();
// Launch attribute of the tcgen05 kernels: programmatic dependent launch (see pdl_wait / pdl_trigger).
inline int tc_launch_attrs(cudaLaunchAttribute* at) {
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  return 1;
}
// bf16 tensor, dims[0] contiguous; strides_bytes[i] is the stride of dims[i+1]
int make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box, const uint32_t* elem_strides, int swizzle_bytes = 128);

}  // namespace stg
