// sm_100a primitives written as inline PTX: mbarrier, TMA (cp.async.bulk.tensor), tcgen05
// (alloc / mma / commit / ld), UMMA shared-memory and instruction descriptors.
// Layout facts used below (canonical UMMA layouts, 16-byte units, bf16 -> T = 8 elements):
//   K-major  SWIZZLE_128B: ((8,m),(T,2)) : ((8T,SBO),(1,T))  rows of 128 B, 8-row atoms of 1024 B
//   MN-major SWIZZLE_128B: ((T,8,m),(8,k)) : ((1,T,LBO),(8T,SBO))  k-rows of 128 B (64 MN elements)
// Both are exactly what a TMA box of 64 bf16 (128 B) x rows with CU_TENSOR_MAP_SWIZZLE_128B
// writes, provided the tile base is 1024-byte aligned.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ---------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {   // generic-proxy smem writes -> async proxy (UMMA/TMA)
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Bounded spin: a wrong descriptor must trap, not hang the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t ok = 0;
#pragma unroll 1
  for (uint32_t it = 0; it < 400000000u; ++it) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
    if (ok) return;
  }
  __trap();
}

// Warp-collective wait: all 32 lanes (converged) poll, the loop exit is decided by a vote, so control
// flow stays warp-uniform and the compiler keeps loop state on the uniform datapath (the issue loops of
// the TMA / MMA warps must stay short: one warp issues every tcgen05.mma of the CTA).
__device__ __forceinline__ void mbar_wait_warp(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
#pragma unroll 1
  for (uint32_t it = 0; it < 400000000u; ++it) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
    if (__all_sync(0xffffffffu, ok)) return;
  }
  __trap();
}

// ---- TMA ----------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
// 2-D tile load: c0 = innermost (contiguous) coordinate, c1 = row coordinate.
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// 3-D tile load (MN-major operands: c0 = element inside a 64-wide column group, c1 = contraction row, c2 = column group).
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// ---- tcgen05 ------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {   // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {      // same warp as alloc
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], bf16 x bf16 -> fp32, issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives once every previously issued MMA of this thread has completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// TMEM -> registers: 32 lanes x 32 consecutive fp32 columns; thread i of the warp gets lane
// (base lane + i).  A warp may only touch lanes [32*(warp%4), 32*(warp%4)+32).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- descriptors --------------------------------------------------------------------------
// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout): start>>4 [0,14),
// LBO>>4 [16,30), SBO>>4 [32,46), version=1 [46,48), layout type [61,64) (2 = SWIZZLE_128B).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFFu);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// K-major SW128 tile (rows x 64 bf16, 128 B per row): SBO = 1024 (8-row atoms), LBO unused (=16 B).
// The k-th UMMA_K=16 slice starts 32*k bytes into the row.
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t tile_addr, int k16) {
  return make_smem_desc(tile_addr + 32u * (uint32_t)k16, 16u, 1024u);
}
// MN-major SW128 tile built from boxes of [64 k-rows x 64 mn]: the 8-k-row atom is 1024 B (SBO),
// consecutive 64-wide MN groups are `mn_group_bytes` apart (LBO).  UMMA_K=16 = two atoms = 2048 B.
__device__ __forceinline__ uint64_t desc_mnmajor(uint32_t tile_addr, int k16, uint32_t mn_group_bytes) {
  return make_smem_desc(tile_addr + 2048u * (uint32_t)k16, mn_group_bytes, 1024u);
}
// Instruction descriptor, kind::f16 (cute::UMMA::InstrDescriptor): D fp32 (1<<4), A/B bf16 (1<<7,
// 1<<10), a_major bit 15, b_major bit 16, N>>3 at [17,23), M>>4 at [24,29).
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// the same with fp16 operands (format field 0).  (The two format fields cannot differ: an fp16 x bf16 kind::f16 MMA
// is an illegal instruction on sm_100a.)
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

// byte offset of element (row r, col c) inside a K-major SW128 tile of 64 bf16 columns
__device__ __forceinline__ uint32_t sw128_offset(int r, int c) {
  return (uint32_t)r * 128u + ((((uint32_t)c >> 3) ^ ((uint32_t)r & 7u)) << 4) + (((uint32_t)c & 7u) << 1);
}

}  // namespace tc

// ---- host: tensor maps -------------------------------------------------------------------
// 2-D bf16 row-major matrix [rows, cols] (cols contiguous) -> boxes of [box_rows x 64 cols], 128B swizzle.
// MN-major operand [k_rows, cols] (cols contiguous, row stride a multiple of 64 elements) seen as
// [cols/64 groups][k_rows][64]: ONE box of `groups` column groups x 64 contraction rows per tile and k block lands in
// shared memory as `groups` consecutive [64 x 128 B] SWIZZLE_128B blocks -- a TMA box costs ~120 ns of issue time
// whatever its size (the TMA fill-rate probe, profiles/r1_c3_phases.txt), so one 32 KB box instead of four 8 KB ones.
int vaeb_make_tmap_bf16_mn(CUtensorMap* out, const void* base, uint64_t k_rows, uint64_t cols, uint64_t row_stride_elems,
                           uint32_t groups, uint32_t k_box = 64);
int vaeb_make_tmap_bf16(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t row_stride_elems,
                        uint32_t box_rows);
