// Shared device-side helpers for the sm_100a kernels of speech_b200:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld),
// UMMA shared-memory + instruction descriptors, bounded spin-waits.
//
// Everything here is inline PTX for sm_100a only.  No CUTLASS/CuTe dependency.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

#define SB_DEVINL __device__ __forceinline__

namespace sb {

// ----------------------------------------------------------------------------------------------
// status codes shared with include/speech_b200.h
// ----------------------------------------------------------------------------------------------
enum : int {
  SB_OK = 0,
  SB_ERR_INVALID = 1,
  SB_ERR_CUDA = 2,
  SB_ERR_UNSUPPORTED = 3,
  SB_ERR_WORKSPACE = 4,
};

// host helper (defined in gemm.cu): number of SMs of the current device
int device_sm_count();

// A spin-wait that can never hang the GPU box: after 2^24 polls (a few seconds) the kernel traps.
#define SB_SPIN_LIMIT (1u << 24)

SB_DEVINL uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

SB_DEVINL uint32_t lane_id() {
  uint32_t l;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
  return l;
}

SB_DEVINL bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
SB_DEVINL void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
SB_DEVINL void mbar_fence_init() {
  // make mbarrier.init visible to the async proxy (TMA / tcgen05.commit)
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
SB_DEVINL void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
SB_DEVINL void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
SB_DEVINL bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
SB_DEVINL void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > SB_SPIN_LIMIT) __trap();
  }
}

// ----------------------------------------------------------------------------------------------
// proxy fences
// ----------------------------------------------------------------------------------------------
SB_DEVINL void fence_proxy_async_smem() {
  // generic-proxy st.shared  ->  async-proxy readers (tcgen05.mma, TMA store)
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
SB_DEVINL void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
SB_DEVINL void fence_proxy_async_global() {
  // generic-proxy st.global -> async-proxy (TMA) readers of global memory
  asm volatile("fence.proxy.async.global;" ::: "memory");
}

// ----------------------------------------------------------------------------------------------
// TMA: tiled tensor loads (global -> shared), completion on an mbarrier
// ----------------------------------------------------------------------------------------------
SB_DEVINL void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
SB_DEVINL void tma_load_2d(void* smem_dst, const void* tmap, uint64_t* bar, int32_t c0,
                           int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)),
        "r"(c0), "r"(c1)
      : "memory");
}
SB_DEVINL void tma_load_3d(void* smem_dst, const void* tmap, uint64_t* bar, int32_t c0,
                           int32_t c1, int32_t c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)),
        "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// ----------------------------------------------------------------------------------------------
// tcgen05: tensor memory allocation
// ----------------------------------------------------------------------------------------------
// Must be executed by one full warp.  ncols: power of two in [32, 512].
SB_DEVINL void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
SB_DEVINL void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
SB_DEVINL void tc_fence_before_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
SB_DEVINL void tc_fence_after_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ----------------------------------------------------------------------------------------------
// UMMA descriptors (layout documented in DESIGN.md §GEMM):
//   shared-memory matrix descriptor, K-major, SWIZZLE_128B:
//     bits [0,14)  start address >> 4
//     bits [16,30) leading byte offset >> 4   (unused for swizzled K-major; 1)
//     bits [32,46) stride byte offset  >> 4   (8 rows x 128 B = 1024 B -> 64)
//     bits [46,48) descriptor version = 1 on sm_100
//     bits [61,64) layout type: 2 = SWIZZLE_128B
// ----------------------------------------------------------------------------------------------
SB_DEVINL uint64_t umma_desc_sw128_kmajor(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// Instruction descriptor for kind::f16 with bf16 A/B (both K-major) and fp32 accumulate.
//   [4,6) c_format=1 (F32); [7,10) a_format=1 (BF16); [10,13) b_format=1 (BF16);
//   bit 15 a_major=0 (K); bit 16 b_major=0 (K); [17,23) N>>3; [24,29) M>>4
SB_DEVINL constexpr uint32_t umma_idesc_bf16_f32(uint32_t M, uint32_t N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]^T ; issued by ONE thread.
SB_DEVINL void umma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                            uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Make all previously issued tcgen05.mma of this thread arrive on an mbarrier when they retire.
SB_DEVINL void umma_commit(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
          smem_u32(bar))
      : "memory");
}

// TMEM -> registers: each warp reads its own 32-lane sub-partition, 32 consecutive columns.
SB_DEVINL void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]),
        "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]),
        "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
SB_DEVINL void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
SB_DEVINL void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Byte offset of element (row, 16-byte chunk `c16` in [0,8)) inside a K-major SWIZZLE_128B tile
// whose rows are 128 bytes (64 bf16) wide.  Same layout TMA produces with CU_TENSOR_MAP_SWIZZLE_128B
// (tile base must be 1024-byte aligned).
SB_DEVINL uint32_t sw128_offset(uint32_t row, uint32_t c16) {
  return (row >> 3) * 1024u + (row & 7u) * 128u + ((c16 ^ (row & 7u)) << 4);
}

// ----------------------------------------------------------------------------------------------
// global-memory helpers for cross-CTA exchange inside a persistent kernel
// ----------------------------------------------------------------------------------------------
SB_DEVINL void red_release_gpu_add(unsigned int* p, unsigned int v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
SB_DEVINL unsigned int ld_acquire_gpu(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
SB_DEVINL uint4 ld_cg_u4(const void* p) {
  uint4 v;
  asm volatile("ld.global.cg.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p)
               : "memory");
  return v;
}
SB_DEVINL float4 ld_cg_f4(const void* p) {
  float4 v;
  asm volatile("ld.global.cg.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p)
               : "memory");
  return v;
}
SB_DEVINL float ld_cg_f(const void* p) {
  float v;
  asm volatile("ld.global.cg.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
  return v;
}

SB_DEVINL float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
SB_DEVINL float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

SB_DEVINL uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}

}  // namespace sb
