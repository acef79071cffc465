// tcgen05 / TMEM / TMA / mbarrier PTX wrappers shared by the sm_100a tensor-core kernels (vit_gemm.cu, vit_attention_tc.cu).
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
// try_wait with a suspend-time hint: the waiting warp is parked until the phase completes (or the hint expires) instead of re-issuing
// the test in a tight loop.  Without the hint the spinning issuer / producer warps of the attention kernels took a large share of
// the issue slots of their SM sub-partitions (ncu: a quarter of all executed instructions were try_wait + branch) and slowed the
// warps doing arithmetic on the same sub-partition.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n\t"
      "@P1 bra DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "DONE:\n\t"
      "}" ::"r"(bar),
      "r"(parity), "r"(0x989680u)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
               "l"(map), "r"(bar), "r"(c0), "r"(c1)
               : "memory");
}
// TMA prefetch of a tile into L2 (no shared-memory destination, no barrier)
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* map, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(map), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128B-swizzled operand tile: rows of 128 bytes, 8-row groups 1024 bytes apart (SBO), LBO unused (=1).
// Bits: [0,14) start>>4, [16,30) LBO>>4, [32,46) SBO>>4, [46,48) version=1 (Blackwell), [61,64) layout (2 = SWIZZLE_128B).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor, kind::f16: D fp32 (bit 4), A/B bf16 (bits 7, 10), A K-major, B K-major or MN-major (bit 16),
// N>>3 at bit 17, M>>4 at bit 24.
__host__ __device__ constexpr uint32_t idesc_bf16(int m, int n, bool b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (b_mn_major ? (1u << 16) : 0u) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}


__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

}  // namespace tc

// host: cached cuTensorMapEncodeTiled for a [rows, cols] bf16 row-major matrix (leading dimension ld elements), box = 64
// columns x box_rows rows, 128-byte swizzle (defined in vit_gemm.cu)
int cg_make_tensor_map_bf16(CUtensorMap* out, const void* ptr, long long rows, long long cols, long long ld, int box_rows);
// host: multiprocessor count of the current device, cached per device (defined in vit_gemm.cu); sizes the persistent grids
int cg_num_sms();

// host: the tcgen05 attention kernels (vit_attention_tc.cu) keep all operands of an (image, head) item in shared memory, which holds
// sequences up to this length; cg_attention_fwd / _bwd run longer ones on the mma.sync kernels of vit_attention.cu
constexpr int ATTN_TC_MAX_T = 272;
int cg_attention_fwd_tc(const void* qkv, int Nimg, int T, int heads, void* ctx, float* lse, cudaStream_t s);
int cg_attention_bwd_tc(const void* qkv, const void* ctx, const void* dctx, const float* lse, int Nimg, int T, int heads, void* dqkv, cudaStream_t s);
