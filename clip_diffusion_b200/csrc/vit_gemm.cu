// bf16 GEMM for the CLIP ViT (QKV / out-proj / MLP / patch-embed and their dgrads) on the 5th-gen tensor
// cores of sm_100a:  acc[M,N] = A[M,K] . B[N,K]^T,  fp32 accumulation in TMEM, fused epilogues.
//
//   * operands staged by TMA (cp.async.bulk.tensor, 128B swizzle) into a 4-stage shared-memory ring;
//   * one elected thread issues tcgen05.mma (cta_group::1, M=128, N=BN, K=16 per instruction);
//   * the accumulator lives in TMEM and is double buffered (2 x BN columns), so the epilogue of tile i
//     overlaps the main loop of tile i+1;
//   * persistent: one CTA per SM walks the tile list (tile = blockIdx.x + i*gridDim.x), consecutive
//     tiles share the A row-block so it is reused out of L2;
//   * warp roles: 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocator, 4..11 = epilogue (tcgen05.ld ->
//     registers -> bias / QuickGELU / residual -> global).  Eight epilogue warps = two per scheduler and per
//     TMEM lane quarter (each takes half of the tile's columns): one warp per scheduler cannot hide its own ALU
//     latency and made the QuickGELU epilogues 2-3x slower than the main loop (profiles/r01_*).
//
// Weights are frozen (models.py:71), so every GEMM of the backward pass is a dgrad with a pre-transposed
// weight copy: all calls have both operands K-major and share this one kernel.
#include <cuda.h>
#include <stdlib.h>
#include <mutex>
#include <unordered_map>
#include "common.cuh"
#include "tcgen05.cuh"

namespace {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 bf16 = 128 bytes = one swizzle atom row
constexpr int STAGES = 4;
constexpr int NUM_EPI_WARPS = 8;
constexpr int NUM_THREADS = 128 + 32 * NUM_EPI_WARPS;

struct GemmArgs {
  int M, N, K;
  const float* bias;
  void* out;
  void* aux;
  long long ldo;
  const float* pos;
  int g2;
  int wide;  // rows of out / aux are 32-byte aligned: the epilogue may use 256-bit global accesses
};

using namespace tc;

// Instruction descriptor for kind::f16: D fp32, A/B bf16, both K-major, M=128, N=BN.
__host__ __device__ constexpr uint32_t make_idesc(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

// sigmoid(1.702 u) = 0.5 * tanh(0.851 u) + 0.5 : one MUFU op instead of ex2 + a full-precision division
__device__ __forceinline__ float sigmoid_1702(float u) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.851f * u));
  return fmaf(0.5f, t, 0.5f);
}
__device__ __forceinline__ float qgelu(float u) { return u * sigmoid_1702(u); }
__device__ __forceinline__ float qgelu_grad(float u) {
  const float s = sigmoid_1702(u);
  return s * fmaf(1.702f * u, 1.f - s, 1.f);
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

// 256-bit global accesses (sm_100: LDG/STG.E.ENL2.256).  In the epilogue a THREAD owns a row (tcgen05.ld 32x32b layout), so a warp
// instruction touches 32 different rows: with 16-byte accesses every 32-byte sector is written in two half-sector transactions; with
// 32-byte accesses each lane fills whole sectors and the number of LSU/L2 transactions halves (the bf16 epilogues were store-path
// bound: 2 TB/s of DRAM traffic at 53 % of the tensor peak).  Needs 32-byte aligned rows: g.wide is set by the host when they are.
__device__ __forceinline__ void st256(void* p, const uint32_t* w) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]),
               "r"(w[6]), "r"(w[7])
               : "memory");
}
__device__ __forceinline__ void ld256(const void* p, uint32_t* w) {
  asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7])
               : "l"(p)
               : "memory");
}
// 32 consecutive fp32 / bf16 values of one row
__device__ __forceinline__ void store_f32x32(float* dst, const float* v, bool wide) {
  if (wide) {
#pragma unroll
    for (int j = 0; j < 4; ++j) st256(dst + 8 * j, reinterpret_cast<const uint32_t*>(v + 8 * j));
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) reinterpret_cast<float4*>(dst)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
  }
}
__device__ __forceinline__ void load_f32x32(const float* src, float* r, bool wide) {
  if (wide) {
#pragma unroll
    for (int j = 0; j < 4; ++j) ld256(src + 8 * j, reinterpret_cast<uint32_t*>(r + 8 * j));
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 p = reinterpret_cast<const float4*>(src)[j];
      r[4 * j] = p.x; r[4 * j + 1] = p.y; r[4 * j + 2] = p.z; r[4 * j + 3] = p.w;
    }
  }
}
__device__ __forceinline__ void store_bf16x32(__nv_bfloat16* dst, const float* v, bool wide) {
  uint32_t w[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) w[j] = pack_bf16(v[2 * j], v[2 * j + 1]);
  if (wide) {
    st256(dst, w);
    st256(dst + 16, w + 8);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) reinterpret_cast<uint4*>(dst)[j] = make_uint4(w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
  }
}
__device__ __forceinline__ void load_bf16x32(const __nv_bfloat16* src, uint32_t* w, bool wide) {
  if (wide) {
    ld256(src, w);
    ld256(src + 16, w + 8);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint4 a = __ldg(reinterpret_cast<const uint4*>(src) + j);
      w[4 * j] = a.x; w[4 * j + 1] = a.y; w[4 * j + 2] = a.z; w[4 * j + 3] = a.w;
    }
  }
}

// one 32-column chunk of one output row
template <int EPI>
__device__ __forceinline__ void epilogue_chunk(const GemmArgs& g, long long row, long long orow, int col, const uint32_t* acc_u) {
  const bool wide = g.wide != 0;
  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(acc_u[j]);
  if (EPI == CG_EPI_BIAS_BF16 || EPI == CG_EPI_BIAS_RESID_F32 || EPI == CG_EPI_BIAS_QGELU_BF16) {
    const float4* b4 = reinterpret_cast<const float4*>(g.bias + col);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 b = __ldg(b4 + j);
      v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
    }
  }
  if (EPI == CG_EPI_BIAS_RESID_F32 || EPI == CG_EPI_F32 || EPI == CG_EPI_PATCH_POS_F32) {
    float* o = reinterpret_cast<float*>(g.out) + orow * g.ldo + col;
    if (EPI == CG_EPI_PATCH_POS_F32) {
      const float4* p4 = reinterpret_cast<const float4*>(g.pos + (1 + row % g.g2) * (long long)g.N + col);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 p = __ldg(p4 + j);
        v[4 * j] += p.x; v[4 * j + 1] += p.y; v[4 * j + 2] += p.z; v[4 * j + 3] += p.w;
      }
    } else if (EPI == CG_EPI_BIAS_RESID_F32) {
      float r[32];
      load_f32x32(reinterpret_cast<const float*>(g.aux) + orow * g.ldo + col, r, wide);
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] += r[j];
    }
    store_f32x32(o, v, wide);
  } else {
    __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(g.out) + orow * g.ldo + col;
    if (EPI == CG_EPI_BIAS_QGELU_BF16) {
      store_bf16x32(reinterpret_cast<__nv_bfloat16*>(g.aux) + orow * g.ldo + col, v, wide);  // pre-activation for the backward
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = qgelu(v[j]);
    } else if (EPI == CG_EPI_DQGELU_BF16) {
      uint32_t w[16];
      load_bf16x32(reinterpret_cast<const __nv_bfloat16*>(g.aux) + orow * g.ldo + col, w, wide);
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const __nv_bfloat162 p = *reinterpret_cast<const __nv_bfloat162*>(&w[j]);
        v[2 * j] *= qgelu_grad(__low2float(p));
        v[2 * j + 1] *= qgelu_grad(__high2float(p));
      }
    }
    store_bf16x32(o, v, wide);
  }
}

template <int BN, int EPI>
__global__ void __launch_bounds__(NUM_THREADS, 1) gemm_bf16_tn_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                       const __grid_constant__ CUtensorMap tmB, const GemmArgs g) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr uint32_t A_BYTES = BM * BK * 2;
  constexpr uint32_t B_BYTES = BN * BK * 2;
  constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr uint32_t TMEM_COLS = 2 * BN;  // 256 or 512: power of two >= 32

  // 1024-byte alignment for the 128B swizzle
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + STAGES * STAGE_BYTES;
  // barriers: full[STAGES], empty[STAGES], tmem_full[2], tmem_empty[2]; then the TMEM base address word
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + 2 + s); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 4);

  cg_griddep_launch();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tiles = (g.M + BM - 1) / BM, n_tiles = g.N / BN;
  const int num_tiles = m_tiles * n_tiles;
  const int k_blocks = g.K / BK;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), NUM_EPI_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  cg_griddep_wait();  // prologue done: from here on the predecessor's output is read (and buffers it may still read are written)
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");

  if (warp == 0) {
    // ================= TMA producer =================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        const int m_blk = t / n_tiles, n_blk = t - m_blk * n_tiles;
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t a_dst = smem_base + stage * STAGE_BYTES, b_dst = a_dst + A_BYTES;
          mbar_arrive_expect_tx(full_bar(stage), STAGE_BYTES);
          tma_load_2d(a_dst, &tmA, full_bar(stage), kb * BK, m_blk * BM);
          tma_load_2d(b_dst, &tmB, full_bar(stage), kb * BK, n_blk * BN);
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(BN);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
        const int as = it & 1;
        const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
        mbar_wait(tempty_bar(as), aphase ^ 1u);  // epilogue has drained this accumulator
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tcgen05_fence_after();
          const uint32_t a_addr = smem_base + stage * STAGE_BYTES, b_addr = a_addr + A_BYTES;
          const uint64_t adesc = make_smem_desc(a_addr), bdesc = make_smem_desc(b_addr);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // advance 16 elements = 32 bytes along K inside the swizzle atom: +2 in the (addr >> 4) field
            umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit(empty_bar(stage));  // smem slot free once these MMAs have read it
          if (kb == k_blocks - 1) umma_commit(tfull_bar(as));
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp >= 4) {
    // ================= epilogue =================
    const int q = warp & 3;             // TMEM lane quarter this warp may touch (warp id % 4)
    const int chalf = (warp - 4) >> 2;  // which half of the tile's columns this warp drains
    int it = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
      const int m_blk = t / n_tiles, n_blk = t - m_blk * n_tiles;
      const int as = it & 1;
      const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
      mbar_wait(tfull_bar(as), aphase);
      tcgen05_fence_after();
      const long long row = (long long)m_blk * BM + q * 32 + lane;
      long long orow = row;
      if (EPI == CG_EPI_PATCH_POS_F32) orow = (row / g.g2) * (g.g2 + 1) + 1 + row % g.g2;
      const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN);
#pragma unroll 1
      for (int c = chalf * (BN / 2); c < (chalf + 1) * (BN / 2); c += 32) {
        uint32_t acc[32];
        tmem_ld32(t_row + (uint32_t)c, acc);
        tmem_ld_wait();
        if (row < g.M) epilogue_chunk<EPI>(g, row, orow, n_blk * BN + c, acc);
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(as));
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ---------------------------------------------------------------------------------- CTA-pair variant
// cta_group::2: two CTAs of one cluster (one TPC) share a 256x256 output tile.  Each CTA stages ITS 128 rows of A and
// HALF of the B tile (128 of the 256 output columns); the leader CTA issues tcgen05.mma.cta_group::2 (M=256), which
// reads both halves of B from both SMs' shared memory, so per 64-deep k-block the pair pulls 64 KB from L2 instead of
// 2 x 48 KB -- the single-CTA kernel is L2->smem bound at ~1.0-1.15 PFLOP/s (profiles/).  6-stage ring (32 KB/stage).
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_smem_addr, uint32_t cta) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(cta));
  return r;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t leader_bar_cluster_addr, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(map), "r"(leader_bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

constexpr int STAGES2 = 6;
constexpr int BN2 = 256;

template <int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
    gemm_bf16_tn_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmArgs g) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr uint32_t A_BYTES = BM * BK * 2;         // this CTA's 128 rows of A
  constexpr uint32_t B_BYTES = (BN2 / 2) * BK * 2;  // this CTA's half of the B tile
  constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr uint32_t TMEM_COLS = 2 * BN2;

  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + STAGES2 * STAGE_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES2 + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * STAGES2 + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * STAGES2 + 2 + s); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES2 + 4);

  cg_griddep_launch();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int m_tiles = (g.M + 2 * BM - 1) / (2 * BM), n_tiles = g.N / BN2;
  const int num_tiles = m_tiles * n_tiles;
  const int k_blocks = g.K / BK;
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES2; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 2 * NUM_EPI_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  cg_griddep_wait();
  tcgen05_fence_before();
  cluster_sync_all();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");

  if (warp == 0) {
    // ================= TMA producer (both CTAs): data into OWN smem, bytes reported to the LEADER's full barrier
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = cluster_id; t < num_tiles; t += num_clusters) {
        const int m_blk = t / n_tiles, n_blk = t - m_blk * n_tiles;
        const int m0 = m_blk * 2 * BM + (int)rank * BM;
        const int n0 = n_blk * BN2 + (int)rank * (BN2 / 2);
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t a_dst = smem_base + stage * STAGE_BYTES, b_dst = a_dst + A_BYTES;
          if (leader) mbar_arrive_expect_tx(full_bar(stage), 2 * STAGE_BYTES);
          const uint32_t lead_bar = map_to_cta(full_bar(stage), 0);
          tma_load_2d_pair(a_dst, &tmA, lead_bar, kb * BK, m0);
          tma_load_2d_pair(b_dst, &tmB, lead_bar, kb * BK, n0);
          if (++stage == STAGES2) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer (leader CTA only)
    if (leader && lane == 0) {
      constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN2 >> 3) << 17) | ((uint32_t)((2 * BM) >> 4) << 24);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int t = cluster_id; t < num_tiles; t += num_clusters, ++it) {
        const int as = it & 1;
        const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
        mbar_wait(tempty_bar(as), aphase ^ 1u);  // both CTAs' epilogues have drained this accumulator
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN2);
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tcgen05_fence_after();
          const uint32_t a_addr = smem_base + stage * STAGE_BYTES, b_addr = a_addr + A_BYTES;
          const uint64_t adesc = make_smem_desc(a_addr), bdesc = make_smem_desc(b_addr);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k)
            umma_bf16_pair(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit_pair(empty_bar(stage));  // frees the slot in BOTH CTAs
          if (kb == k_blocks - 1) umma_commit_pair(tfull_bar(as));
          if (++stage == STAGES2) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp >= 4) {
    // ================= epilogue (both CTAs, own 128 rows)
    const int q = warp & 3;
    const int chalf = (warp - 4) >> 2;
    int it = 0;
    for (int t = cluster_id; t < num_tiles; t += num_clusters, ++it) {
      const int m_blk = t / n_tiles, n_blk = t - m_blk * n_tiles;
      const int as = it & 1;
      const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
      mbar_wait(tfull_bar(as), aphase);
      tcgen05_fence_after();
      const long long row = (long long)m_blk * 2 * BM + (long long)rank * BM + q * 32 + lane;
      long long orow = row;
      if (EPI == CG_EPI_PATCH_POS_F32) orow = (row / g.g2) * (g.g2 + 1) + 1 + row % g.g2;
      const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN2);
#pragma unroll 1
      for (int c = chalf * (BN2 / 2); c < (chalf + 1) * (BN2 / 2); c += 32) {
        uint32_t acc[32];
        tmem_ld32(t_row + (uint32_t)c, acc);
        tmem_ld_wait();
        if (row < g.M) epilogue_chunk<EPI>(g, row, orow, n_blk * BN2 + c, acc);
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(map_to_cta(tempty_bar(as), 0));
    }
  }
  tcgen05_fence_before();
  cluster_sync_all();  // nobody leaves (or frees TMEM) while the peer may still read this CTA's shared memory
  if (warp == 2) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ---------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

struct MapKey {
  const void* ptr;
  long long rows, cols, ld;
  int box_rows;
  bool operator==(const MapKey& o) const { return ptr == o.ptr && rows == o.rows && cols == o.cols && ld == o.ld && box_rows == o.box_rows; }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    size_t h = std::hash<const void*>()(k.ptr);
    h ^= std::hash<long long>()(k.rows * 1315423911LL + k.cols * 2654435761LL + k.ld * 97LL + k.box_rows) + 0x9e3779b97f4a7c15ULL + (h << 6) + (h >> 2);
    return h;
  }
};

}  // namespace

// [rows, cols] bf16 row-major with leading dimension ld; box = 64 columns x box_rows rows, 128B swizzle.
int cg_make_tensor_map_bf16(CUtensorMap* out, const void* ptr, long long rows, long long cols, long long ld, int box_rows) {
  static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> cache;
  static std::mutex mu;
  const MapKey key = {ptr, rows, cols, ld, box_rows};
  {
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(key);
    if (it != cache.end()) { *out = it->second; return 0; }
  }
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) { cg_set_error("cuTensorMapEncodeTiled is not available from the driver"); return CG_EARCH; }
  const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)ld * 2};
  const cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { cg_set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld cols=%lld ld=%lld)", (int)r, rows, cols, ld); return CG_EINVAL; }
  std::lock_guard<std::mutex> lk(mu);
  if (cache.size() > 4096) cache.clear();
  cache[key] = *out;
  return 0;
}

int cg_num_sms() {
  static int per_device[CG_MAX_DEVICES] = {};
  const int dev = cg_device_index();
  if (per_device[dev] == 0) {
    int n = 0;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    per_device[dev] = n > 0 ? n : CG_NUM_SMS;
  }
  return per_device[dev];
}

namespace {

template <int BN, int EPI>
int launch(const CUtensorMap& ta, const CUtensorMap& tb, const GemmArgs& g, cudaStream_t s) {
  constexpr size_t smem = (size_t)STAGES * (BM * BK * 2 + BN * BK * 2) + 1024 /*align slack*/ + 256 /*barriers*/;
  static bool configured[CG_MAX_DEVICES] = {};  // function attributes are per device
  const int dev = cg_device_index();
  if (!configured[dev]) {
    CG_CUDA(cudaFuncSetAttribute(gemm_bf16_tn_kernel<BN, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured[dev] = true;
  }
  const int tiles = ((g.M + BM - 1) / BM) * (g.N / BN);
  const int grid = tiles < cg_num_sms() ? tiles : cg_num_sms();
  CG_CUDA(cg_launch_pdl(gemm_bf16_tn_kernel<BN, EPI>, dim3(grid), dim3(NUM_THREADS), smem, s, ta, tb, g));
  return 0;
}

template <int BN>
int dispatch(int epi, const CUtensorMap& ta, const CUtensorMap& tb, const GemmArgs& g, cudaStream_t s) {
  switch (epi) {
    case CG_EPI_BIAS_BF16: return launch<BN, CG_EPI_BIAS_BF16>(ta, tb, g, s);
    case CG_EPI_BIAS_RESID_F32: return launch<BN, CG_EPI_BIAS_RESID_F32>(ta, tb, g, s);
    case CG_EPI_BIAS_QGELU_BF16: return launch<BN, CG_EPI_BIAS_QGELU_BF16>(ta, tb, g, s);
    case CG_EPI_DQGELU_BF16: return launch<BN, CG_EPI_DQGELU_BF16>(ta, tb, g, s);
    case CG_EPI_F32: return launch<BN, CG_EPI_F32>(ta, tb, g, s);
    case CG_EPI_BF16: return launch<BN, CG_EPI_BF16>(ta, tb, g, s);
    case CG_EPI_PATCH_POS_F32: return launch<BN, CG_EPI_PATCH_POS_F32>(ta, tb, g, s);
  }
  cg_set_error("cg_gemm_bf16_tn: unknown epilogue %d", epi);
  return CG_EINVAL;
}

template <int EPI>
int launch_pair(const CUtensorMap& ta, const CUtensorMap& tb, const GemmArgs& g, cudaStream_t s) {
  constexpr size_t smem = (size_t)STAGES2 * (BM * BK * 2 + (BN2 / 2) * BK * 2) + 1024 + 256;
  static bool configured[CG_MAX_DEVICES] = {};
  const int dev = cg_device_index();
  if (!configured[dev]) {
    CG_CUDA(cudaFuncSetAttribute(gemm_bf16_tn_pair_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured[dev] = true;
  }
  const int tiles = ((g.M + 2 * BM - 1) / (2 * BM)) * (g.N / BN2);
  int clusters = cg_num_sms() / 2;
  if (tiles < clusters) clusters = tiles;
  CG_CUDA(cg_launch_pdl(gemm_bf16_tn_pair_kernel<EPI>, dim3(2 * clusters), dim3(NUM_THREADS), smem, s, ta, tb, g));
  return 0;
}

int dispatch_pair(int epi, const CUtensorMap& ta, const CUtensorMap& tb, const GemmArgs& g, cudaStream_t s) {
  switch (epi) {
    case CG_EPI_BIAS_BF16: return launch_pair<CG_EPI_BIAS_BF16>(ta, tb, g, s);
    case CG_EPI_BIAS_RESID_F32: return launch_pair<CG_EPI_BIAS_RESID_F32>(ta, tb, g, s);
    case CG_EPI_BIAS_QGELU_BF16: return launch_pair<CG_EPI_BIAS_QGELU_BF16>(ta, tb, g, s);
    case CG_EPI_DQGELU_BF16: return launch_pair<CG_EPI_DQGELU_BF16>(ta, tb, g, s);
    case CG_EPI_F32: return launch_pair<CG_EPI_F32>(ta, tb, g, s);
    case CG_EPI_BF16: return launch_pair<CG_EPI_BF16>(ta, tb, g, s);
    case CG_EPI_PATCH_POS_F32: return launch_pair<CG_EPI_PATCH_POS_F32>(ta, tb, g, s);
  }
  cg_set_error("cg_gemm_bf16_tn: unknown epilogue %d", epi);
  return CG_EINVAL;
}

// (pair kernel, ViT-L/14 x 64: +16% on K=4096 fp32-out GEMMs, +3..7% on bias/bf16 epilogues, -2% on the QuickGELU epilogues which
// are epilogue-bound; 256x256 tiles lose when they quantise badly, e.g. 75 tiles on 74 clusters)
// Tile shape per problem.  The kernels are persistent (one CTA or CTA pair per SM walks the tile list), so the cost of a shape is
// waves x columns-per-tile: ceil(tiles / slots) x BN, with the measured per-shape efficiency (B200, tools/bench_gemm_shapes.py ->
// profiles/r02_gemm_tile_selection.txt):
//   128 x 256 single CTA   the default: L2 -> smem bound at ~1.0-1.15 PFLOP/s
//   128 x 128 single CTA   half the columns per tile => half the quantisation step (M = 6304, N = 768: 150 tiles = 2 waves of 256
//                          columns become 300 tiles = 3 waves of 128; M = 2056 per rank at 8-way strong scaling: 68 -> 136 tiles on
//                          148 SMs), but each CTA re-reads the A tile for half the work: ~0.85 of the 256-column efficiency
//   256 x 256 CTA pair     each CTA stages half of B: lifts the L2 bound when K is long (>= 1024) and the epilogue is cheap
// CG_GEMM_PAIR=0/1 and CG_GEMM_BN=128/256 force a variant (A/B measurements).
int env_choice(const char* name) {
  const char* e = getenv(name);
  return e ? atoi(e) : -1;
}
enum { TILE_256 = 0, TILE_128 = 1, TILE_PAIR = 2 };
int choose_tile(int M, int N, int K, int epilogue) {
  static const int force_pair = env_choice("CG_GEMM_PAIR"), force_bn = env_choice("CG_GEMM_BN");
  const bool can256 = N % 256 == 0;
  const bool can_pair = can256 && M > 2 * BM;
  if (!can256 || force_bn == 128) return TILE_128;
  if (force_pair == 1 && can_pair) return TILE_PAIR;
  const int sms = cg_num_sms();
  const long long mt = (M + BM - 1) / BM, mt2 = (M + 2 * BM - 1) / (2 * BM);
  auto waves = [](long long tiles, long long slots) { return (double)((tiles + slots - 1) / slots); };
  const double c256 = waves(mt * (N / 256), sms) * 256.0;
  const double c128 = waves(mt * (N / 128), sms) * 128.0 / (K > 1024 ? 0.75 : 0.85);  // the A tile is re-read for half the work: worse with long K
  const bool heavy_epi = epilogue == CG_EPI_BIAS_QGELU_BF16 || epilogue == CG_EPI_DQGELU_BF16;
  // a pair tile is two CTAs' worth of rows: per-SM cost = waves x 256 columns, ~10 % faster per tile when K is long
  const double cpair = (can_pair && force_pair != 0 && !heavy_epi && K >= 1024) ? waves(mt2 * (N / BN2), sms / 2) * 256.0 / (K >= 2048 ? 1.10 : 1.02) : 1e30;
  if (force_bn == 256) return cpair < c256 ? TILE_PAIR : TILE_256;
  if (cpair <= c256 && cpair <= c128) return TILE_PAIR;
  return c128 < c256 ? TILE_128 : TILE_256;
}

}  // namespace

extern "C" int cg_gemm_bf16_tn(const void* A, const void* B, int M, int N, int K, int64_t lda, int64_t ldb, int epilogue, const float* bias,
                               void* out, void* aux, int64_t ldo, const float* pos, int g2, void* stream) {
  CG_REQUIRE(A && B && out, "cg_gemm_bf16_tn: null operand");
  CG_REQUIRE(M > 0 && N > 0 && K > 0, "cg_gemm_bf16_tn: bad sizes M=%d N=%d K=%d", M, N, K);
  CG_REQUIRE(K % BK == 0, "cg_gemm_bf16_tn: K=%d must be a multiple of %d", K, BK);
  CG_REQUIRE(N % 128 == 0, "cg_gemm_bf16_tn: N=%d must be a multiple of 128", N);
  CG_REQUIRE(lda % 8 == 0 && ldb % 8 == 0 && lda >= K && ldb >= K, "cg_gemm_bf16_tn: leading dimensions must be >= K and multiples of 8");
  CG_REQUIRE(((uintptr_t)A & 15) == 0 && ((uintptr_t)B & 15) == 0 && ((uintptr_t)out & 15) == 0, "cg_gemm_bf16_tn: pointers must be 16-byte aligned");
  CG_REQUIRE(ldo % 8 == 0 && ldo >= N, "cg_gemm_bf16_tn: ldo=%lld must be >= N and a multiple of 8", (long long)ldo);
  const bool needs_bias = epilogue == CG_EPI_BIAS_BF16 || epilogue == CG_EPI_BIAS_RESID_F32 || epilogue == CG_EPI_BIAS_QGELU_BF16;
  CG_REQUIRE(!needs_bias || bias, "cg_gemm_bf16_tn: epilogue %d needs a bias", epilogue);
  CG_REQUIRE((epilogue != CG_EPI_BIAS_QGELU_BF16 && epilogue != CG_EPI_DQGELU_BF16 && epilogue != CG_EPI_BIAS_RESID_F32) || aux, "cg_gemm_bf16_tn: epilogue %d needs aux", epilogue);
  CG_REQUIRE(epilogue != CG_EPI_PATCH_POS_F32 || (pos && g2 > 0 && M % g2 == 0), "cg_gemm_bf16_tn: patch epilogue needs pos and g2 | M");
  // 256-bit epilogue accesses: every row start of out (and aux) must be 32-byte aligned.  Element size: fp32 outputs 4, bf16 2;
  // aux is fp32 for the residual epilogue, bf16 for the QuickGELU ones.  CG_GEMM_WIDE=0 forces the 128-bit path.
  static int wide_env = -1;
  if (wide_env < 0) {
    const char* e = getenv("CG_GEMM_WIDE");
    wide_env = (e && atoi(e) == 0) ? 0 : 1;
  }
  const bool out_f32 = epilogue == CG_EPI_BIAS_RESID_F32 || epilogue == CG_EPI_F32 || epilogue == CG_EPI_PATCH_POS_F32;
  const long long row_bytes = (long long)ldo * (out_f32 ? 4 : 2);
  const long long aux_row_bytes = (long long)ldo * (epilogue == CG_EPI_BIAS_RESID_F32 ? 4 : 2);
  const int wide = (wide_env && epilogue != CG_EPI_PATCH_POS_F32 && ((uintptr_t)out & 31) == 0 && row_bytes % 32 == 0 &&
                    (!aux || (((uintptr_t)aux & 31) == 0 && aux_row_bytes % 32 == 0)))
                       ? 1
                       : 0;
  const int tile = choose_tile(M, N, K, epilogue);
  CUtensorMap ta, tb;
  int rc = cg_make_tensor_map_bf16(&ta, A, M, K, lda, BM);
  if (rc) return rc;
  if (tile == TILE_PAIR) {
    rc = cg_make_tensor_map_bf16(&tb, B, N, K, ldb, BN2 / 2);
    if (rc) return rc;
    GemmArgs gp = {M, N, K, bias, out, aux, (long long)ldo, pos, g2, wide};
    return dispatch_pair(epilogue, ta, tb, gp, cg_stream(stream));
  }
  const int bn = tile == TILE_256 ? 256 : 128;
  rc = cg_make_tensor_map_bf16(&tb, B, N, K, ldb, bn);
  if (rc) return rc;
  GemmArgs g = {M, N, K, bias, out, aux, (long long)ldo, pos, g2, wide};
  cudaStream_t s = cg_stream(stream);
  return bn == 256 ? dispatch<256>(epilogue, ta, tb, g, s) : dispatch<128>(epilogue, ta, tb, g, s);
}
