// Fused multi-head self-attention of the CLIP ViT on the 5th-gen tensor cores (tcgen05 + TMEM + TMA), forward AND
// backward, for the short sequences of the 224-pixel towers (T <= ATTN_TC_MAX_T = 272: ViT-B/32 T=50, ViT-B/16 T=197, ViT-L/14
// T=257); cg_attention_fwd / _bwd (vit_attention.cu) run every such T here.  The causal forward is the text transformer's attention.
// Replaces nn.MultiheadAttention inside clip_model.encode_image (clip_diffusion/utils/functional.py:97-102) and its
// autograd backward (sample.py:199-214).  Scores never leave the SM.
//
// Both kernels are PERSISTENT: one CTA per SM walks the (image, head) items, and the block stream -- S / dP blocks of 128 rows x 64
// columns in multi-buffered TMEM, bf16 P / dS tiles in shared-memory staging buffers, accumulators in TMEM -- runs ACROSS items, so
// an item's epilogue, the TMEM hand-over and the operand reload overlap the next item's MMAs.  Operands are loaded once per item
// by TMA into 128B-swizzled shared memory (Q, K, V(, dO); <= 272 x 64 bf16 each), one mbarrier per 64-row block; the next item's
// tiles are pulled into L2 by a TMA prefetch while the current item runs.  Roles (16 warps):
//
//   MMA issuers (warp-converged loops, elect.sync lane; with head_dim 64 a single issuing thread was the bottleneck)
//       forward   warps 0 / 1: S = Q K^T of the even / odd blocks    warp 2: O += P V    warp 3: TMA producer
//       backward  warp 0: S (S^T)   warp 1: dP (dP^T)   warp 2: dQ | dV   warp 3: dK + TMA producer
//   softmax   warps 4-7 / 8-11: two warpgroups, block g goes to warpgroup g & 1; a thread owns one row (= one TMEM lane): tcgen05.ld,
//             exp2 / dS arithmetic in registers, bf16 result written to the staging buffer in the K-major 128B-swizzled operand
//             layout; the forward reads each S block from TMEM twice to stay inside 128 registers (a spill costs an L2 round trip
//             here: shared memory leaves ~28 KB of L1)
//   epilogue  warps 12-15: finished accumulators -> bf16 -> HBM; the backward's per-token constants (-lse log2e, delta = rowsum(dO O)
//             computed here from the two global tensors, one item ahead); the edge token
//
//   forward   ONE pass, online softmax without a row-maximum pre-pass: each warpgroup keeps its own reference maximum and row sum
//             and accumulates ITS blocks into ITS OWN O accumulator; the reference only moves when a block exceeds it by 2^8 (then
//             the accumulator is rescaled in TMEM: tcgen05.ld / tcgen05.st); the epilogue merges the partial results.
//   backward  phase A (lane = query):  S = Q K^T, dP = dO V^T, dS = P (dP - delta) scale, dQ += dS K
//             phase B (lane = key):    S^T = K Q^T, dP^T = V dO^T, dV += P^T dO, dK += dS^T Q
//             P is recomputed from the saved log-sum-exp; two orientations instead of a transposed smem operand, no atomics,
//             deterministic.  Rows / columns beyond T are masked (tail block only) or never stored.
//
// Edge token (non-causal kernels).  T = 64 m + 1 (ViT-L/14: 16 x 16 patches + class token = 257) would leave the pipeline with a
// 1-row tile and a 1-column block per tile, each costing a full S -> softmax -> MMA round trip (25-30% of an item).  The LAST token
// is therefore kept out of the pipeline, which then sees only full tiles and blocks: its row and column of the score matrix are
// matrix-vector products, done by the epilogue warps with warp-level m16n8k16 MMAs on the TMA-written tiles (ldmatrix), and folded
// in when a tile is written
// (forward: a third partial result of the online-softmax merge; backward: rank-1 corrections dQ_i += dS_ie K_e, dK_j += dS_ej Q_e,
// dV_j += p_ej dO_e, plus the three reductions that give row e of dQ, dK, dV).
//
// All smem / TMEM operand forms are the ones vit_gemm.cu validated: K-major SW128 A and B, MN-major SW128 B with N = 64.  Every
// mbarrier waiter sees every phase of its barrier (a parity wait is only sound then): warps without real rows still arrive in
// step, no consumer skips a use of a shared buffer, and the issuers observe all operand barriers of every item.
//
// Measured on B200 (profiles/r02_kernel_rooflines.txt, r02_ncu_vit_kernels_digest.txt, time lines with `make trace` +
// tools/trace_attn.py), T = 257 x 64 images x 16 heads, per layer: forward 70 us, backward (incl. delta) 185 us; round 1 mma.sync
// kernels: 104 / 349 + 24; first tcgen05 version of this round (one CTA per item, 1-row tile in the pipeline): 102 / 214 + 24.  In SM
// cycles per item: forward 29 000 -> 14 500, backward 61 000 -> 36 000.  What bounds them now: a softmax warp spends ~2400 cycles per
// 64-column block (MUFU-bound share 1024: two warps per SM sub-partition, 8 cycles per MUFU.EX2 warp instruction), i.e. ~10 000
// cycles per item and warpgroup in the forward; the forward's epilogue warps (tile merges + ~9000 cycles of edge work per item) are
// its critical resource; the backward pays ~4000 cycles per item for the single-buffered operand reload (220 KB of shared memory
// are in use).  Under load the GPU runs these kernels at 1.45-1.8 GHz (sw_power_cap), not at 1.965.
#include "common.cuh"
#include "tcgen05.cuh"

using namespace tc;

namespace {

constexpr int AT_THREADS = 512;
constexpr int MAX_BLK = 5;  // 64-row blocks per operand
static_assert((ATTN_TC_MAX_T + 63) / 64 <= MAX_BLK, "operand blocks of the longest sequence");
constexpr float LOG2E_F = 1.4426950408889634f;
constexpr uint32_t BLK_BYTES = 64 * 128;     // one 64-row operand block
constexpr uint32_t TILE_BYTES = 128 * 128;   // one 128-row tile of an operand = one [128 x 64] staging tile

__device__ __forceinline__ uint32_t pack_bf2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float warp_max_f(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
        "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred;
}
__device__ __forceinline__ void st_shared_v4(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ void st256g(void* p, const uint32_t* w) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]),
               "r"(w[6]), "r"(w[7])
               : "memory");
}
// 64 fp32 accumulator values of one row (two tcgen05.ld x32) * mul -> 64 bf16 = 128 contiguous bytes
__device__ __forceinline__ void store_row64_bf16(__nv_bfloat16* dst, const uint32_t* a, const uint32_t* b, float mul) {
  uint32_t w[32];
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    w[j] = pack_bf2(__uint_as_float(a[2 * j]) * mul, __uint_as_float(a[2 * j + 1]) * mul);
    w[16 + j] = pack_bf2(__uint_as_float(b[2 * j]) * mul, __uint_as_float(b[2 * j + 1]) * mul);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) st256g(dst + 16 * j, w + 8 * j);
}

// ---- shared-memory / bf16 helpers of the "edge token" path (T = 64 m + 1: the last token is handled outside the tensor-core pipeline)
__device__ __forceinline__ uint32_t lds32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ float bf_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf_hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }
// dot product of two packed groups of 8 bf16
__device__ __forceinline__ float dot8p(const uint4 a, const uint4 b, float acc) {
  acc = fmaf(bf_lo(a.x), bf_lo(b.x), acc); acc = fmaf(bf_hi(a.x), bf_hi(b.x), acc); acc = fmaf(bf_lo(a.y), bf_lo(b.y), acc); acc = fmaf(bf_hi(a.y), bf_hi(b.y), acc);
  acc = fmaf(bf_lo(a.z), bf_lo(b.z), acc); acc = fmaf(bf_hi(a.z), bf_hi(b.z), acc); acc = fmaf(bf_lo(a.w), bf_lo(b.w), acc); acc = fmaf(bf_hi(a.w), bf_hi(b.w), acc);
  return acc;
}

struct AttnParams {
  int T, heads, ntiles, nblk, tail_rows;  // tiles / 64-wide blocks of the tensor-core pipeline; tail_rows: rows of its last block, rounded up to 16
  int nitems;                             // forward (persistent kernel): (image, head) items = Nimg * heads
  int edge, nblk_ld, ld_tail;             // edge = 1: T = 64 m + 1, token T-1 is handled on CUDA cores and the pipeline covers T-1 tokens;
                                          // operand blocks LOADED per operand (pipeline blocks + the edge block) and rows of the last one
  float scale;
  __nv_bfloat16* ctx;        // forward out [Nimg*T, D]
  float* lse;                // [Nimg, heads, T]  (forward out, backward in)
  const __nv_bfloat16* ctx_in;   // backward in: forward output [Nimg*T, D] and its gradient [Nimg*T, D] (delta = rowsum(dO * O) is computed
  const __nv_bfloat16* dctx_in;  // by the epilogue warps)
  __nv_bfloat16* dqkv;       // backward out [Nimg*T, 3D]
  long long* trace;          // debug: clock64() time line of CTA (0,0) (tools/trace_attn.py); nullptr in production
};

// ------------------------------------------------------------------------------------------------ forward (online softmax, persistent)
// PERSISTENT kernel: one CTA per SM walks the (image, head) items w = blockIdx.x, blockIdx.x + gridDim.x, ... and the block stream runs
// ACROSS items: the S MMAs, the softmax and the P V MMAs of item i+1 start while the last tile of item i is still being finished and
// written out, Q / K of item i+1 are loaded as soon as the last S MMA of item i has completed, V is double buffered.  (One CTA per item
// spent ~35% of its life outside the steady state: CTA launch + barrier / TMEM set-up ~3700 cycles, first TMA round trip ~1000, epilogue
// tail ~3000 of ~26000 -- measured with the time-line probes.)
//
// One pass over the score blocks of an item.  Block gg (running index over all items) goes to warpgroup gg & 1; each warpgroup keeps
// ITS OWN running reference maximum and row sum and accumulates its blocks into ITS OWN O accumulator in TMEM, so the two never wait for
// each other; the epilogue merges the partial results (flash-decoding style).  The reference maximum only moves when a block exceeds it
// by more than 2^8 (P stays <= 256: exact in fp32 / bf16 range), in which case the warpgroup rescales its accumulator in TMEM
// (tcgen05.ld / tcgen05.st) -- rare after the first block.
//
// T = 64 m + 1 (ViT-L/14: 257): the LAST token ("edge") stays out of the tensor-core pipeline, which then sees only full blocks and
// tiles (a 1-row tile costs the pipeline nblk dependent S -> softmax -> PV round trips: 25% of the item).  The epilogue warps compute
// the edge query row against all keys on CUDA cores while the first tile is in flight, and fold the edge key into every other row as
// a third partial result (one column: s_e = q . k_e, accumulator v_e, row sum 1) when they merge a tile.
//
//   warps 0 / 1   S = Q K^T of the even / odd blocks        warp 2   O += P V, TMEM allocation        warp 3   TMA producer
//   warps 4-11    two softmax warpgroups                    warps 12-15   epilogue + edge token
//   TMEM: S buffers 4 x 64 columns [0, 256); O[wg][tile & 1] at 256 + (2 wg + (tile & 1)) * 64.
struct FBars {
  uint32_t base;
  __device__ __forceinline__ uint32_t sfull(int b) const { return base + 8u * b; }                       // S block in TMEM buffer b            (tcgen05.commit)
  __device__ __forceinline__ uint32_t sfree(int b) const { return base + 32u + 8u * b; }                 // its warpgroup has read it           (4 warps)
  __device__ __forceinline__ uint32_t pready(int b) const { return base + 64u + 8u * b; }                // staging buffer b is written         (4 warps)
  __device__ __forceinline__ uint32_t pfree(int b) const { return base + 96u + 8u * b; }                 // the P V MMAs have consumed it       (tcgen05.commit)
  __device__ __forceinline__ uint32_t accfull(int a) const { return base + 128u + 8u * a; }              // accumulator a = 2 wg + (tile & 1)   (tcgen05.commit)
  __device__ __forceinline__ uint32_t accfree(int a) const { return base + 160u + 8u * a; }              // epilogue has read it                (4 warps)
  __device__ __forceinline__ uint32_t mready(int a, uint32_t r) const { return base + 192u + 8u * (2u * a + r); }  // row maxima / sums of use r (mod 2) of slot a (4 warps)
  __device__ __forceinline__ uint32_t opq(int blk) const { return base + 256u + 8u * blk; }              // operand blocks                      (TMA)
  __device__ __forceinline__ uint32_t opk(int blk) const { return base + 296u + 8u * blk; }
  __device__ __forceinline__ uint32_t opv(int vb, int blk) const { return base + 336u + 8u * (vb * MAX_BLK + blk); }
  __device__ __forceinline__ uint32_t qkfree() const { return base + 416u; }                             // Q / K of the item are no longer read (2 issuers + 4 epilogue warps)
  __device__ __forceinline__ uint32_t vfree(int vb) const { return base + 424u + 8u * vb; }              // V buffer vb                          (1 issuer + 4 epilogue warps)
  __device__ __forceinline__ uint32_t tmem_slot() const { return base + 440u; }
};
constexpr uint32_t FBARS_BYTES = 448 + 16;
constexpr uint32_t FWD_FLOATS = 4096 + 1024;  // sm[4][4][128], sl[4][4][128], edge scratch [1024]
constexpr float RESCALE_LOG2 = 8.f;

__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]),
      "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]),
      "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]),
      "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- warp-level mma.sync helpers of the edge-token path.  The edge token needs matrix-VECTOR products only (a [rows x 64] operand
// against one 64-long row, and one weight vector against the rows of an operand); on CUDA cores they cost ~3000 instructions per thread
// and item and slowed the softmax warps sharing the SM sub-partitions.  As m16n8k16 MMAs with the vector in column 0 of B (or row 0 of
// A) they take a few hundred instructions per warp; operands are read with ldmatrix straight from the TMA-written 128B-swizzled tiles.
__device__ __forceinline__ uint32_t swz_off(int row, int chunk) { return (uint32_t)(row * 128 + ((chunk ^ (row & 7)) << 4)); }
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr) : "memory");
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr) : "memory");
}
__device__ __forceinline__ void mma_bf16_16816(float c[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
// B fragments of a 64-long bf16 row (row `r` of an operand buffer, r % 8 == 0: not permuted by the swizzle) placed in column 0 of B:
// vb[2 kk], vb[2 kk + 1] for the four k-steps; zero in the lanes that hold other columns
__device__ __forceinline__ void load_vec_bfrag(uint32_t buf, int r, uint32_t vb[8]) {
  const int lane = threadIdx.x & 31, t = lane & 3;
  const uint32_t rowb = buf + (uint32_t)r * 128u;
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
    vb[2 * kk] = lane < 4 ? lds32(rowb + (uint32_t)(8 * kk + t) * 4u) : 0u;
    vb[2 * kk + 1] = lane < 4 ? lds32(rowb + (uint32_t)(8 * kk + t + 4) * 4u) : 0u;
  }
}
// rows [r0, r0 + 16) of a swizzled [rows x 64] bf16 buffer times the vector of vb: lanes with (lane & 3) == 0 return the products of rows
// r0 + (lane >> 2) (.x) and r0 + (lane >> 2) + 8 (.y)
__device__ __forceinline__ float2 mv16(uint32_t buf, int r0, const uint32_t vb[8]) {
  const int lane = threadIdx.x & 31;
  const int row = r0 + (lane & 7) + ((lane >> 3) & 1) * 8;
  float c[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
    uint32_t a0, a1, a2, a3;
    ldsm_x4(buf + swz_off(row, kk * 2 + (lane >> 4)), a0, a1, a2, a3);
    mma_bf16_16816(c, a0, a1, a2, a3, vb[2 * kk], vb[2 * kk + 1]);
  }
  return make_float2(c[0], c[2]);
}
// two independent row groups at once (the four chained MMAs of one group leave the pipe mostly idle)
__device__ __forceinline__ void mv16x2(uint32_t buf, int r0a, int r0b, const uint32_t vb[8], float2& ra, float2& rb) {
  const int lane = threadIdx.x & 31;
  const int rowa = r0a + (lane & 7) + ((lane >> 3) & 1) * 8, rowb = r0b + (lane & 7) + ((lane >> 3) & 1) * 8;
  float ca[4] = {0.f, 0.f, 0.f, 0.f}, cb[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
    uint32_t a0, a1, a2, a3, b0, b1, b2, b3;
    ldsm_x4(buf + swz_off(rowa, kk * 2 + (lane >> 4)), a0, a1, a2, a3);
    ldsm_x4(buf + swz_off(rowb, kk * 2 + (lane >> 4)), b0, b1, b2, b3);
    mma_bf16_16816(ca, a0, a1, a2, a3, vb[2 * kk], vb[2 * kk + 1]);
    mma_bf16_16816(cb, b0, b1, b2, b3, vb[2 * kk], vb[2 * kk + 1]);
  }
  ra = make_float2(ca[0], ca[2]);
  rb = make_float2(cb[0], cb[2]);
}
// acc[n][.] += vec[k0 .. k0 + 16) (fp32 in shared memory, rounded to bf16 like the staged P / dS of the pipeline) times rows [k0, k0 + 16)
// of a swizzled [rows x 64] bf16 buffer: the vector sits in row 0 of A; lanes 0-3 hold the result, acc[n][0..1] = columns 8 n + 2 t, + 1
__device__ __forceinline__ void vm16(uint32_t buf, int k0, const float* vec, float acc[8][4]) {
  const int lane = threadIdx.x & 31, t = lane & 3;
  uint32_t a0 = 0u, a2 = 0u;
  if (lane < 4) {
    const float2 x = *reinterpret_cast<const float2*>(vec + k0 + 2 * t), y = *reinterpret_cast<const float2*>(vec + k0 + 2 * t + 8);
    a0 = pack_bf2(x.x, x.y);
    a2 = pack_bf2(y.x, y.y);
  }
  const int row = k0 + (lane & 7) + ((lane >> 3) & 1) * 8;
  uint32_t b[4][4];
#pragma unroll
  for (int cp = 0; cp < 4; ++cp) ldsm_x4_t(buf + swz_off(row, cp * 2 + (lane >> 4)), b[cp][0], b[cp][1], b[cp][2], b[cp][3]);
#pragma unroll
  for (int cp = 0; cp < 4; ++cp) {
    mma_bf16_16816(acc[2 * cp], a0, 0u, a2, 0u, b[cp][0], b[cp][1]);
    mma_bf16_16816(acc[2 * cp + 1], a0, 0u, a2, 0u, b[cp][2], b[cp][3]);
  }
}

// The edge token of the forward (T = Tp + 1, Tp a multiple of 64), by the four epilogue warps (128 threads) with warp-level MMAs:
//   * the edge QUERY row against all T keys (scores = K q_e, softmax, O_e = p V) -> ctx_row (64 bf16), lse_out
//   * the edge KEY against every other row (Q k_e) -> returned for this thread's rows rl and 128 + rl (log2 units, -inf beyond Tp): the
//     third partial result of the tile merge;  v_e as floats -> pvec[552 .. 616)
// scratch pvec: [288] scores / numerators, [8] reductions, [4][64] partial outputs, [256] edge-key scores; vedge: [64] v_e as floats
#ifdef CG_ATTN_TRACE
#define TRE(ev) do { if (tr != nullptr && (threadIdx.x & 31) == 0) tr[ev] = clock64(); } while (0)
#else
#define TRE(ev) do { } while (0)
#endif
// Two parts: A reads Q and K (scores of the edge query, scores of the edge key), B reads V (softmax of the edge query row, its output
// row, v_e) -- the caller runs A early, because Q / K are single buffered and their reload waits for it, and B later.
__device__ __forceinline__ float2 fwd_edge_token_a(uint32_t sQ, uint32_t sK, int Tp, float sl2, float* pvec, long long* tr) {
  const int rl = threadIdx.x & 127, q = rl >> 5, lane = rl & 31, g = lane >> 2, t = lane & 3;
  const int T = Tp + 1;
  float* sev = pvec + 552;    // [256]
  {
    uint32_t vb[8];
    load_vec_bfrag(sQ, Tp, vb);  // q_e
    const int ng = Tp >> 4;  // full key groups; group ng holds the edge key itself in its row 0
#pragma unroll 1
    for (int rg = q; rg <= ng; rg += 8) {  // two groups per step (independent MMA chains)
      const int rg2 = rg + 4 <= ng ? rg + 4 : rg;
      float2 c, c2;
      mv16x2(sK, rg * 16, rg2 * 16, vb, c, c2);
      if (t == 0) {
        const int j0 = rg * 16 + g, j1 = j0 + 8, k0 = rg2 * 16 + g, k1 = k0 + 8;
        pvec[j0] = j0 < T ? c.x * sl2 : -INFINITY;
        pvec[j1] = j1 < T ? c.y * sl2 : -INFINITY;
        pvec[k0] = k0 < T ? c2.x * sl2 : -INFINITY;
        pvec[k1] = k1 < T ? c2.y * sl2 : -INFINITY;
      }
    }
    TRE(0);
    load_vec_bfrag(sK, Tp, vb);  // k_e
#pragma unroll 1
    for (int rg = q; rg < ng; rg += 8) {
      const int rg2 = rg + 4 < ng ? rg + 4 : rg;
      float2 c, c2;
      mv16x2(sQ, rg * 16, rg2 * 16, vb, c, c2);
      if (t == 0) {
        sev[rg * 16 + g] = c.x * sl2; sev[rg * 16 + g + 8] = c.y * sl2;
        sev[rg2 * 16 + g] = c2.x * sl2; sev[rg2 * 16 + g + 8] = c2.y * sl2;
      }
    }
  }
  TRE(1);
  asm volatile("bar.sync 2, 128;" ::: "memory");
  return make_float2(rl < Tp ? sev[rl] : -INFINITY, 128 + rl < Tp ? sev[128 + rl] : -INFINITY);
}
__device__ __forceinline__ void fwd_edge_token_b(uint32_t sV, int Tp, float* pvec, float* vedge, __nv_bfloat16* ctx_row, float* lse_out, long long* tr) {
  const int rl = threadIdx.x & 127, q = rl >> 5, lane = rl & 31;
  float* red = pvec + 288;
  float* part = pvec + 296;   // [4][64]
  if (rl < 32) {
    const uint32_t v2 = lds32(sV + (uint32_t)Tp * 128u + (uint32_t)rl * 4u);
    vedge[2 * rl] = bf_lo(v2);
    vedge[2 * rl + 1] = bf_hi(v2);
  }
  TRE(2);
  const int ngrp = (Tp >> 4) + 1;  // pvec holds 16 ngrp entries
  float mx = -INFINITY;
  for (int j = rl; j < 16 * ngrp; j += 128) mx = fmaxf(mx, pvec[j]);
  mx = warp_max_f(mx);
  if (lane == 0) red[q] = mx;
  asm volatile("bar.sync 2, 128;" ::: "memory");
  mx = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
  float l = 0.f;
  for (int j = rl; j < 16 * ngrp; j += 128) {
    const float pj = ex2f(pvec[j] - mx);  // 0 beyond T
    pvec[j] = pj;
    l += pj;
  }
  l = warp_sum(l);
  if (lane == 0) red[4 + q] = l;
  asm volatile("bar.sync 2, 128;" ::: "memory");
  l = (red[4] + red[5]) + (red[6] + red[7]);
  TRE(3);
  {
    // O_e = sum_j p_j V[j] on CUDA cores: warp q takes the keys j = q (mod 4), lane owns d = 2 lane, 2 lane + 1 (one 32-bit word of a V
    // row: conflict free).  (As 16-key MMA steps this took twice as long: legacy mma.sync next to running tcgen05 MMAs, ~700 cycles a step.)
    const int T = Tp + 1;
    const uint32_t vcol = ((uint32_t)(lane >> 2) << 4), vin = (uint32_t)(lane & 3) << 2;
    float o0 = 0.f, o1 = 0.f, o2 = 0.f, o3 = 0.f;
    int j = q;
#pragma unroll 4
    for (; j + 4 < T; j += 8) {
      const uint32_t va = lds32(sV + (uint32_t)j * 128u + (vcol ^ ((uint32_t)(j & 7) << 4)) + vin);
      const uint32_t vb = lds32(sV + (uint32_t)(j + 4) * 128u + (vcol ^ ((uint32_t)((j + 4) & 7) << 4)) + vin);
      const float pa = pvec[j], pb = pvec[j + 4];
      o0 = fmaf(pa, bf_lo(va), o0); o1 = fmaf(pa, bf_hi(va), o1);
      o2 = fmaf(pb, bf_lo(vb), o2); o3 = fmaf(pb, bf_hi(vb), o3);
    }
    if (j < T) {
      const uint32_t va = lds32(sV + (uint32_t)j * 128u + (vcol ^ ((uint32_t)(j & 7) << 4)) + vin);
      o0 = fmaf(pvec[j], bf_lo(va), o0); o1 = fmaf(pvec[j], bf_hi(va), o1);
    }
    *reinterpret_cast<float2*>(part + q * 64 + 2 * lane) = make_float2(o0 + o2, o1 + o3);
  }
  TRE(4);
  asm volatile("bar.sync 2, 128;" ::: "memory");
  TRE(5);
  if (q == 0) {
    const float inv = __fdividef(1.f, l);
    const float2 a0 = *reinterpret_cast<const float2*>(part + 2 * lane), a1 = *reinterpret_cast<const float2*>(part + 64 + 2 * lane);
    const float2 a2 = *reinterpret_cast<const float2*>(part + 128 + 2 * lane), a3 = *reinterpret_cast<const float2*>(part + 192 + 2 * lane);
    reinterpret_cast<uint32_t*>(ctx_row)[lane] = pack_bf2(((a0.x + a1.x) + (a2.x + a3.x)) * inv, ((a0.y + a1.y) + (a2.y + a3.y)) * inv);
    if (lane == 0) *lse_out = mx * (1.f / LOG2E_F) + logf(l);
  }
  asm volatile("bar.sync 2, 128;" ::: "memory");  // vedge is complete for every epilogue warp; pvec / part may be reused
}

// time-line probe of the persistent kernel: CTA 0, its third item (warm caches, steady state)
#ifdef CG_ATTN_TRACE
#define TRF(slot, idx, ev)                                                                                   \
  do {                                                                                                       \
    if (p.trace != nullptr && blockIdx.x == 0 && it == 2 && (threadIdx.x & 31) == 0)                         \
      p.trace[(((slot) * 64 + (idx)) << 3) + (ev)] = clock64();                                              \
  } while (0)
// every item of CTA 0: idx = 32 + item iteration (< 24)
#define TRI(slot, ev)                                                                                        \
  do {                                                                                                       \
    if (p.trace != nullptr && blockIdx.x == 0 && it < 24 && (threadIdx.x & 31) == 0)                         \
      p.trace[(((slot) * 64 + 32 + it) << 3) + (ev)] = clock64();                                            \
  } while (0)
#else
#define TRF(slot, idx, ev) do { } while (0)
#define TRI(slot, ev) do { } while (0)
#endif

// CAUSAL (the CLIP text transformer): column j of row i is masked (-inf) when j > i, with i = tile * 128 + row and j = block * 64 +
// column.  Fully masked blocks are NOT skipped -- every block still runs through every role, so the barrier phases stay as described
// above (at T = 77 such a block costs little).  A row whose share of a block is fully masked stages P = 0 for all 64 columns (a
// select, never an exp of -inf - -inf), keeps its row sum at 0 and, if this was the warpgroup's first block of the tile, its
// reference maximum at -inf; the next block with a kept column rescales the (zero) accumulator by ex2(-inf) = 0 like any other
// reference move.  In the epilogue merge such a partial result weighs ex2(-inf - M) = 0, and M is finite because column 0 is kept
// for every row, so the other warpgroup's result stands.  The edge token is off (p.edge = 0, compiled out here).
template <bool CAUSAL>
__global__ void __launch_bounds__(AT_THREADS, 1)
    attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmQKVtail, const AttnParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  cg_griddep_launch();
  const int T = p.T, heads = p.heads, D = heads * 64;
  const int edge = CAUSAL ? 0 : p.edge, Tp = T - edge;  // Tp tokens go through the tensor-core pipeline; with edge = 1 token Tp is handled on CUDA cores
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ntiles = p.ntiles, nblk = p.nblk, nblk_ld = p.nblk_ld;
  const int G = ntiles * nblk, nitems = p.nitems;
  const uint32_t opb = (uint32_t)((nblk_ld - 1) * 64 + p.ld_tail) * 128u;
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sQ = base, sK = base + opb, sV0 = base + 2 * opb;  // Q, K, V[2]
  const uint32_t sStage = base + 4 * opb;                            // 4 x [128 x 64] bf16 P tiles
  const uint32_t sF = sStage + 4 * TILE_BYTES;
  float* fscr = reinterpret_cast<float*>(smem_raw + (sF - smem_u32(smem_raw)));
  float* sm = fscr;           // [4 slots][4 uses][128] reference maxima (log2 units) of a warpgroup's share of a tile
  float* sl = fscr + 2048;    // [4 slots][4 uses][128] partial row sums
  float* pvec = fscr + 4096;  // edge scratch: softmax numerators of the edge query row [288], reductions [8 + 256], v_e [64]
  FBars bars{sF + FWD_FLOATS * 4};

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQKV) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQKVtail) : "memory");
    for (int b = 0; b < 4; ++b) {
      mbar_init(bars.sfull(b), 1); mbar_init(bars.sfree(b), 4); mbar_init(bars.pready(b), 4); mbar_init(bars.pfree(b), 1);
      mbar_init(bars.accfull(b), 1); mbar_init(bars.accfree(b), 4);
      mbar_init(bars.mready(b, 0), 4); mbar_init(bars.mready(b, 1), 4);
    }
    for (int k = 0; k < MAX_BLK; ++k) { mbar_init(bars.opq(k), 1); mbar_init(bars.opk(k), 1); mbar_init(bars.opv(0, k), 1); mbar_init(bars.opv(1, k), 1); }
    mbar_init(bars.qkfree(), 6);
    mbar_init(bars.vfree(0), 5);
    mbar_init(bars.vfree(1), 5);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(bars.tmem_slot()), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  cg_griddep_wait();  // everything below reads the predecessor's output or overwrites its input
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(bars.tmem_slot()) : "memory");

  if (warp == 3) {
    // ================= TMA producer: Q / K single buffered (reloaded when the item's last S MMA and edge reads are done), V double buffered
    if (lane == 0) {
      int it = 0;
      for (int w = blockIdx.x; w < nitems; w += gridDim.x, ++it) {
        const int n = w / heads, h = w - n * heads, row0 = n * T, vb = it & 1;
        auto load = [&](uint32_t dst0, uint32_t bar, int col, int blk) {
          const bool tail = blk == nblk_ld - 1;
          mbar_arrive_expect_tx(bar, (uint32_t)(tail ? p.ld_tail : 64) * 128u);
          tma_load_2d(dst0 + blk * BLK_BYTES, tail ? &tmQKVtail : &tmQKV, bar, col, row0 + blk * 64);
        };
        const int qc = h * 64, kc = D + h * 64, vc = 2 * D + h * 64;
        const uint32_t sVb = sV0 + vb * opb;
        // rolled loops on purpose (code size).  V first: its buffer has been free for a whole item, while Q / K have to wait for the
        // previous item's last S MMA
        if (it >= 2) mbar_wait(bars.vfree(vb), (uint32_t)((it >> 1) - 1) & 1u);  // item it - 2 has left this V buffer
#pragma unroll 1
        for (int k = 0; k < nblk_ld; ++k) load(sVb, bars.opv(vb, k), vc, k);
        if (it >= 1) mbar_wait(bars.qkfree(), (uint32_t)(it - 1) & 1u);           // item it - 1 has left Q and K
#pragma unroll 1
        for (int k = 0; k < nblk_ld; ++k) {
          load(sK, bars.opk(k), kc, k);
          load(sQ, bars.opq(k), qc, k);
        }
        // the operands are single (V: double) buffered, so the next item's loads cannot be issued early: pull its tiles into L2 now
        if (w + (int)gridDim.x < nitems) {
          const int w2 = w + gridDim.x, n2 = w2 / heads, h2 = w2 - n2 * heads;
#pragma unroll 1
          for (int k = 0; k < nblk_ld; ++k) {
            const CUtensorMap* tm = k == nblk_ld - 1 ? &tmQKVtail : &tmQKV;
            tma_prefetch_2d(tm, D + h2 * 64, n2 * T + k * 64);
            tma_prefetch_2d(tm, h2 * 64, n2 * T + k * 64);
            tma_prefetch_2d(tm, 2 * D + h2 * 64, n2 * T + k * 64);
          }
        }
      }
    }
  } else if (warp < 2) {
    // ================= S issuers (warp-converged loops, elected lane): warp = parity of the running block index
    const uint32_t elected = elect_one();
    const uint32_t id_full = idesc_bf16(128, 64, false), id_tail = idesc_bf16(128, p.tail_rows, false);
    int it = 0, gg0 = 0;
    for (int w = blockIdx.x; w < nitems; w += gridDim.x, ++it, gg0 += G) {
      const uint32_t opar = (uint32_t)it & 1u;
      uint32_t loaded = 0;  // bit blk: Q block seen complete, bit 8 + blk: K block
      auto need = [&](uint32_t bar, uint32_t bit) {
        if (!(loaded & bit)) { mbar_wait(bar, opar); loaded |= bit; }
      };
      int g = ((gg0 & 1) == warp) ? 0 : 1;
      int tile = 0, blk = g;
      while (blk >= nblk) { blk -= nblk; ++tile; }
      bool any = false;
      for (; g < G; g += 2) {
        const int gg = gg0 + g, b = gg & 3;
        need(bars.opq(2 * tile), 1u << (2 * tile));
        if (2 * tile + 1 < nblk) need(bars.opq(2 * tile + 1), 1u << (2 * tile + 1));
        need(bars.opk(blk), 256u << blk);
        mbar_wait(bars.sfree(b), ((uint32_t)(gg >> 2) & 1u) ^ 1u);
        TRF(warp, g, 0);
        tcgen05_fence_after();
        const uint32_t d_s = tmem_base + (uint32_t)(b * 64);
        const uint64_t ad = make_smem_desc(sQ + tile * TILE_BYTES), bd = make_smem_desc(sK + blk * BLK_BYTES);
        const uint32_t idesc = blk == nblk - 1 ? id_tail : id_full;
        if (elected) {
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16(d_s, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, k != 0 ? 1u : 0u);
          umma_commit(bars.sfull(b));
        }
        __syncwarp();
        TRF(warp, g, 1);
        any = true;
        blk += 2;
        while (blk >= nblk) { blk -= nblk; ++tile; }
      }
      // a parity wait is only sound for a waiter that sees EVERY phase: with an odd block count the blocks (and operand barriers) this
      // warp needs alternate from item to item, so it also observes the ones it did not need
#pragma unroll 1
      for (int k = 0; k < nblk_ld; ++k) { need(bars.opq(k), 1u << k); need(bars.opk(k), 256u << k); }
      if (elected) {  // this warp is done with Q and K of the item
        if (any) umma_commit(bars.qkfree());
        else mbar_arrive(bars.qkfree());
      }
      __syncwarp();
    }
  } else if (warp == 2) {
    // ================= P V issuer
    const uint32_t elected = elect_one();
    const uint32_t id_acc = idesc_bf16(128, 64, true);
    uint32_t accpar = 0;  // bit a: parity of the use count of accumulator slot a
    int it = 0, gg0 = 0;
    for (int w = blockIdx.x; w < nitems; w += gridDim.x, ++it, gg0 += G) {
      const int vb = it & 1;
      const uint32_t vpar = (uint32_t)(it >> 1) & 1u, sVb = sV0 + vb * opb;
      uint32_t loaded = 0;
      int tile = 0, blk = 0;
      for (int g = 0; g < G; ++g) {
        const int gg = gg0 + g, pb = gg & 3, wg = gg & 1, a = 2 * wg + (tile & 1);
        const bool first = blk < 2, last = blk + 2 >= nblk;  // first / last block of THIS warpgroup in the tile
        if (!(loaded & (1u << blk))) { mbar_wait(bars.opv(vb, blk), vpar); loaded |= 1u << blk; }
        mbar_wait(bars.pready(pb), (uint32_t)(gg >> 2) & 1u);
        TRF(warp, g, 0);
        if (first) mbar_wait(bars.accfree(a), ((accpar >> a) & 1u) ^ 1u);
        tcgen05_fence_after();
        const uint32_t d_acc = tmem_base + 256u + (uint32_t)(a * 64);
        const uint64_t ad = make_smem_desc(sStage + pb * TILE_BYTES), bd = make_smem_desc(sVb + blk * BLK_BYTES);
        if (elected) {
          if (blk != nblk - 1) {
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16(d_acc, ad + (uint64_t)(2 * k), bd + (uint64_t)(128 * k), id_acc, (!first || k != 0) ? 1u : 0u);
          } else {
            const int ksteps = p.tail_rows >> 4;
            for (int k = 0; k < ksteps; ++k) umma_bf16(d_acc, ad + (uint64_t)(2 * k), bd + (uint64_t)(128 * k), id_acc, (!first || k != 0) ? 1u : 0u);
          }
          umma_commit(bars.pfree(pb));
          if (last) umma_commit(bars.accfull(a));
        }
        __syncwarp();
        TRF(warp, g, 1);
        if (last) accpar ^= 1u << a;
        if (++blk == nblk) { blk = 0; ++tile; }
      }
      if (elected) umma_commit(bars.vfree(vb));  // this V buffer may be refilled once the item's last P V MMA has completed
      __syncwarp();
    }
  } else if (warp < 12) {
    // ================= softmax warpgroups
    const int wg = (warp - 4) >> 2;
    const int q = warp & 3;
    const int rl = q * 32 + lane;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    const float sl2 = p.scale * LOG2E_F;
    const int tail_cols = Tp - (nblk - 1) * 64;
    const uint32_t sx = (uint32_t)(rl & 7) << 4;  // 128B swizzle of this thread's row of a staged tile: 16-byte chunk c sits at (c << 4) ^ sx
    uint32_t wuse0 = 0, wuse1 = 0;  // uses of this warpgroup's two accumulator slots (tile parity 0 / 1)
    int it = 0, gg0 = 0;
    for (int w = blockIdx.x; w < nitems; w += gridDim.x, ++it, gg0 += G) {
      float mref = -INFINITY, lsum = 0.f;  // running reference maximum (log2 units) and row sum of this warpgroup in the current tile
      int cur_tile = -1;
      int g = ((gg0 & 1) == wg) ? 0 : 1;
      int tile = 0, blk = g;
      while (blk >= nblk) { blk -= nblk; ++tile; }
      for (; g < G; g += 2) {
        const int gg = gg0 + g;
        const bool first = tile != cur_tile;
        cur_tile = tile;
        const bool wvalid = tile * 128 + q * 32 < Tp;
        const bool rvalid = tile * 128 + rl < Tp;
        const bool tail = blk == nblk - 1, last_in_tile = blk + 2 >= nblk;
        const int b = gg & 3;                 // S buffer and staging buffer
        const uint32_t use = (uint32_t)(gg >> 2);
        mbar_wait(bars.sfull(b), use & 1u);
        TRF(warp, g, 1);
        tcgen05_fence_after();
        if (!wvalid) {
          tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bars.sfree(b));
          mbar_wait(bars.pfree(b), (use & 1u) ^ 1u);  // stay in step with the barrier phases (see the backward kernel)
        } else {
          // Register budget (512 threads x 128 registers, and the local memory of a spill lives in L2 here: shared memory leaves ~28 KB of
          // L1): the block is read from TMEM TWICE.  Pass 1 takes the block maximum over both 32-column halves; the first half is then
          // dropped, the second half is exponentiated and staged, the first half is fetched again (a TMEM read costs a few dozen cycles).
          uint32_t sa[32], sb[32], w[16];
          const uint32_t t_s = t_lane + (uint32_t)(b * 64);
          tmem_ld32(t_s, sa);
          tmem_ld32(t_s + 32u, sb);  // (a tail block narrower than 32 columns leaves stale columns here: masked below)
          tmem_ld_wait();
          TRF(warp, g, 0);
          // block maximum over the valid columns
          float bm = -INFINITY;
          // causal: columns [0, lim) of this block are kept for this thread's row (lim <= 0: none)
          const int lim = CAUSAL ? min(tail ? tail_cols : 64, tile * 128 + rl - blk * 64 + 1) : 64;
          if constexpr (CAUSAL) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              if (j < lim) bm = fmaxf(bm, __uint_as_float(sa[j]));
              if (32 + j < lim) bm = fmaxf(bm, __uint_as_float(sb[j]));
            }
          } else if (!tail) {
#pragma unroll
            for (int j = 0; j < 32; ++j) bm = fmaxf(bm, fmaxf(__uint_as_float(sa[j]), __uint_as_float(sb[j])));
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              if (j < tail_cols) bm = fmaxf(bm, __uint_as_float(sa[j]));
              if (32 + j < tail_cols) bm = fmaxf(bm, __uint_as_float(sb[j]));
            }
          }
          bm *= sl2;
          TRF(warp, g, 4);
          if (first) {
            mref = bm;
            lsum = 0.f;
          } else {
            const bool grow = rvalid && bm > mref + RESCALE_LOG2;
            if (__any_sync(0xffffffffu, grow)) {
              // the reference moves: rescale this warpgroup's accumulator.  Its previous block (gg - 2) must have left the tensor pipe.
              const int pbp = (gg - 2) & 3;
              mbar_wait(bars.pfree(pbp), (uint32_t)((gg - 2) >> 2) & 1u);
              tcgen05_fence_after();
              const float f = grow ? ex2f(mref - bm) : 1.f;
              const uint32_t t_o = t_lane + 256u + (uint32_t)((2 * wg + (tile & 1)) * 64);
              if constexpr (CAUSAL) {
                // 16 columns at a time: lim stays live across this block, and 32 more registers next to sb would spill
#pragma unroll
                for (int c = 0; c < 64; c += 16) {
                  tmem_ld16(t_o + (uint32_t)c, sa);
                  tmem_ld_wait();
#pragma unroll
                  for (int j = 0; j < 16; ++j) sa[j] = __float_as_uint(__uint_as_float(sa[j]) * f);
                  tmem_st16(t_o + (uint32_t)c, sa);
                }
              } else {
#pragma unroll
                for (int c = 0; c < 64; c += 32) {  // (sa is dead here: it is fetched again below)
                  tmem_ld32(t_o + (uint32_t)c, sa);
                  tmem_ld_wait();
#pragma unroll
                  for (int j = 0; j < 32; ++j) sa[j] = __float_as_uint(__uint_as_float(sa[j]) * f);
                  tmem_st32(t_o + (uint32_t)c, sa);
                }
              }
              tmem_st_wait();
              tcgen05_fence_before();
              lsum *= f;
              if (grow) mref = bm;
            }
          }
          bool waited = false;
#pragma unroll
          for (int pass = 0; pass < 2; ++pass) {
            const int hlf = 1 - pass;  // second half first (it is still in registers), then the first half again
            if (pass == 1) {
              tmem_ld32(t_s, sa);
              tmem_ld_wait();
              tcgen05_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(bars.sfree(b));  // every TMEM read of this block has completed
            }
            const uint32_t* sv = hlf ? sb : sa;
            float a0 = 0.f, a1 = 0.f;  // independent partial sums
            if constexpr (CAUSAL) {
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                float p0 = ex2f(fmaf(__uint_as_float(sv[2 * j]), sl2, -mref)), p1 = ex2f(fmaf(__uint_as_float(sv[2 * j + 1]), sl2, -mref));
                if (hlf * 32 + 2 * j >= lim) p0 = 0.f;  // (also replaces the inf / NaN of a fully masked row: mref = -inf)
                if (hlf * 32 + 2 * j + 1 >= lim) p1 = 0.f;
                a0 += p0;
                a1 += p1;
                w[j] = pack_bf2(p0, p1);
              }
            } else if (!tail) {
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const float p0 = ex2f(fmaf(__uint_as_float(sv[2 * j]), sl2, -mref)), p1 = ex2f(fmaf(__uint_as_float(sv[2 * j + 1]), sl2, -mref));
                a0 += p0;
                a1 += p1;
                w[j] = pack_bf2(p0, p1);
              }
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                float p0 = ex2f(fmaf(__uint_as_float(sv[2 * j]), sl2, -mref)), p1 = ex2f(fmaf(__uint_as_float(sv[2 * j + 1]), sl2, -mref));
                if (hlf * 32 + 2 * j >= tail_cols) p0 = 0.f;
                if (hlf * 32 + 2 * j + 1 >= tail_cols) p1 = 0.f;
                a0 += p0;
                a1 += p1;
                w[j] = pack_bf2(p0, p1);
              }
            }
            lsum += a0 + a1;
            TRF(warp, g, 5 + hlf);
            if (!waited) { mbar_wait(bars.pfree(b), (use & 1u) ^ 1u); waited = true; }  // staging buffer free again
            const uint32_t hb = sStage + b * TILE_BYTES + (uint32_t)rl * 128u;
            st_shared_v4(hb + (((uint32_t)(hlf * 64)) ^ sx), w[0], w[1], w[2], w[3]);
            st_shared_v4(hb + (((uint32_t)(hlf * 64 + 16)) ^ sx), w[4], w[5], w[6], w[7]);
            st_shared_v4(hb + (((uint32_t)(hlf * 64 + 32)) ^ sx), w[8], w[9], w[10], w[11]);
            st_shared_v4(hb + (((uint32_t)(hlf * 64 + 48)) ^ sx), w[12], w[13], w[14], w[15]);
          }
        }
        if (last_in_tile) {
          // this warpgroup's share of the tile is complete: hand its reference maximum and row sum to the epilogue (ring of 4 per
          // slot: the staging depth lets a warpgroup run at most two uses of a slot ahead of the epilogue)
          const int tp = tile & 1, a = 2 * wg + tp;
          const uint32_t u = tp ? wuse1 : wuse0;
          if (wvalid) {
            sm[(a * 4 + (int)(u & 3u)) * 128 + rl] = mref;
            sl[(a * 4 + (int)(u & 3u)) * 128 + rl] = lsum;
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(bars.mready(a, u & 1u));
          if (tp) wuse1 = u + 1; else wuse0 = u + 1;
        }
        TRF(warp, g, 2);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(bars.pready(b));
        TRF(warp, g, 3);
        blk += 2;
        while (blk >= nblk) { blk -= nblk; ++tile; }
      }
    }
  } else {
    // ================= epilogue warps: edge token, then merge the two warpgroups' partial results of every tile -> ctx (bf16), lse
    const int q = warp & 3;
    const int rl = q * 32 + lane;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    const float sl2 = p.scale * LOG2E_F;
    float* vedge2 = pvec + 808;                               // [2][64] v_e as floats (written by fwd_edge_token), by item parity
    uint32_t euse = 0;  // 4 bits per accumulator slot: its use count (mod 16)
    // The edge token of item i + 1 is processed BETWEEN the first and the remaining tiles of item i (its Q / K arrive once the S MMAs of
    // item i are done, V is double buffered): the edge work then never sits between the end of one item and the reload of Q / K for the
    // next.  (Measured alternatives: at the start of the item's own iteration -> the Q / K reload waits for it, +10% cycles; V part
    // after the last tile -> no gain.)  This role stays the forward's critical resource at T = 257: ~2 x 2100 cycles of tile merges +
    // ~9000 of edge work per item against ~12 000 of softmax per warpgroup.  se0 / se1: edge-key scores of this thread's rows in tile 0 / 1.
    auto edge_a = [&](int wi, int eit, float& s0, float& s1) {  // Q / K part of the edge token of item wi (iteration eit)
      const uint32_t opar = (uint32_t)eit & 1u;
      if (edge) {
        for (int b = 0; b < nblk_ld; ++b) { mbar_wait(bars.opk(b), opar); mbar_wait(bars.opq(b), opar); }
#ifdef CG_ATTN_TRACE
        long long* etr = (p.trace != nullptr && blockIdx.x == 0 && eit == 3) ? p.trace + ((warp * 64 + 60) << 3) : nullptr;
#else
        long long* etr = nullptr;
#endif
        const float2 se = fwd_edge_token_a(sQ, sK, Tp, sl2, pvec, etr);
        s0 = se.x;
        s1 = se.y;
      } else if (eit > 0) {
        mbar_wait(bars.qkfree(), (uint32_t)(eit - 1) & 1u);  // the arrival below must not land in the previous item's phase
      }
      // this role no longer reads Q and K of that item from shared memory (the arrival orders the reads above before the refill)
      __syncwarp();
      if (lane == 0) mbar_arrive(bars.qkfree());
    };
    auto edge_b = [&](int wi, int eit) {  // V part
      const int n = wi / heads, h = wi - n * heads, row0 = n * T, vb = eit & 1;
      if (edge) {
        for (int b = 0; b < nblk_ld; ++b) mbar_wait(bars.opv(vb, b), (uint32_t)(eit >> 1) & 1u);
#ifdef CG_ATTN_TRACE
        long long* etr = (p.trace != nullptr && blockIdx.x == 0 && eit == 3) ? p.trace + ((warp * 64 + 60) << 3) : nullptr;
#else
        long long* etr = nullptr;
#endif
        fwd_edge_token_b(sV0 + vb * opb, Tp, pvec, vedge2 + vb * 64, p.ctx + ((long long)(row0 + Tp)) * D + h * 64, p.lse + ((long long)n * heads + h) * T + Tp, etr);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bars.vfree(vb));
    };
    float se0 = -INFINITY, se1 = -INFINITY, nse0 = -INFINITY, nse1 = -INFINITY;
    if ((int)blockIdx.x < nitems) { edge_a(blockIdx.x, 0, se0, se1); edge_b(blockIdx.x, 0); }
    int it = 0, gg0 = 0;
    for (int w = blockIdx.x; w < nitems; w += gridDim.x, ++it, gg0 += G) {
      const int n = w / heads, h = w - n * heads, row0 = n * T;
      const float* vedge = vedge2 + (it & 1) * 64;
      TRF(warp, 62, 0);
      TRI(warp, 0);
      for (int tile = 0; tile < ntiles; ++tile) {
        const int tp = tile & 1, a0 = tp, a1 = 2 + tp;
        // with a single block per tile only warpgroup (running block index) & 1 takes part
        const int ggt = gg0 + tile * nblk;
        const bool has0 = nblk > 1 || (ggt & 1) == 0, has1 = nblk > 1 || (ggt & 1) == 1;
        const uint32_t u0 = (euse >> (4 * a0)) & 15u, u1 = (euse >> (4 * a1)) & 15u;
        if (has0) { mbar_wait(bars.mready(a0, u0 & 1u), (u0 >> 1) & 1u); mbar_wait(bars.accfull(a0), u0 & 1u); }
        if (has1) { mbar_wait(bars.mready(a1, u1 & 1u), (u1 >> 1) & 1u); mbar_wait(bars.accfull(a1), u1 & 1u); }
        TRF(warp, tile, 0);
        tcgen05_fence_after();
        const int row = tile * 128 + rl;
        if (tile * 128 + q * 32 < Tp) {
          const float m0 = has0 ? sm[(a0 * 4 + (int)(u0 & 3u)) * 128 + rl] : -INFINITY, m1 = has1 ? sm[(a1 * 4 + (int)(u1 & 3u)) * 128 + rl] : -INFINITY;
          const float l0 = has0 ? sl[(a0 * 4 + (int)(u0 & 3u)) * 128 + rl] : 0.f, l1 = has1 ? sl[(a1 * 4 + (int)(u1 & 3u)) * 128 + rl] : 0.f;
          const float se = tile == 0 ? se0 : se1;  // -inf without an edge token (and for tiles >= 2, which only exist without one)
          const float M = fmaxf(fmaxf(m0, m1), se);
          const float f0 = has0 ? ex2f(m0 - M) : 0.f, f1 = has1 ? ex2f(m1 - M) : 0.f, fe = ex2f(se - M);
          const float L = l0 * f0 + l1 * f1 + fe;
          const float invL = __fdividef(1.f, L);
          const float g0 = f0 * invL, g1 = f1 * invL, ge = fe * invL;
          __nv_bfloat16* dst = p.ctx + ((long long)(row0 + row)) * D + h * 64;
#pragma unroll
          for (int c = 0; c < 64; c += 32) {
            uint32_t v0[32], v1[32], wv[16];
            if (has0) tmem_ld32(t_lane + 256u + (uint32_t)(a0 * 64 + c), v0);
            if (has1) tmem_ld32(t_lane + 256u + (uint32_t)(a1 * 64 + c), v1);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float x0 = (has0 ? __uint_as_float(v0[2 * j]) * g0 : 0.f) + (has1 ? __uint_as_float(v1[2 * j]) * g1 : 0.f);
              float x1 = (has0 ? __uint_as_float(v0[2 * j + 1]) * g0 : 0.f) + (has1 ? __uint_as_float(v1[2 * j + 1]) * g1 : 0.f);
              if (edge) {
                const float2 ve = *reinterpret_cast<const float2*>(vedge + c + 2 * j);  // broadcast read
                x0 = fmaf(ge, ve.x, x0);
                x1 = fmaf(ge, ve.y, x1);
              }
              wv[j] = pack_bf2(x0, x1);
            }
            if (row < Tp) { st256g(dst + c, wv); st256g(dst + c + 16, wv + 8); }
          }
          if (row < Tp) p.lse[((long long)n * heads + h) * T + row] = M * (1.f / LOG2E_F) + logf(L);
        }
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (has0) mbar_arrive(bars.accfree(a0));
          if (has1) mbar_arrive(bars.accfree(a1));
        }
        if (has0) euse = (euse & ~(15u << (4 * a0))) | (((u0 + 1u) & 15u) << (4 * a0));
        if (has1) euse = (euse & ~(15u << (4 * a1))) | (((u1 + 1u) & 15u) << (4 * a1));
        TRF(warp, tile, 1);
        if (tile == 0 && w + (int)gridDim.x < nitems) {
          TRF(warp, 61, 0);
          edge_a(w + gridDim.x, it + 1, nse0, nse1);
          edge_b(w + gridDim.x, it + 1);
          TRF(warp, 61, 1);
        }
      }
      se0 = nse0;
      se1 = nse1;
      TRF(warp, 62, 1);
      TRI(warp, 1);
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------ backward (persistent)
// Same organisation as the forward: one CTA per SM walks the (image, head) items; the block stream, the TMEM / staging buffers and all
// mbarrier phases run across items, so the epilogue of an item's last tile, the edge-token work and the TMEM hand-over overlap the
// next item.  The four operands (Q, K, V, dO: 4 x 34 KB for T = 257) are single buffered -- all of them are read until the item's last
// MMAs -- so the next item's loads start when those have completed (one TMA round trip per item instead of a CTA launch, barrier and
// TMEM set-up, constant loads and a serial epilogue: 13 000 of 61 000 cycles per item before).
//
//   phase A (lane = query):  S = Q K^T, dP = dO V^T, dS = P (dP - delta) scale, dQ += dS K
//   phase B (lane = key):    S^T = K Q^T, dP^T = V dO^T, dV += P^T dO, dK += dS^T Q
//   P is recomputed from the saved log-sum-exp; two orientations instead of a transposed smem operand, no atomics, deterministic.
//
//   warp 0   S (S^T) MMAs            warp 1   dP (dP^T) MMAs         warp 2   dQ | dV MMAs       warp 3   dK MMAs + TMA producer
//   warps 4-11   two softmax warpgroups (block gg -> warpgroup gg & 1, staging buffer gg & 1)      warps 12-15   epilogue + edge token
//   TMEM: S | dP buffers 3 x (64 + 64) columns [0, 384); dQ slots 0 / 1 at 384 + 64 (tile & 1); phase B: dV at 384, dK at 448 (slot 2,
//   overlaying the dQ slots: the issuers wait until the epilogue has drained them).
//
// Edge token (T = 64 m + 1, e = T - 1): the pipeline covers the first Tp = T - 1 queries and keys.  The epilogue warps compute on CUDA
// cores  column e:  p_ie, dS_ie (all queries i)   and   row e:  p_ej, dS_ej (all keys j)   from four 64-long dot products per index,
// then  dQ_e = sum_j dS_ej K_j,  dK_e = sum_i dS_ie Q_i,  dV_e = sum_i p_ie dO_i  and, when they write a tile,
//   dQ_i += dS_ie K_e        dK_j += dS_ej Q_e        dV_j += p_ej dO_e.
struct BBars {
  uint32_t base;
  __device__ __forceinline__ uint32_t sfull(int b) const { return base + 8u * b; }                // S and dP block in TMEM buffer b     (2 x tcgen05.commit)
  __device__ __forceinline__ uint32_t sfree(int b) const { return base + 24u + 8u * b; }          // its warpgroup has read it           (4 warps)
  __device__ __forceinline__ uint32_t pready(int pb) const { return base + 48u + 8u * pb; }       // staging buffer pb is written        (4 warps)
  __device__ __forceinline__ uint32_t pfree(int pb) const { return base + 64u + 8u * pb; }        // accumulator MMAs have consumed it   (2 issuers)
  __device__ __forceinline__ uint32_t accfull(int a) const { return base + 80u + 8u * a; }        // accumulator slot a is complete      (2 issuers)
  __device__ __forceinline__ uint32_t accfree(int a) const { return base + 104u + 8u * a; }       // epilogue has read it                (4 warps)
  __device__ __forceinline__ uint32_t op(int o, int blk) const { return base + 128u + 8u * (o * MAX_BLK + blk); }  // operand o (Q, K, V, dO), 64-row block (TMA)
  __device__ __forceinline__ uint32_t opfree() const { return base + 288u; }                      // the item's operands are no longer read (4 issuers + 4 epilogue warps)
  __device__ __forceinline__ uint32_t cready(int par) const { return base + 296u + 8u * par; }    // per-token constants of an item are in smem (4 warps)
  __device__ __forceinline__ uint32_t tmem_slot() const { return base + 312u; }
};
constexpr uint32_t BBARS_BYTES = 320 + 16;
// float scratch: constants [2][640] (-lse log2e [320], -scale delta [320]); edge vectors [4][288] (p_ie, dS_ie, p_ej, dS_ej); K_e, Q_e, dO_e as
// floats [3][64]; partial sums [3][4][32] float2
constexpr uint32_t BWD_FLOATS = 1280 + 1152 + 192 + 768;

#ifdef CG_ATTN_TRACE
#define TRB(slot, idx, ev) TRF(slot, idx, ev)
#else
#define TRB(slot, idx, ev) do { } while (0)
#endif

// 64 fp32 accumulator values of one row + coef * vec[0..64) -> 64 bf16 = 128 contiguous bytes (vec: broadcast reads from shared memory)
__device__ __forceinline__ void store_row64_bf16_axpy(__nv_bfloat16* dst, const uint32_t* a, const uint32_t* b, float coef, const float* vec) {
  uint32_t w[32];
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const float2 v0 = *reinterpret_cast<const float2*>(vec + 2 * j), v1 = *reinterpret_cast<const float2*>(vec + 32 + 2 * j);
    w[j] = pack_bf2(fmaf(coef, v0.x, __uint_as_float(a[2 * j])), fmaf(coef, v0.y, __uint_as_float(a[2 * j + 1])));
    w[16 + j] = pack_bf2(fmaf(coef, v1.x, __uint_as_float(b[2 * j])), fmaf(coef, v1.y, __uint_as_float(b[2 * j + 1])));
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) st256g(dst + 16 * j, w + 8 * j);
}

__global__ void __launch_bounds__(AT_THREADS, 1)
    attn_bwd_tc_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmQKVtail, const __grid_constant__ CUtensorMap tmDO,
                       const __grid_constant__ CUtensorMap tmDOtail, const AttnParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  cg_griddep_launch();
  constexpr int NSB = 3;
  constexpr uint32_t STAGE_BYTES = 2 * TILE_BYTES;  // phase B stages P^T and dS^T
  const int T = p.T, heads = p.heads, D = heads * 64;
  const int edge = p.edge, Tp = T - edge;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ntiles = p.ntiles, nblk = p.nblk, nblk_ld = p.nblk_ld;
  const int per_phase = ntiles * nblk, G = 2 * per_phase, nitems = p.nitems;
  const uint32_t opb = (uint32_t)((nblk_ld - 1) * 64 + p.ld_tail) * 128u;  // bytes per operand buffer (multiple of 2048)
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sOp0 = base;                                   // operands 0 = Q, 1 = K, 2 = V, 3 = dO
  const uint32_t sStage = base + 4 * opb;                       // 2 x 32 KB; also absorbs the A-operand over-read of the last tile
  const uint32_t sF = sStage + 2 * STAGE_BYTES;
  float* fscr = reinterpret_cast<float*>(smem_raw + (sF - smem_u32(smem_raw)));
  float* csts = fscr;          // [2][640]
  float* ev = fscr + 1280;     // [4][288]
  float* evec = fscr + 2432;   // [3][64]: K_e, Q_e, dO_e
  float* epart = fscr + 2624;  // [3][4][32] float2
  BBars bars{sF + BWD_FLOATS * 4};

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQKV) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQKVtail) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmDO) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmDOtail) : "memory");
    for (int b = 0; b < 3; ++b) {
      mbar_init(bars.sfull(b), 2); mbar_init(bars.sfree(b), 4);
      mbar_init(bars.accfull(b), 2); mbar_init(bars.accfree(b), 4);
    }
    for (int b = 0; b < 2; ++b) { mbar_init(bars.pready(b), 4); mbar_init(bars.pfree(b), 2); mbar_init(bars.cready(b), 4); }
    for (int o = 0; o < 4; ++o)
      for (int k = 0; k < MAX_BLK; ++k) mbar_init(bars.op(o, k), 1);
    mbar_init(bars.opfree(), 8);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(bars.tmem_slot()), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  cg_griddep_wait();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(bars.tmem_slot()) : "memory");

  if (warp < 4) {
    // ================= four MMA issuer warps (warp-converged loops, elected lane); warp 3 is also the TMA producer
    const uint32_t elected = elect_one();
    const uint32_t id_full = idesc_bf16(128, 64, false), id_tail = idesc_bf16(128, p.tail_rows, false), id_acc = idesc_bf16(128, 64, true);
    uint32_t cuse = 0;  // accumulator issuers: bit a = parity of the number of uses of slot a issued so far
    int it = 0, gg0 = 0;
    for (int w = blockIdx.x; w < nitems; w += gridDim.x, ++it, gg0 += G) {
      const uint32_t opar = (uint32_t)it & 1u;
      uint32_t loaded = 0;  // operand blocks already seen complete (bit o * MAX_BLK + blk)
      auto need = [&](int o, int blk) {
        const uint32_t bit = 1u << (o * MAX_BLK + blk);
        if (!(loaded & bit)) { mbar_wait(bars.op(o, blk), opar); loaded |= bit; }
      };
      if (warp == 3) {
        if (elected) {
          // ---- TMA producer: every operand block of the item once, in the order phase A needs them
          if (it > 0) mbar_wait(bars.opfree(), (uint32_t)(it - 1) & 1u);  // nobody reads the previous item's operands any more
          const int n = w / heads, h = w - n * heads, row0 = n * T;
          auto load = [&](int o, int blk) {
            const bool tail = blk == nblk_ld - 1;
            const uint32_t bar = bars.op(o, blk);
            mbar_arrive_expect_tx(bar, (uint32_t)(tail ? p.ld_tail : 64) * 128u);
            if (o < 3) tma_load_2d(sOp0 + o * opb + blk * BLK_BYTES, tail ? &tmQKVtail : &tmQKV, bar, o * D + h * 64, row0 + blk * 64);
            else tma_load_2d(sOp0 + o * opb + blk * BLK_BYTES, tail ? &tmDOtail : &tmDO, bar, h * 64, row0 + blk * 64);
          };
          const int first = nblk_ld < 2 ? nblk_ld : 2;
          load(1, 0);
#pragma unroll 1
          for (int k = 0; k < first; ++k) load(0, k);
          load(2, 0);
#pragma unroll 1
          for (int k = 0; k < first; ++k) load(3, k);
#pragma unroll 1
          for (int k = 1; k < nblk_ld; ++k) { load(1, k); load(2, k); }
#pragma unroll 1
          for (int k = first; k < nblk_ld; ++k) { load(0, k); load(3, k); }
          // single-buffered operands: the next item's loads cannot be issued before this item is finished -- pull its tiles into L2 now
          if (w + (int)gridDim.x < nitems) {
            const int w2 = w + gridDim.x, n2 = w2 / heads, h2 = w2 - n2 * heads;
#pragma unroll 1
            for (int k = 0; k < nblk_ld; ++k) {
              const bool tail = k == nblk_ld - 1;
#pragma unroll 1
              for (int o = 0; o < 3; ++o) tma_prefetch_2d(tail ? &tmQKVtail : &tmQKV, o * D + h2 * 64, n2 * T + k * 64);
              tma_prefetch_2d(tail ? &tmDOtail : &tmDO, h2 * 64, n2 * T + k * 64);
            }
          }
        }
        __syncwarp();
      }
      int phase = 0, tile = 0, blk = 0;
      if (warp < 2) {
        // ---- S-type MMAs: D[128 x ncols] = A_tile[128 x 64] . B_blk[ncols x 64]^T, 4 k-steps of 16.  warp 0: S = Q K^T (S^T = K Q^T);
        // warp 1: dP = dO V^T (dP^T = V dO^T)
        for (int g = 0; g < G; ++g) {
          const int gg = gg0 + g, b = gg % NSB;
          const bool transposed = phase == 1;
          const int oa = warp == 0 ? (transposed ? 1 : 0) : (transposed ? 2 : 3);
          const int ob = warp == 0 ? (transposed ? 0 : 1) : (transposed ? 3 : 2);
          need(oa, 2 * tile);
          if (2 * tile + 1 < nblk) need(oa, 2 * tile + 1);
          need(ob, blk);
          mbar_wait(bars.sfree(b), ((uint32_t)(gg / NSB) & 1u) ^ 1u);
          TRB(warp, g, 0);
          tcgen05_fence_after();
          const uint32_t d_s = tmem_base + (uint32_t)(b * 128) + (warp == 1 ? 64u : 0u);
          const uint64_t ad = make_smem_desc(sOp0 + oa * opb + tile * TILE_BYTES), bd = make_smem_desc(sOp0 + ob * opb + blk * BLK_BYTES);
          const uint32_t idesc = blk == nblk - 1 ? id_tail : id_full;
          if (elected) {
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16(d_s, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, k != 0 ? 1u : 0u);
            umma_commit(bars.sfull(b));
          }
          __syncwarp();
          TRB(warp, g, 1);
          if (++blk == nblk) { blk = 0; if (++tile == ntiles) { tile = 0; ++phase; } }
        }
      } else {
        // ---- accumulator MMAs of the staged blocks: D[128 x 64] += A_stage[128 x ncols] . B_blk[ncols x 64] (B in MN-major form)
        // warp 2: dQ += dS K (phase A), dV += P^T dO (phase B); warp 3: dK += dS^T Q (phase B), plain arrivals in phase A
        const int wi = warp - 2;
        for (int g = 0; g < G; ++g) {
          const int gg = gg0 + g, pb = gg & 1;
          const int a = phase == 1 ? 2 : (tile & 1);
          const bool does_mma = phase == 1 || wi == 0;
          const int ob = phase == 0 ? 1 : (wi == 0 ? 3 : 0);
          if (does_mma) need(ob, blk);
          mbar_wait(bars.pready(pb), (uint32_t)(gg >> 1) & 1u);
          TRB(warp, g, 0);
          if (blk == 0) {
            // the slot's previous use must have been read by the epilogue.  Slot 2 (dV | dK) overlays the two dQ slots: phase B waits for
            // the latest use of both of them, phase A for the latest use of slot 2 (the previous item's last tile).
            if (phase == 1) {
              mbar_wait(bars.accfree(2), ((cuse >> 2) & 1u) ^ 1u);
              if (tile == 0) { mbar_wait(bars.accfree(0), (cuse & 1u) ^ 1u); mbar_wait(bars.accfree(1), ((cuse >> 1) & 1u) ^ 1u); }
            } else {
              mbar_wait(bars.accfree(a), ((cuse >> a) & 1u) ^ 1u);
              mbar_wait(bars.accfree(2), ((cuse >> 2) & 1u) ^ 1u);
            }
          }
          tcgen05_fence_after();
          const int ksteps = (blk == nblk - 1 ? p.tail_rows : 64) >> 4;
          const uint32_t stage = sStage + pb * STAGE_BYTES + (wi == 1 ? TILE_BYTES : 0u);  // warp 3: dS^T (second staged tile)
          const uint32_t d_acc = tmem_base + (a == 2 ? 384u : 384u + 64u * a) + (wi == 1 ? 64u : 0u);
          const uint64_t ad = make_smem_desc(stage), bd = make_smem_desc(sOp0 + ob * opb + blk * BLK_BYTES);
          const bool last = blk == nblk - 1;
          if (elected) {
            if (does_mma) {
              for (int k = 0; k < ksteps; ++k) umma_bf16(d_acc, ad + (uint64_t)(2 * k), bd + (uint64_t)(128 * k), id_acc, (blk | k) != 0 ? 1u : 0u);
              umma_commit(bars.pfree(pb));
              if (last) umma_commit(bars.accfull(a));
            } else {  // phase A, warp 3: nothing to multiply, keep the two-arrival barriers in step
              mbar_arrive(bars.pfree(pb));
              if (last) mbar_arrive(bars.accfull(a));
            }
          }
          __syncwarp();
          TRB(warp, g, 1);
          if (last) cuse ^= 1u << a;
          if (++blk == nblk) { blk = 0; if (++tile == ntiles) { tile = 0; ++phase; } }
        }
      }
      // observe every phase of every operand barrier (a parity wait is only sound then), then release the operands: the arrival fires
      // when all MMAs this warp has issued so far have completed
#pragma unroll 1
      for (int o = 0; o < 4; ++o)
#pragma unroll 1
        for (int k = 0; k < nblk_ld; ++k) need(o, k);
      if (elected) umma_commit(bars.opfree());
      __syncwarp();
    }
  } else if (warp < 12) {
    // ================= softmax warpgroups: block gg belongs to warpgroup gg & 1 (G is even: g & 1); thread = one row (TMEM lane) of the tile
    const int wg = (warp - 4) >> 2;
    const int q = warp & 3;
    const int rl = q * 32 + lane;  // row inside the 128-row tile
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    const float scale = p.scale, sl2 = p.scale * LOG2E_F;
    const int tail_cols = Tp - (nblk - 1) * 64, tail_cols16 = p.tail_rows;
    const uint32_t sx = (uint32_t)(rl & 7) << 4;  // 128B swizzle of this thread's row of a staged tile: 16-byte chunk c sits at (c << 4) ^ sx
    int it = 0, gg0 = 0;
    for (int w = blockIdx.x; w < nitems; w += gridDim.x, ++it, gg0 += G) {
      mbar_wait(bars.cready(it & 1), (uint32_t)(it >> 1) & 1u);
      const float* cst = csts + (it & 1) * 640;  // [0, 320): -lse log2e (-inf beyond T), [320, 640): -scale delta
      float rc0 = 0.f, rc1 = 0.f;  // phase A: -lse * log2e and delta of this thread's query row
      int phase = 0, tile = 0, blk = wg, cur_tile = -1;
      while (blk >= nblk) { blk -= nblk; if (++tile == ntiles) { tile = 0; ++phase; } }
      for (int g = wg; g < G; g += 2) {
        const int gg = gg0 + g;
        if (phase == 0 && tile != cur_tile) {
          const int row = tile * 128 + rl;
          rc0 = row < Tp ? cst[row] : 0.f;
          rc1 = row < Tp ? cst[320 + row] : 0.f;  // -scale delta: dS = P (scale dP - scale delta) is one FFMA + one FMUL per element
          cur_tile = tile;
        }
        const bool wvalid = tile * 128 + q * 32 < Tp;  // warp-uniform: this warp has at least one real row
        const bool tail = blk == nblk - 1;
        const int ncols = tail ? tail_cols : 64, ncols16 = tail ? tail_cols16 : 64;
        const int b = gg % NSB, pb = gg & 1;
        const uint32_t suse = (uint32_t)(gg / NSB), puse = (uint32_t)(gg >> 1);
        TRB(warp, g, 0);
        mbar_wait(bars.sfull(b), suse & 1u);
        TRB(warp, g, 1);
        tcgen05_fence_after();
        const uint32_t t_s = t_lane + (uint32_t)(b * 128);
        const uint32_t stage = sStage + pb * STAGE_BYTES + (uint32_t)rl * 128u;
        if (!wvalid) {
          tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bars.sfree(b));
          // a warp without real rows stages nothing, but it must not run ahead of the barrier phases: its pready arrival for this use
          // may only happen once the previous use of the staging buffer has been consumed (otherwise early arrivals of LATER blocks
          // complete the current phase before the warp that does have rows has written its data)
          mbar_wait(bars.pfree(pb), (puse & 1u) ^ 1u);
        } else {
          // S and dP in 16-column pieces, the loads of piece i+1 in flight while piece i is processed
          uint32_t sv[2][16], dv[2][16], w0[8], w1[8];
          const int npieces = ncols16 >> 4;
          tmem_ld16(t_s, sv[0]);
          tmem_ld16(t_s + 64u, dv[0]);
          tmem_ld_wait();
          bool waited = false;
#pragma unroll
          for (int pc = 0; pc < 4; ++pc) {
            if (pc < npieces) {
              const int cur = pc & 1;
              if (pc + 1 < npieces) {
                tmem_ld16(t_s + (uint32_t)(16 * (pc + 1)), sv[cur ^ 1]);
                tmem_ld16(t_s + 64u + (uint32_t)(16 * (pc + 1)), dv[cur ^ 1]);
              }
              if (phase == 0) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  float p0 = ex2f(fmaf(__uint_as_float(sv[cur][2 * j]), sl2, rc0)), p1 = ex2f(fmaf(__uint_as_float(sv[cur][2 * j + 1]), sl2, rc0));
                  if (tail) { if (16 * pc + 2 * j >= ncols) p0 = 0.f; if (16 * pc + 2 * j + 1 >= ncols) p1 = 0.f; }
                  w0[j] = pack_bf2(p0 * fmaf(__uint_as_float(dv[cur][2 * j]), scale, rc1), p1 * fmaf(__uint_as_float(dv[cur][2 * j + 1]), scale, rc1));
                }
              } else {
                const float* nl = cst + blk * 64 + 16 * pc;  // per-query constants: broadcast reads
                const float* dl = nl + 320;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const float2 l2 = *reinterpret_cast<const float2*>(nl + 2 * j), d2 = *reinterpret_cast<const float2*>(dl + 2 * j);
                  float p0 = ex2f(fmaf(__uint_as_float(sv[cur][2 * j]), sl2, l2.x)), p1 = ex2f(fmaf(__uint_as_float(sv[cur][2 * j + 1]), sl2, l2.y));
                  if (tail) { if (16 * pc + 2 * j >= ncols) p0 = 0.f; if (16 * pc + 2 * j + 1 >= ncols) p1 = 0.f; }
                  w0[j] = pack_bf2(p0, p1);
                  w1[j] = pack_bf2(p0 * fmaf(__uint_as_float(dv[cur][2 * j]), scale, d2.x), p1 * fmaf(__uint_as_float(dv[cur][2 * j + 1]), scale, d2.y));
                }
              }
              if (!waited) { mbar_wait(bars.pfree(pb), (puse & 1u) ^ 1u); waited = true; }  // staging buffer free again
              {
                const uint32_t c0 = ((uint32_t)(pc * 32)) ^ sx, c1 = ((uint32_t)(pc * 32 + 16)) ^ sx;
                st_shared_v4(stage + c0, w0[0], w0[1], w0[2], w0[3]);
                st_shared_v4(stage + c1, w0[4], w0[5], w0[6], w0[7]);
                if (phase == 1) {
                  st_shared_v4(stage + TILE_BYTES + c0, w1[0], w1[1], w1[2], w1[3]);
                  st_shared_v4(stage + TILE_BYTES + c1, w1[4], w1[5], w1[6], w1[7]);
                }
              }
              if (pc + 1 < npieces) {
                tmem_ld_wait();
              } else {  // every TMEM read of this block has completed (the wait of the previous piece covered this one's loads)
                tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bars.sfree(b));
              }
            }
          }
        }
        TRB(warp, g, 2);
        fence_proxy_async_smem();  // generic-proxy writes of the staged operand -> visible to the tensor core (async proxy)
        __syncwarp();
        if (lane == 0) mbar_arrive(bars.pready(pb));
        TRB(warp, g, 3);
        blk += 2;
        while (blk >= nblk) { blk -= nblk; if (++tile == ntiles) { tile = 0; ++phase; } }
      }
    }
  } else {
    // ================= epilogue warps: per-token constants, edge token, finished accumulator tiles -> HBM
    const int q = warp & 3;
    const int rl = q * 32 + lane;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    const float scale = p.scale, sl2 = p.scale * LOG2E_F;
    uint32_t euse = 0;  // bit a: parity of the use count of accumulator slot a
    auto load_consts = [&](int item, int par) {
      // per-token constants of an item: -lse log2e, and delta_i = sum_d dO_i[d] O_i[d] straight from the two global tensors (the
      // separate row-dot-product kernel cost 24 us per layer; these warps have the slack)
      const int n = item / heads, h = item - n * heads;
      const float* lb = p.lse + ((long long)n * heads + h) * T;
      const __nv_bfloat16* ob = p.ctx_in + ((long long)n * T) * D + h * 64;
      const __nv_bfloat16* gb = p.dctx_in + ((long long)n * T) * D + h * 64;
      float* c = csts + par * 640;
      for (int i = rl; i < 320; i += 128) {
        float dl = 0.f, nl = -INFINITY;
        if (i < T) {
          const uint4* o4 = reinterpret_cast<const uint4*>(ob + (long long)i * D);
          const uint4* g4 = reinterpret_cast<const uint4*>(gb + (long long)i * D);
          uint4 xo[8], xg[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) { xo[k] = __ldg(o4 + k); xg[k] = __ldg(g4 + k); }
          float d0 = 0.f, d1 = 0.f;
#pragma unroll
          for (int k = 0; k < 8; k += 2) { d0 = dot8p(xo[k], xg[k], d0); d1 = dot8p(xo[k + 1], xg[k + 1], d1); }
          dl = d0 + d1;
          nl = -lb[i] * LOG2E_F;
        }
        c[i] = nl;
        c[320 + i] = -p.scale * dl;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bars.cready(par));
    };
    if ((int)blockIdx.x < nitems) load_consts(blockIdx.x, 0);
    int it = 0;
    for (int w = blockIdx.x; w < nitems; w += gridDim.x, ++it) {
      const int n = w / heads, h = w - n * heads, row0 = n * T;
      const uint32_t opar = (uint32_t)it & 1u;
      // constants of the NEXT item (its buffer was last read by item it - 1, whose tiles this role has already finished)
      if (w + (int)gridDim.x < nitems) load_consts(w + gridDim.x, (it + 1) & 1);
      const float* cst = csts + (it & 1) * 640;
      __nv_bfloat16* out = p.dqkv + ((long long)row0) * 3 * D + h * 64;  // row r of this item: + r * 3D; dQ at +0, dK at +D, dV at +2D
      TRB(warp, 62, 0);
      TRI(warp, 0);
      if (edge) {
        for (int o = 0; o < 4; ++o)
          for (int k = 0; k < nblk_ld; ++k) mbar_wait(bars.op(o, k), opar);
        mbar_wait(bars.cready(it & 1), (uint32_t)(it >> 1) & 1u);  // (this role wrote them, but not necessarily this warp)
        TRB(warp, 61, 0);
        const uint32_t sQ = sOp0, sK = sOp0 + opb, sV = sOp0 + 2 * opb, sDO = sOp0 + 3 * opb;
        const float nle = cst[Tp], dle = cst[320 + Tp];  // (-scale delta_e)
        const int g = lane >> 2, t = lane & 3;
        {
          // column e (key e against every query i: Q k_e, dO v_e) and row e (query e against every key i: K q_e, V dO_e) as warp-level MMAs
          uint32_t vbk[8], vbv[8], vbq[8], vbd[8];
          load_vec_bfrag(sK, Tp, vbk);
          load_vec_bfrag(sV, Tp, vbv);
          load_vec_bfrag(sQ, Tp, vbq);
          load_vec_bfrag(sDO, Tp, vbd);
#pragma unroll 1
          for (int rg = q; rg < (Tp >> 4); rg += 4) {
            const float2 s_c = mv16(sQ, rg * 16, vbk), dp_c = mv16(sDO, rg * 16, vbv), s_r = mv16(sK, rg * 16, vbq), dp_r = mv16(sV, rg * 16, vbd);
            if (t == 0) {
#pragma unroll
              for (int hh = 0; hh < 2; ++hh) {
                const int i = rg * 16 + g + 8 * hh;
                const float p_c = ex2f(fmaf(hh ? s_c.y : s_c.x, sl2, cst[i]));
                ev[i] = p_c;
                ev[288 + i] = p_c * fmaf(hh ? dp_c.y : dp_c.x, scale, cst[320 + i]);
                const float p_r = ex2f(fmaf(hh ? s_r.y : s_r.x, sl2, nle));
                ev[576 + i] = p_r;
                ev[864 + i] = p_r * fmaf(hh ? dp_r.y : dp_r.x, scale, dle);
              }
            }
          }
        }
        {  // corner (e, e): every warp computes it redundantly (row Tp of an operand is not permuted by the swizzle: Tp % 8 == 0)
          const uint32_t eo = (uint32_t)Tp * 128u + (uint32_t)lane * 4u;
          const uint32_t wq = lds32(sQ + eo), wk = lds32(sK + eo), wv = lds32(sV + eo), wd = lds32(sDO + eo);
          const float s_e = warp_sum(fmaf(bf_lo(wq), bf_lo(wk), bf_hi(wq) * bf_hi(wk)));
          const float dp_e = warp_sum(fmaf(bf_lo(wd), bf_lo(wv), bf_hi(wd) * bf_hi(wv)));
          const float p_e = ex2f(fmaf(s_e, sl2, nle)), ds_e = p_e * fmaf(dp_e, scale, dle);
          if (rl == 0) { ev[Tp] = p_e; ev[288 + Tp] = ds_e; ev[576 + Tp] = p_e; ev[864 + Tp] = ds_e; }
          if (rl >= 1 && rl < 16) { ev[Tp + rl] = 0.f; ev[288 + Tp + rl] = 0.f; ev[576 + Tp + rl] = 0.f; ev[864 + Tp + rl] = 0.f; }  // pad the last 16-group
          if (q == 0) {  // K_e, Q_e, dO_e as floats for the tile corrections
            evec[2 * lane] = bf_lo(wk); evec[2 * lane + 1] = bf_hi(wk);
            evec[64 + 2 * lane] = bf_lo(wq); evec[64 + 2 * lane + 1] = bf_hi(wq);
            evec[128 + 2 * lane] = bf_lo(wd); evec[128 + 2 * lane + 1] = bf_hi(wd);
          }
        }
        asm volatile("bar.sync 2, 128;" ::: "memory");
        {
          // dQ_e = sum_j dS_ej K_j, dK_e = sum_i dS_ie Q_i, dV_e = sum_i p_ie dO_i over all T tokens: warp q takes the 16-token groups
          // ks = q (mod 4); lanes 0-3 hold the partial results
          const int ngrp = (Tp >> 4) + 1;
#pragma unroll 1
          for (int pr = 0; pr < 3; ++pr) {
            const uint32_t buf = pr == 0 ? sK : (pr == 1 ? sQ : sDO);
            const float* vec = ev + (pr == 0 ? 864 : (pr == 1 ? 288 : 0));
            float acc[8][4];
#pragma unroll
            for (int nn = 0; nn < 8; ++nn) acc[nn][0] = acc[nn][1] = acc[nn][2] = acc[nn][3] = 0.f;
#pragma unroll 1
            for (int ks = q; ks < ngrp; ks += 4) vm16(buf, ks * 16, vec, acc);
            if (lane < 4) {
#pragma unroll
              for (int nn = 0; nn < 8; ++nn) *reinterpret_cast<float2*>(epart + (pr * 4 + q) * 64 + 8 * nn + 2 * t) = make_float2(acc[nn][0], acc[nn][1]);
            }
          }
          asm volatile("bar.sync 2, 128;" ::: "memory");
          if (q < 3) {  // warp 0: dQ_e, warp 1: dK_e, warp 2: dV_e
            const float* pp = epart + q * 256 + 2 * lane;
            const float2 x0 = *reinterpret_cast<const float2*>(pp), x1 = *reinterpret_cast<const float2*>(pp + 64);
            const float2 x2 = *reinterpret_cast<const float2*>(pp + 128), x3 = *reinterpret_cast<const float2*>(pp + 192);
            reinterpret_cast<uint32_t*>(out + (long long)Tp * 3 * D + q * D)[lane] = pack_bf2((x0.x + x1.x) + (x2.x + x3.x), (x0.y + x1.y) + (x2.y + x3.y));
          }
        }
        TRB(warp, 61, 1);
      }
      // this role no longer reads the item's operands from shared memory
      __syncwarp();
      if (lane == 0) mbar_arrive(bars.opfree());
      for (int tc = 0; tc < 2 * ntiles; ++tc) {
        const int phase = tc >= ntiles ? 1 : 0, tile = tc - phase * ntiles;
        const int a = phase == 1 ? 2 : (tile & 1);
        const int row = tile * 128 + rl;
        mbar_wait(bars.accfull(a), (euse >> a) & 1u);
        TRB(warp, tc, 0);
        tcgen05_fence_after();
        if (tile * 128 + q * 32 < Tp) {
          uint32_t v0[32], v1[32];
          const uint32_t col = a == 2 ? 384u : 384u + 64u * a;
          tmem_ld32(t_lane + col, v0);
          tmem_ld32(t_lane + col + 32u, v1);
          tmem_ld_wait();
          __nv_bfloat16* orow = out + (long long)row * 3 * D;
          if (phase == 0) {
            if (row < Tp) {
              if (edge) store_row64_bf16_axpy(orow, v0, v1, ev[288 + row], evec);            // dQ_i += dS_ie K_e
              else store_row64_bf16(orow, v0, v1, 1.f);
            }
          } else {
            if (row < Tp) {
              if (edge) store_row64_bf16_axpy(orow + 2 * D, v0, v1, ev[576 + row], evec + 128);  // dV_j += p_ej dO_e
              else store_row64_bf16(orow + 2 * D, v0, v1, 1.f);
            }
            tmem_ld32(t_lane + col + 64u, v0);
            tmem_ld32(t_lane + col + 96u, v1);
            tmem_ld_wait();
            if (row < Tp) {
              if (edge) store_row64_bf16_axpy(orow + D, v0, v1, ev[864 + row], evec + 64);       // dK_j += dS_ej Q_e
              else store_row64_bf16(orow + D, v0, v1, 1.f);
            }
          }
        }
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bars.accfree(a));
        euse ^= 1u << a;
        TRB(warp, tc, 1);
      }
      TRB(warp, 62, 1);
      TRI(warp, 1);
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

long long* g_trace = nullptr;

// Parameters and pipeline / load geometry of one launch.  T = 64 m + 1 (ViT-L/14: 16 x 16 patches + class token = 257): the non-causal
// kernels take the LAST token out of the tensor-core pipeline ("edge"), which then sees only full 64-wide blocks and full 128-row tiles.
void set_geometry(AttnParams& p, int T, int heads, bool causal) {
  p.T = T; p.heads = heads; p.scale = 0.125f;
  p.trace = g_trace;
  p.edge = (!causal && T > 1 && (T - 1) % 64 == 0) ? 1 : 0;
  const int Tp = T - p.edge;
  p.ntiles = (Tp + 127) / 128;
  p.nblk = (Tp + 63) / 64;
  p.tail_rows = ((Tp - (p.nblk - 1) * 64) + 15) & ~15;
  p.nblk_ld = p.nblk + p.edge;
  p.ld_tail = p.edge ? 16 : p.tail_rows;
}

// TMA maps of a [rows, cols] bf16 operand: one for its full 64-row blocks, one for the last block loaded (ld_tail rows)
int make_operand_maps(CUtensorMap& full, CUtensorMap& tail, const void* ptr, long long rows, long long cols, const AttnParams& p) {
  const int rc = cg_make_tensor_map_bf16(&full, ptr, rows, cols, cols, 64);
  return rc ? rc : cg_make_tensor_map_bf16(&tail, ptr, rows, cols, cols, p.ld_tail);
}

// Persistent launch: one CTA per SM walks the Nimg * heads items.  Shared memory: four operand buffers, four staging tiles and
// `extra` bytes of per-kernel data.  The static cache is per instantiation, i.e. per kernel (function attributes are per kernel and device).
template <auto kernel, typename... Maps>
int launch_persistent(AttnParams& p, int Nimg, size_t extra, cudaStream_t s, const Maps&... maps) {
  const size_t opb = (size_t)((p.nblk_ld - 1) * 64 + p.ld_tail) * 128;
  const size_t smem = 1024 + 4 * opb + 4 * (size_t)TILE_BYTES + extra;
  p.nitems = Nimg * p.heads;
  const int grid = p.nitems < cg_num_sms() ? p.nitems : cg_num_sms();
  static size_t configured[CG_MAX_DEVICES] = {};
  const int dev = cg_device_index();
  if (smem > configured[dev]) {
    CG_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured[dev] = smem;
  }
  CG_CUDA(cg_launch_pdl(kernel, dim3(grid), dim3(AT_THREADS), smem, s, maps..., p));
  return 0;
}

template <bool CAUSAL>
int launch_attn_fwd_tc(const void* qkv, int Nimg, int T, int heads, void* ctx, float* lse, cudaStream_t s) {
  AttnParams p = {};
  p.ctx = reinterpret_cast<__nv_bfloat16*>(ctx);
  p.lse = lse;
  set_geometry(p, T, heads, CAUSAL);
  CUtensorMap tq, tqt;
  const int rc = make_operand_maps(tq, tqt, qkv, (long long)Nimg * T, 3LL * heads * 64, p);
  if (rc) return rc;
  return launch_persistent<attn_fwd_tc_kernel<CAUSAL>>(p, Nimg, FWD_FLOATS * 4 + FBARS_BYTES, s, tq, tqt);
}

}  // namespace

int cg_attention_fwd_tc(const void* qkv, int Nimg, int T, int heads, void* ctx, float* lse, cudaStream_t s) {
  return launch_attn_fwd_tc<false>(qkv, Nimg, T, heads, ctx, lse, s);
}

// The CLIP text transformer's attention (OpenAI encode_text, utils/functional.py:91-94): tcgen05 path only, no edge token.
extern "C" int cg_attention_causal_fwd(const void* qkv, int Nseq, int T, int heads, void* ctx, float* lse, void* stream) {
  CG_REQUIRE(qkv && ctx && lse && Nseq > 0 && T > 0 && heads > 0, "cg_attention_causal_fwd: bad arguments");
  CG_REQUIRE(T <= ATTN_TC_MAX_T, "cg_attention_causal_fwd: T=%d exceeds the tcgen05 kernel's limit (%d)", T, ATTN_TC_MAX_T);
  return launch_attn_fwd_tc<true>(qkv, Nseq, T, heads, ctx, lse, cg_stream(stream));
}

int cg_attention_bwd_tc(const void* qkv, const void* ctx, const void* dctx, const float* lse, int Nimg, int T, int heads, void* dqkv, cudaStream_t s) {
  AttnParams p = {};
  p.lse = const_cast<float*>(lse);
  p.ctx_in = reinterpret_cast<const __nv_bfloat16*>(ctx);
  p.dctx_in = reinterpret_cast<const __nv_bfloat16*>(dctx);
  p.dqkv = reinterpret_cast<__nv_bfloat16*>(dqkv);
  set_geometry(p, T, heads, false);
  const int D = heads * 64;
  CUtensorMap tq, tqt, td, tdt;
  int rc = make_operand_maps(tq, tqt, qkv, (long long)Nimg * T, 3LL * D, p);
  if (!rc) rc = make_operand_maps(td, tdt, dctx, (long long)Nimg * T, D, p);
  if (rc) return rc;
  return launch_persistent<attn_bwd_tc_kernel>(p, Nimg, BWD_FLOATS * 4 + BBARS_BYTES, s, tq, tqt, td, tdt);
}

// debug only (tools/trace_attn.py): device buffer of 16 * 64 * 8 int64 that CTA (0,0) of the next launches fills with clock64() stamps
extern "C" void cg_debug_attention_trace(void* buf) { g_trace = reinterpret_cast<long long*>(buf); }
