// Fused multi-head self-attention of the CLIP ViT (head_dim 64, many (cutout, head) problems), forward and dgrad, for the
// sequences too long for the tcgen05 kernels of vit_attention_tc.cu (T > ATTN_TC_MAX_T: ViT-L/14@336, T = 577); the entry
// points below choose between the two from T.  Scores never touch HBM.
//
// Layout: packed qkv [Nimg*T, 3*D] bf16 (q | k | v; head h = columns h*64..h*64+63 of each third).
// One CTA = one (image, head): the whole K/V (forward, dQ) or Q/dO (dK/dV) of that head is loaded into shared
// memory ONCE (<= 640 x 64 bf16 each, XOR-swizzled 16-byte chunks so ldmatrix is conflict free); its W warps walk
// the 16-row tiles of the other operand (tile = warp, warp+W, ...; W chosen per T so that ceil(T/16) tiles fill
// the warps with < 8% idle slots), staging each tile through a private 2 KB buffer and keeping the accumulators in
// registers (mma.sync m16n8k16 bf16, fp32 accumulate).  Ragged tails are skipped at 8-key granularity.
// These are ~5% of the tower's FLOPs; the dense GEMMs run on tcgen05 (vit_gemm.cu).
//
// backward = delta kernel (rowsum dO*O) + dQ kernel (per query block) + dK/dV kernel (per key block): P is
// recomputed from q, k and the saved log-sum-exp; no atomics, deterministic.
#include "common.cuh"
#include "tcgen05.cuh"

namespace {

constexpr int HD = 64;       // head dim
constexpr int MAX_WARPS = 8;
constexpr float LOG2E = 1.4426950408889634f;

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// element (row, col) of a [rows][64] bf16 tile with 16B-chunk XOR swizzle
__device__ __forceinline__ uint32_t swz(int row, int chunk) { return (uint32_t)(row * 128 + ((chunk ^ (row & 7)) << 4)); }

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, bool valid) {
  const int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float c[4], const uint32_t a[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// 2^x in ONE MUFU op (exp2f adds range handling; every softmax element pays it and the kernels are issue bound)
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

// Load `rows` rows (row r = global row row0 + r, valid if < T) x 64 columns starting at `src` (row stride ld) into a
// swizzled smem tile.  All threads participate.
__device__ __forceinline__ void load_tile(uint32_t dst, const __nv_bfloat16* src, long long ld, int row0, int rows, int T) {
  for (int i = threadIdx.x; i < rows * 8; i += blockDim.x) {
    const int r = i >> 3, c = i & 7;
    const bool ok = row0 + r < T;
    cp_async16(dst + swz(r, c), src + (long long)(ok ? row0 + r : 0) * ld + c * 8, ok);
  }
}

// One warp stages a 16-row tile (rows row0..row0+15 of src, zero beyond T) into its private buffer and waits for it.
__device__ __forceinline__ void warp_stage_tile16(uint32_t dst, const __nv_bfloat16* src, long long ld, int row0, int T) {
  const int lane = threadIdx.x & 31;
  __syncwarp();  // every lane is done reading the previous tile
#pragma unroll
  for (int i = lane; i < 128; i += 32) {
    const int r = i >> 3, c = i & 7;
    const bool ok = row0 + r < T;
    cp_async16(dst + swz(r, c), src + (long long)(ok ? row0 + r : 0) * ld + c * 8, ok);
  }
}

// A-operand fragments (16 rows x 64 cols) of rows [r0, r0+16) of a swizzled tile: a[kk][4], kk = 16-col step
__device__ __forceinline__ void load_a_frags(uint32_t tile, int r0, uint32_t a[4][4]) {
  const int lane = threadIdx.x & 31;
  const int row = r0 + (lane & 7) + ((lane >> 3) & 1) * 8;
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) ldsm_x4(tile + swz(row, kk * 2 + (lane >> 4)), a[kk][0], a[kk][1], a[kk][2], a[kk][3]);
}

// B fragments for C[.., n = tile rows n0..n0+7] with k = tile columns (non-transposed: B[k][n] = tile[n][k]).
// Returns b[kk][2] for the 4 k-steps (64 columns).
__device__ __forceinline__ void load_b_frags_nk(uint32_t tile, int n0, uint32_t b[4][2]) {
  const int lane = threadIdx.x & 31;
  const int row = n0 + (lane & 7);
  // matrices: chunk (lane>>3) = columns 8*(lane>>3).. -> regs 0..3 = k 0-7, 8-15, 16-23, 24-31
  uint32_t r0, r1, r2, r3;
  ldsm_x4(tile + swz(row, lane >> 3), r0, r1, r2, r3);
  b[0][0] = r0; b[0][1] = r1; b[1][0] = r2; b[1][1] = r3;
  ldsm_x4(tile + swz(row, 4 + (lane >> 3)), r0, r1, r2, r3);
  b[2][0] = r0; b[2][1] = r1; b[3][0] = r2; b[3][1] = r3;
}

// B fragments for C[.., n = tile columns c0*8..] with k = tile rows k0..k0+15 (transposed: B[k][n] = tile[k][n]).
// One ldmatrix.x4.trans gives (b0,b1) for two adjacent 8-column groups: chunk cpair*2 and cpair*2+1.
__device__ __forceinline__ void load_b_frags_kn(uint32_t tile, int k0, int cpair, uint32_t& b00, uint32_t& b01, uint32_t& b10, uint32_t& b11) {
  const int lane = threadIdx.x & 31;
  const int row = k0 + (lane & 7) + ((lane >> 3) & 1) * 8;
  ldsm_x4_t(tile + swz(row, cpair * 2 + (lane >> 4)), b00, b01, b10, b11);
}

// ---------------------------------------------------------------------------------------------- forward
__global__ void __launch_bounds__(MAX_WARPS * 32) attn_fwd_kernel(const __nv_bfloat16* __restrict__ qkv, int T, int heads, float scale_log2,
                                                                 __nv_bfloat16* __restrict__ ctx, float* __restrict__ lse) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int Tp = (T + 63) & ~63;
  const int D = heads * HD;
  const long long ld = 3LL * D;
  const int h = blockIdx.x, n = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const uint32_t sK = smem_addr(smem), sV = sK + Tp * 128, sQ = sV + Tp * 128 + warp * 2048;
  const __nv_bfloat16* base = qkv + (long long)n * T * ld + h * HD;
  load_tile(sK, base + D, ld, 0, Tp, T);
  load_tile(sV, base + 2 * D, ld, 0, Tp, T);
  cp_async_wait_all();
  __syncthreads();
  const int g = lane >> 2, t4 = lane & 3;
  for (int r0 = warp * 16; r0 < T; r0 += nwarps * 16) {
  warp_stage_tile16(sQ, base, ld, r0, T);
  cp_async_wait_all();
  __syncwarp();
  uint32_t qa[4][4];
  load_a_frags(sQ, 0, qa);
  float o[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;  // rows g and g+8

  for (int kc = 0; kc < Tp; kc += 64) {
    float s[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
      if (kc + nt * 8 < T) {  // ragged tail: whole 8-key tiles beyond T are skipped (warp-uniform)
        uint32_t b[4][2];
        load_b_frags_nk(sK, kc + nt * 8, b);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) mma_bf16(s[nt], qa[kk], b[kk][0], b[kk][1]);
      }
    }
    float mx0 = m0, mx1 = m1;
    if (kc + 64 > T) {  // only the last chunk has keys beyond T (warp-uniform branch)
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const int key = kc + nt * 8 + t4 * 2;
        if (key >= T) { s[nt][0] = -INFINITY; s[nt][2] = -INFINITY; }
        if (key + 1 >= T) { s[nt][1] = -INFINITY; s[nt][3] = -INFINITY; }
      }
    }
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      mx0 = fmaxf(mx0, fmaxf(s[nt][0], s[nt][1]));
      mx1 = fmaxf(mx1, fmaxf(s[nt][2], s[nt][3]));
    }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    const float c0 = ex2((m0 - mx0) * scale_log2), c1 = ex2((m1 - mx1) * scale_log2);
    m0 = mx0; m1 = mx1;
    const float nm0 = -m0 * scale_log2, nm1 = -m1 * scale_log2;
    l0 *= c0; l1 *= c1;
#pragma unroll
    for (int i = 0; i < 8; ++i) { o[i][0] *= c0; o[i][1] *= c0; o[i][2] *= c1; o[i][3] *= c1; }
    uint32_t pa[4][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const float p0 = ex2(fmaf(s[nt][0], scale_log2, nm0)), p1 = ex2(fmaf(s[nt][1], scale_log2, nm0));
      const float p2 = ex2(fmaf(s[nt][2], scale_log2, nm1)), p3 = ex2(fmaf(s[nt][3], scale_log2, nm1));
      l0 += p0 + p1; l1 += p2 + p3;
      pa[nt >> 1][(nt & 1) * 2] = pack2(p0, p1);
      pa[nt >> 1][(nt & 1) * 2 + 1] = pack2(p2, p3);
    }
    // O += P V : k = keys (4 steps of 16), n = d (8 groups of 8)
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      if (kc + kk * 16 >= T) continue;  // P is exactly 0 there
#pragma unroll
      for (int cp = 0; cp < 4; ++cp) {
        uint32_t b00, b01, b10, b11;
        load_b_frags_kn(sV, kc + kk * 16, cp, b00, b01, b10, b11);
        mma_bf16(o[cp * 2], pa[kk], b00, b01);
        mma_bf16(o[cp * 2 + 1], pa[kk], b10, b11);
      }
    }
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const int q0 = r0 + g, q1 = q0 + 8;
  const float i0 = 1.f / l0, i1 = 1.f / l1;
  __nv_bfloat16* cb = ctx + (long long)n * T * D + h * HD;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const int d = nt * 8 + t4 * 2;
    if (q0 < T) *reinterpret_cast<uint32_t*>(cb + (long long)q0 * D + d) = pack2(o[nt][0] * i0, o[nt][1] * i0);
    if (q1 < T) *reinterpret_cast<uint32_t*>(cb + (long long)q1 * D + d) = pack2(o[nt][2] * i1, o[nt][3] * i1);
  }
  if (t4 == 0) {
    float* lb = lse + ((long long)n * heads + h) * T;
    // natural-log LSE of the scaled scores: scale*m + ln(l)
    if (q0 < T) lb[q0] = m0 * scale_log2 / LOG2E + logf(l0);
    if (q1 < T) lb[q1] = m1 * scale_log2 / LOG2E + logf(l1);
  }
  }  // tile loop
}

// ---------------------------------------------------------------------------------------------- backward
// delta[n,h,q] = sum_d dO[q,d] * O[q,d]; one warp per (n, q), all heads
__global__ void __launch_bounds__(256) attn_delta_kernel(const __nv_bfloat16* __restrict__ ctx, const __nv_bfloat16* __restrict__ dctx, int T,
                                                         int heads, long long rows, float* __restrict__ delta) {
  cg_griddep_launch();
  cg_griddep_wait();
  const long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int D = heads * HD;
  const long long n = row / T;
  const int q = (int)(row - n * T);
  for (int h = 0; h < heads; ++h) {
    const uint32_t a = *reinterpret_cast<const uint32_t*>(ctx + row * D + h * HD + lane * 2);
    const uint32_t b = *reinterpret_cast<const uint32_t*>(dctx + row * D + h * HD + lane * 2);
    const __nv_bfloat162 av = *reinterpret_cast<const __nv_bfloat162*>(&a), bv = *reinterpret_cast<const __nv_bfloat162*>(&b);
    float s = __low2float(av) * __low2float(bv) + __high2float(av) * __high2float(bv);
    s = warp_sum(s);
    if (lane == 0) delta[(n * heads + h) * T + q] = s;
  }
}

// dQ: CTA = 64 queries; K, V whole in smem.  dS = P*(dP - delta)*scale;  dQ = dS K.
__global__ void __launch_bounds__(MAX_WARPS * 32) attn_bwd_dq_kernel(const __nv_bfloat16* __restrict__ qkv, const __nv_bfloat16* __restrict__ dctx,
                                                                    const float* __restrict__ lse, const float* __restrict__ delta, int T, int heads,
                                                                    float scale, __nv_bfloat16* __restrict__ dqkv) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int Tp = (T + 63) & ~63;
  const int D = heads * HD;
  const long long ld = 3LL * D;
  const int h = blockIdx.x, n = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const uint32_t sK = smem_addr(smem), sV = sK + Tp * 128, sQ = sV + Tp * 128 + warp * 4096, sdO = sQ + 2048;
  const __nv_bfloat16* base = qkv + (long long)n * T * ld + h * HD;
  const __nv_bfloat16* dbase = dctx + (long long)n * T * D + h * HD;
  load_tile(sK, base + D, ld, 0, Tp, T);
  load_tile(sV, base + 2 * D, ld, 0, Tp, T);
  cp_async_wait_all();
  __syncthreads();
  const int g = lane >> 2, t4 = lane & 3;
  const float* lb = lse + ((long long)n * heads + h) * T;
  const float* db = delta + ((long long)n * heads + h) * T;
  for (int r0 = warp * 16; r0 < T; r0 += nwarps * 16) {
  warp_stage_tile16(sQ, base, ld, r0, T);
  warp_stage_tile16(sdO, dbase, D, r0, T);
  cp_async_wait_all();
  __syncwarp();
  uint32_t qa[4][4], da[4][4];
  load_a_frags(sQ, 0, qa);
  load_a_frags(sdO, 0, da);
  const int q0 = r0 + g, q1 = q0 + 8;
  // P = exp(s*scale - lse) = 2^(s*scale*log2e - lse*log2e): one FFMA + one MUFU per element
  const float sl2 = scale * LOG2E;
  const float lse0 = q0 < T ? -lb[q0] * LOG2E : 0.f, lse1 = q1 < T ? -lb[q1] * LOG2E : 0.f;
  const float dl0 = q0 < T ? db[q0] : 0.f, dl1 = q1 < T ? db[q1] : 0.f;
  float dq[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) dq[i][0] = dq[i][1] = dq[i][2] = dq[i][3] = 0.f;
  for (int kc = 0; kc < Tp; kc += 64) {
    uint32_t dsa[4][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      float s[4] = {0.f, 0.f, 0.f, 0.f}, dp[4] = {0.f, 0.f, 0.f, 0.f};
      if (kc + nt * 8 < T) {
        uint32_t bk[4][2], bv[4][2];
        load_b_frags_nk(sK, kc + nt * 8, bk);
        load_b_frags_nk(sV, kc + nt * 8, bv);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) { mma_bf16(s, qa[kk], bk[kk][0], bk[kk][1]); mma_bf16(dp, da[kk], bv[kk][0], bv[kk][1]); }
      }
      float p0 = ex2(fmaf(s[0], sl2, lse0)), p1 = ex2(fmaf(s[1], sl2, lse0));
      float p2 = ex2(fmaf(s[2], sl2, lse1)), p3 = ex2(fmaf(s[3], sl2, lse1));
      if (kc + 64 > T) {  // keys beyond T exist only in the last chunk
        const int key = kc + nt * 8 + t4 * 2;
        if (key >= T) { p0 = 0.f; p2 = 0.f; }
        if (key + 1 >= T) { p1 = 0.f; p3 = 0.f; }
      }
      p0 *= scale; p1 *= scale; p2 *= scale; p3 *= scale;
      dsa[nt >> 1][(nt & 1) * 2] = pack2(p0 * (dp[0] - dl0), p1 * (dp[1] - dl0));
      dsa[nt >> 1][(nt & 1) * 2 + 1] = pack2(p2 * (dp[2] - dl1), p3 * (dp[3] - dl1));
    }
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      if (kc + kk * 16 >= T) continue;
#pragma unroll
      for (int cp = 0; cp < 4; ++cp) {
        uint32_t b00, b01, b10, b11;
        load_b_frags_kn(sK, kc + kk * 16, cp, b00, b01, b10, b11);
        mma_bf16(dq[cp * 2], dsa[kk], b00, b01);
        mma_bf16(dq[cp * 2 + 1], dsa[kk], b10, b11);
      }
    }
  }
  __nv_bfloat16* ob = dqkv + (long long)n * T * ld + h * HD;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const int d = nt * 8 + t4 * 2;
    if (q0 < T) *reinterpret_cast<uint32_t*>(ob + (long long)q0 * ld + d) = pack2(dq[nt][0], dq[nt][1]);
    if (q1 < T) *reinterpret_cast<uint32_t*>(ob + (long long)q1 * ld + d) = pack2(dq[nt][2], dq[nt][3]);
  }
  }  // tile loop
}

// dK, dV: CTA = 64 keys; Q, dO whole in smem (+ lse, delta).  Works on the transposed problem:
// S^T = K Q^T, P^T = exp(S^T*scale - lse[q]);  dV = P^T dO;  dP^T = V dO^T;  dS^T = P^T*(dP^T - delta[q])*scale;  dK = dS^T Q.
template <int MAXW, int MINB>
__global__ void __launch_bounds__(MAXW * 32, MINB) attn_bwd_dkv_kernel(const __nv_bfloat16* __restrict__ qkv, const __nv_bfloat16* __restrict__ dctx,
                                                                     const float* __restrict__ lse, const float* __restrict__ delta, int T, int heads,
                                                                     float scale, __nv_bfloat16* __restrict__ dqkv) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int Tp = (T + 63) & ~63;
  const int D = heads * HD;
  const long long ld = 3LL * D;
  const int h = blockIdx.x, n = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const uint32_t sQ = smem_addr(smem), sdO = sQ + Tp * 128;
  float* s_lse = reinterpret_cast<float*>(smem + (size_t)(2 * Tp) * 128);
  float* s_dl = s_lse + Tp;
  const uint32_t sK = sdO + Tp * 128 + 2 * Tp * 4 + warp * 4096, sV = sK + 2048;
  const __nv_bfloat16* base = qkv + (long long)n * T * ld + h * HD;
  load_tile(sQ, base, ld, 0, Tp, T);
  load_tile(sdO, dctx + (long long)n * T * D + h * HD, D, 0, Tp, T);
  const float* lb = lse + ((long long)n * heads + h) * T;
  const float* db = delta + ((long long)n * heads + h) * T;
  // s_lse holds -lse*log2e so that P^T = 2^(s*scale*log2e + s_lse): one FFMA + one MUFU per element
  for (int i = threadIdx.x; i < Tp; i += blockDim.x) { s_lse[i] = i < T ? -lb[i] * LOG2E : 0.f; s_dl[i] = i < T ? db[i] : 0.f; }
  const float sl2 = scale * LOG2E;
  cp_async_wait_all();
  __syncthreads();
  const int g = lane >> 2, t4 = lane & 3;
  for (int r0 = warp * 16; r0 < T; r0 += nwarps * 16) {
  warp_stage_tile16(sK, base + D, ld, r0, T);
  warp_stage_tile16(sV, base + 2 * D, ld, r0, T);
  cp_async_wait_all();
  __syncwarp();
  uint32_t ka[4][4], va[4][4];
  load_a_frags(sK, 0, ka);
  load_a_frags(sV, 0, va);
  float dk[8][4], dv[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) { dk[i][0] = dk[i][1] = dk[i][2] = dk[i][3] = 0.f; dv[i][0] = dv[i][1] = dv[i][2] = dv[i][3] = 0.f; }
  for (int qc = 0; qc < Tp; qc += 64) {
    uint32_t pta[4][4], dsta[4][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      float s[4] = {0.f, 0.f, 0.f, 0.f}, dp[4] = {0.f, 0.f, 0.f, 0.f};
      if (qc + nt * 8 < T) {
        uint32_t bq[4][2], bo[4][2];
        load_b_frags_nk(sQ, qc + nt * 8, bq);
        load_b_frags_nk(sdO, qc + nt * 8, bo);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) { mma_bf16(s, ka[kk], bq[kk][0], bq[kk][1]); mma_bf16(dp, va[kk], bo[kk][0], bo[kk][1]); }
      }
      const int q = qc + nt * 8 + t4 * 2;  // columns of the transposed tile are queries
      const float2 ls = *reinterpret_cast<const float2*>(s_lse + q), dd = *reinterpret_cast<const float2*>(s_dl + q);
      const float ls0 = ls.x, ls1 = ls.y, d0 = dd.x, d1 = dd.y;
      float p0 = ex2(fmaf(s[0], sl2, ls0)), p1 = ex2(fmaf(s[1], sl2, ls1));
      float p2 = ex2(fmaf(s[2], sl2, ls0)), p3 = ex2(fmaf(s[3], sl2, ls1));
      if (qc + 64 > T) {  // queries beyond T exist only in the last chunk
        if (q >= T) { p0 = 0.f; p2 = 0.f; }
        if (q + 1 >= T) { p1 = 0.f; p3 = 0.f; }
      }
      pta[nt >> 1][(nt & 1) * 2] = pack2(p0, p1);
      pta[nt >> 1][(nt & 1) * 2 + 1] = pack2(p2, p3);
      dsta[nt >> 1][(nt & 1) * 2] = pack2(p0 * (dp[0] - d0) * scale, p1 * (dp[1] - d1) * scale);
      dsta[nt >> 1][(nt & 1) * 2 + 1] = pack2(p2 * (dp[2] - d0) * scale, p3 * (dp[3] - d1) * scale);
    }
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      if (qc + kk * 16 >= T) continue;
#pragma unroll
      for (int cp = 0; cp < 4; ++cp) {
        uint32_t b00, b01, b10, b11;
        load_b_frags_kn(sdO, qc + kk * 16, cp, b00, b01, b10, b11);
        mma_bf16(dv[cp * 2], pta[kk], b00, b01);
        mma_bf16(dv[cp * 2 + 1], pta[kk], b10, b11);
        load_b_frags_kn(sQ, qc + kk * 16, cp, b00, b01, b10, b11);
        mma_bf16(dk[cp * 2], dsta[kk], b00, b01);
        mma_bf16(dk[cp * 2 + 1], dsta[kk], b10, b11);
      }
    }
  }
  const int k0 = r0 + g, k1 = k0 + 8;
  __nv_bfloat16* ob = dqkv + (long long)n * T * ld + h * HD;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const int d = nt * 8 + t4 * 2;
    if (k0 < T) {
      *reinterpret_cast<uint32_t*>(ob + (long long)k0 * ld + D + d) = pack2(dk[nt][0], dk[nt][1]);
      *reinterpret_cast<uint32_t*>(ob + (long long)k0 * ld + 2 * D + d) = pack2(dv[nt][0], dv[nt][1]);
    }
    if (k1 < T) {
      *reinterpret_cast<uint32_t*>(ob + (long long)k1 * ld + D + d) = pack2(dk[nt][2], dk[nt][3]);
      *reinterpret_cast<uint32_t*>(ob + (long long)k1 * ld + 2 * D + d) = pack2(dv[nt][2], dv[nt][3]);
    }
  }
  }  // tile loop
}

template <typename K>
int set_smem(K kernel, size_t bytes) {
  CG_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return 0;
}

}  // namespace

// warps per CTA: fill ceil(T/16) row tiles with the fewest idle slots (ties -> more warps)
static int pick_warps(int T) {
  const int tiles = (T + 15) / 16;
  int best = 4;
  double best_eff = 0.0;
  for (int w = 4; w <= MAX_WARPS; ++w) {
    const int rounds = (tiles + w - 1) / w;
    const double eff = (double)tiles / (double)(rounds * w);
    if (eff >= best_eff - 1e-9) { best_eff = eff; best = w; }
  }
  return best;
}

extern "C" int cg_attention_fwd(const void* qkv, int Nimg, int T, int heads, void* ctx, float* lse, void* stream) {
  CG_REQUIRE(qkv && ctx && lse && Nimg > 0 && T > 0 && heads > 0, "cg_attention_fwd: bad arguments");
  // the tcgen05/TMEM kernels (vit_attention_tc.cu) take every sequence that fits them: all 224-pixel towers
  if (T <= ATTN_TC_MAX_T) return cg_attention_fwd_tc(qkv, Nimg, T, heads, ctx, lse, cg_stream(stream));
  const int Tp = (T + 63) & ~63;
  CG_REQUIRE(Tp <= 640, "cg_attention_fwd: T=%d exceeds the shared-memory resident limit (640)", T);
  const int W = pick_warps(T);
  const size_t smem = (size_t)(2 * Tp) * 128 + (size_t)W * 2048;
  int rc = set_smem(attn_fwd_kernel, smem);
  if (rc) return rc;
  const float scale_log2 = 0.125f * LOG2E;  // 1/sqrt(64)
  attn_fwd_kernel<<<dim3(heads, Nimg), W * 32, smem, cg_stream(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(qkv), T, heads, scale_log2,
                                                                        reinterpret_cast<__nv_bfloat16*>(ctx), lse);
  CG_LAUNCH_CHECK();
  return 0;
}

extern "C" int cg_attention_bwd(const void* qkv, const void* ctx, const void* dctx, const float* lse, int Nimg, int T, int heads, void* dqkv,
                                float* delta_ws, void* stream) {
  CG_REQUIRE(qkv && ctx && dctx && lse && dqkv && delta_ws && Nimg > 0 && T > 0 && heads > 0, "cg_attention_bwd: bad arguments");
  const int Tp = (T + 63) & ~63;
  CG_REQUIRE(Tp <= 640, "cg_attention_bwd: T=%d exceeds the shared-memory resident limit (640)", T);
  cudaStream_t s = cg_stream(stream);
  // the tcgen05 kernel computes delta = rowsum(dO * O) itself (its epilogue warps, one item ahead)
  if (T <= ATTN_TC_MAX_T) return cg_attention_bwd_tc(qkv, ctx, dctx, lse, Nimg, T, heads, dqkv, s);
  const long long rows = (long long)Nimg * T;
  CG_CUDA(cg_launch_pdl(attn_delta_kernel, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0, s, reinterpret_cast<const __nv_bfloat16*>(ctx),
                        reinterpret_cast<const __nv_bfloat16*>(dctx), T, heads, rows, delta_ws));
  const int W = pick_warps(T);
  const size_t smem_q = (size_t)(2 * Tp) * 128 + (size_t)W * 4096;
  int rc = set_smem(attn_bwd_dq_kernel, smem_q);
  if (rc) return rc;
  attn_bwd_dq_kernel<<<dim3(heads, Nimg), W * 32, smem_q, s>>>(reinterpret_cast<const __nv_bfloat16*>(qkv), reinterpret_cast<const __nv_bfloat16*>(dctx), lse,
                                                             delta_ws, T, heads, 0.125f, reinterpret_cast<__nv_bfloat16*>(dqkv));
  CG_LAUNCH_CHECK();
  const size_t smem_kv = (size_t)(2 * Tp) * 128 + 2 * sizeof(float) * Tp + (size_t)W * 4096;
  // <= 6 warps and <= 113 KB: cap registers so that two CTAs fit one SM (the kernel is latency bound)
  if (W <= 6 && smem_kv <= 113 * 1024) {
    rc = set_smem(attn_bwd_dkv_kernel<6, 2>, smem_kv);
    if (rc) return rc;
    attn_bwd_dkv_kernel<6, 2><<<dim3(heads, Nimg), W * 32, smem_kv, s>>>(reinterpret_cast<const __nv_bfloat16*>(qkv), reinterpret_cast<const __nv_bfloat16*>(dctx),
                                                                       lse, delta_ws, T, heads, 0.125f, reinterpret_cast<__nv_bfloat16*>(dqkv));
  } else {
    rc = set_smem(attn_bwd_dkv_kernel<MAX_WARPS, 1>, smem_kv);
    if (rc) return rc;
    attn_bwd_dkv_kernel<MAX_WARPS, 1><<<dim3(heads, Nimg), W * 32, smem_kv, s>>>(reinterpret_cast<const __nv_bfloat16*>(qkv),
                                                                               reinterpret_cast<const __nv_bfloat16*>(dctx), lse, delta_ws, T, heads, 0.125f,
                                                                               reinterpret_cast<__nv_bfloat16*>(dqkv));
  }
  CG_LAUNCH_CHECK();
  return 0;
}
