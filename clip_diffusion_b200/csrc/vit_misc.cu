// Warp-level kernels of the CLIP ViT that are not contractions: LayerNorm forward/backward (fp32 residual
// stream -> bf16 GEMM operand), class-token rows, the tiny final projection, token / patch layout converters.
// All HBM-bound: one pass over the data, 128-bit accesses, one warp per row.
#include "common.cuh"

namespace {

constexpr float LN_EPS = 1e-5f;
constexpr int LN_MAX_PER_LANE = 40;  // D <= 1280

__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

// one warp per row; D = 128*NV (each lane owns NV float4 groups strided by 32 lanes, fully unrolled in registers)
template <int NV>
__global__ void __launch_bounds__(256) ln_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                                                     int M, int D, long long row_stride, __nv_bfloat16* __restrict__ yb, float* __restrict__ yf,
                                                     float* __restrict__ mean_out, float* __restrict__ rstd_out) {
  cg_griddep_launch();
  cg_griddep_wait();
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const float4* xr = reinterpret_cast<const float4*>(x + (long long)row * row_stride);
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) { v[i] = xr[i * 32 + lane]; s += v[i].x + v[i].y + v[i].z + v[i].w; }
  s = warp_sum(s);
  const float mean = s / (float)D;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    q += a * a + b * b + c * c + d * d;
  }
  q = warp_sum(q);
  const float rstd = rsqrtf(q / (float)D + LN_EPS);
  if (lane == 0) { mean_out[row] = mean; rstd_out[row] = rstd; }
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  const float4* b4 = reinterpret_cast<const float4*>(beta);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
      const float4 g = __ldg(g4 + i * 32 + lane), b = __ldg(b4 + i * 32 + lane);
      float4 y;
      y.x = (v[i].x - mean) * rstd * g.x + b.x; y.y = (v[i].y - mean) * rstd * g.y + b.y;
      y.z = (v[i].z - mean) * rstd * g.z + b.z; y.w = (v[i].w - mean) * rstd * g.w + b.w;
      if (yf) reinterpret_cast<float4*>(yf + (long long)row * D)[i * 32 + lane] = y;
      if (yb) reinterpret_cast<uint2*>(yb + (long long)row * D)[i * 32 + lane] = make_uint2(pack2(y.x, y.y), pack2(y.z, y.w));
    }
}

template <int NV>
__global__ void __launch_bounds__(256) ln_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ gamma,
                                                     const float* __restrict__ mean_in, const float* __restrict__ rstd_in, int M, int D,
                                                     long long row_stride, int accumulate, float* __restrict__ dx, __nv_bfloat16* __restrict__ dxb) {
  cg_griddep_launch();
  cg_griddep_wait();
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const float4* xr = reinterpret_cast<const float4*>(x + (long long)row * row_stride);
  const float4* dyr = reinterpret_cast<const float4*>(dy + (long long)row * D);
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  const float mean = mean_in[row], rstd = rstd_in[row];
  float4 xh[NV], dh[NV];
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
      const float4 xv = xr[i * 32 + lane], d = dyr[i * 32 + lane], g = __ldg(g4 + i * 32 + lane);
      xh[i] = make_float4((xv.x - mean) * rstd, (xv.y - mean) * rstd, (xv.z - mean) * rstd, (xv.w - mean) * rstd);
      dh[i] = make_float4(d.x * g.x, d.y * g.y, d.z * g.z, d.w * g.w);
      s1 += dh[i].x + dh[i].y + dh[i].z + dh[i].w;
      s2 += dh[i].x * xh[i].x + dh[i].y * xh[i].y + dh[i].z * xh[i].z + dh[i].w * xh[i].w;
    }
  s1 = warp_sum(s1) / (float)D;
  s2 = warp_sum(s2) / (float)D;
  float4* dxr = reinterpret_cast<float4*>(dx + (long long)row * row_stride);
  // finish r in place (x^ is dead afterwards), THEN fetch the whole previous-gradient row in one batch into the freed registers:
  // as a load -> add -> store per float4 the accumulate path was NV serialised DRAM round trips per row
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    dh[i].x = rstd * (dh[i].x - s1 - xh[i].x * s2); dh[i].y = rstd * (dh[i].y - s1 - xh[i].y * s2);
    dh[i].z = rstd * (dh[i].z - s1 - xh[i].z * s2); dh[i].w = rstd * (dh[i].w - s1 - xh[i].w * s2);
  }
  if (accumulate) {
#pragma unroll
    for (int i = 0; i < NV; ++i)
      asm volatile("ld.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(xh[i].x), "=f"(xh[i].y), "=f"(xh[i].z), "=f"(xh[i].w) : "l"(dxr + i * 32 + lane));
#pragma unroll
    for (int i = 0; i < NV; ++i) { dh[i].x += xh[i].x; dh[i].y += xh[i].y; dh[i].z += xh[i].z; dh[i].w += xh[i].w; }
  }
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    dxr[i * 32 + lane] = dh[i];
    if (dxb) reinterpret_cast<uint2*>(dxb + (long long)row * row_stride)[i * 32 + lane] = make_uint2(pack2(dh[i].x, dh[i].y), pack2(dh[i].z, dh[i].w));
  }
}

__global__ void set_cls_kernel(const float* __restrict__ cls, const float* __restrict__ pos, int T, int D, float* __restrict__ x) {
  const int n = blockIdx.x;
  for (int d = threadIdx.x; d < D; d += blockDim.x) x[(long long)n * T * D + d] = cls[d] + pos[d];
}

// emb[n,e] = sum_d y[n,d] proj[d,e];  block = (n, 128 e-columns), y row staged in smem
__global__ void __launch_bounds__(128) proj_fwd_kernel(const float* __restrict__ y, const float* __restrict__ proj, int D, int E,
                                                       float* __restrict__ emb) {
  extern __shared__ float ys[];
  const int n = blockIdx.y;
  for (int d = threadIdx.x; d < D; d += blockDim.x) ys[d] = y[(long long)n * D + d];
  __syncthreads();
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  // eight independent loads in flight and four accumulators (a single dependent chain of D L2 round trips took 75-110 us)
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  const float* pp = proj + e;
  int d = 0;
  for (; d + 8 <= D; d += 8) {
    float w[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) w[k] = __ldg(pp + (long long)(d + k) * E);
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k & 3] = fmaf(ys[d + k], w[k], acc[k & 3]);
  }
  for (; d < D; ++d) acc[0] = fmaf(ys[d], __ldg(pp + (long long)d * E), acc[0]);
  emb[(long long)n * E + e] = (acc[0] + acc[1]) + (acc[2] + acc[3]);
}

// dy[n,d] = sum_e demb[n,e] proj[d,e];  one warp per (n,d)
__global__ void __launch_bounds__(256) proj_bwd_kernel(const float* __restrict__ demb, const float* __restrict__ proj, int N, int D, int E,
                                                       float* __restrict__ dy) {
  const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= (long long)N * D) return;
  const int n = (int)(w / D), d = (int)(w % D);
  float acc = 0.f;
  for (int e = lane; e < E; e += 32) acc = fmaf(demb[(long long)n * E + e], __ldg(proj + (long long)d * E + e), acc);
  acc = warp_sum(acc);
  if (lane == 0) dy[w] = acc;
}

__global__ void __launch_bounds__(256) tokens_to_bf16_kernel(const float* __restrict__ x, int T, int D, int drop, long long total4,
                                                             __nv_bfloat16* __restrict__ out) {
  const int D4 = D >> 2;
  const int To = T - drop;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const long long orow = i / D4;
    const int c4 = (int)(i - orow * D4);
    const long long n = orow / To;
    const long long irow = n * T + drop + (orow - n * To);
    const float4 v = reinterpret_cast<const float4*>(x + irow * D)[c4];
    reinterpret_cast<uint2*>(out + orow * D)[c4] = make_uint2(pack2(v.x, v.y), pack2(v.z, v.w));
  }
}

__constant__ float c_clip_mean[3] = {0.48145466f, 0.4578275f, 0.40821073f};
__constant__ float c_clip_std[3] = {0.26862954f, 0.26130258f, 0.27577711f};

// thread per (n, patch j, k) of the output row-major [N*g2, kpad]; reads are patch-row contiguous
template <bool BWD>
__global__ void __launch_bounds__(256) patchify_kernel(float* __restrict__ img, __nv_bfloat16* __restrict__ pm, const float* __restrict__ pm32, int cs,
                                                       int patch, int kpad, int normalize, long long total) {
  const int g = cs / patch, pp = patch * patch;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(i % kpad);
    const long long pj = i / kpad;
    if (k >= 3 * pp) { if (!BWD) pm[i] = __float2bfloat16(0.f); continue; }
    const int j = (int)(pj % (g * g));
    const long long n = pj / (g * g);
    const int c = k / pp, r = k - c * pp, iy = r / patch, ix = r - iy * patch;
    const int oy = (j / g) * patch + iy, ox = (j % g) * patch + ix;
    const long long io = ((n * 3 + c) * cs + oy) * cs + ox;
    if (!BWD) {
      float v = img[io];
      if (normalize) v = (v - c_clip_mean[c]) / c_clip_std[c];
      pm[i] = __float2bfloat16(v);
    } else {
      float v = pm32 ? pm32[i] : __bfloat162float(pm[i]);
      if (normalize) v = v / c_clip_std[c];
      img[io] = v;
    }
  }
}

int rows_grid(int M) { return (M + 7) / 8; }  // 8 warps (rows) per 256-thread block
bool cg_aligned(const void* p, uintptr_t bytes) { return ((uintptr_t)p & (bytes - 1)) == 0; }  // NULL counts as aligned

}  // namespace

extern "C" int cg_layernorm_fwd(const float* x, const float* gamma, const float* beta, int M, int D, int64_t row_stride, void* y_bf16,
                                float* y_f32, float* mean, float* rstd, void* stream) {
  CG_REQUIRE(x && gamma && beta && mean && rstd && (y_bf16 || y_f32), "cg_layernorm_fwd: null pointer");
  CG_REQUIRE(M > 0 && D > 0 && D % 128 == 0 && D / 32 <= LN_MAX_PER_LANE, "cg_layernorm_fwd: D=%d must be a multiple of 128 and <= %d", D, 32 * LN_MAX_PER_LANE);
  CG_REQUIRE(row_stride >= D && row_stride % 4 == 0, "cg_layernorm_fwd: bad row stride");
  // float4 loads of x, gamma, beta and float4 / 4 x bf16 stores of y
  CG_REQUIRE(cg_aligned(x, 16) && cg_aligned(gamma, 16) && cg_aligned(beta, 16) && cg_aligned(y_f32, 16) && cg_aligned(y_bf16, 8),
             "cg_layernorm_fwd: x, gamma, beta and y_f32 must be 16-byte aligned, y_bf16 8-byte aligned");
#define CG_LN_FWD(NV) \
  case NV: CG_CUDA(cg_launch_pdl(ln_fwd_kernel<NV>, dim3(rows_grid(M)), dim3(256), 0, cg_stream(stream), x, gamma, beta, M, D, (long long)row_stride, reinterpret_cast<__nv_bfloat16*>(y_bf16), y_f32, mean, rstd)); break;
  switch (D / 128) {
    CG_LN_FWD(1) CG_LN_FWD(2) CG_LN_FWD(3) CG_LN_FWD(4) CG_LN_FWD(5) CG_LN_FWD(6) CG_LN_FWD(7) CG_LN_FWD(8) CG_LN_FWD(9) CG_LN_FWD(10)
    default: cg_set_error("cg_layernorm_fwd: unsupported D=%d", D); return CG_EINVAL;
  }
#undef CG_LN_FWD
  CG_LAUNCH_CHECK();
  return 0;
}

extern "C" int cg_layernorm_bwd(const float* dy, const float* x, const float* gamma, const float* mean, const float* rstd, int M, int D,
                                int64_t row_stride, int accumulate, float* dx, void* dx_bf16, void* stream) {
  CG_REQUIRE(dy && x && gamma && mean && rstd && dx, "cg_layernorm_bwd: null pointer");
  CG_REQUIRE(M > 0 && D > 0 && D % 128 == 0 && D / 32 <= LN_MAX_PER_LANE, "cg_layernorm_bwd: D=%d must be a multiple of 128 and <= %d", D, 32 * LN_MAX_PER_LANE);
  CG_REQUIRE(row_stride >= D && row_stride % 4 == 0, "cg_layernorm_bwd: bad row stride");
  CG_REQUIRE(cg_aligned(dy, 16) && cg_aligned(x, 16) && cg_aligned(gamma, 16) && cg_aligned(dx, 16) && cg_aligned(dx_bf16, 8),
             "cg_layernorm_bwd: dy, x, gamma and dx must be 16-byte aligned, dx_bf16 8-byte aligned");
#define CG_LN_BWD(NV) \
  case NV: CG_CUDA(cg_launch_pdl(ln_bwd_kernel<NV>, dim3(rows_grid(M)), dim3(256), 0, cg_stream(stream), dy, x, gamma, mean, rstd, M, D, (long long)row_stride, accumulate, dx, reinterpret_cast<__nv_bfloat16*>(dx_bf16))); break;
  switch (D / 128) {
    CG_LN_BWD(1) CG_LN_BWD(2) CG_LN_BWD(3) CG_LN_BWD(4) CG_LN_BWD(5) CG_LN_BWD(6) CG_LN_BWD(7) CG_LN_BWD(8) CG_LN_BWD(9) CG_LN_BWD(10)
    default: cg_set_error("cg_layernorm_bwd: unsupported D=%d", D); return CG_EINVAL;
  }
#undef CG_LN_BWD
  CG_LAUNCH_CHECK();
  return 0;
}

extern "C" int cg_vit_set_cls_rows(const float* cls, const float* pos, int Nimg, int T, int D, float* x, void* stream) {
  CG_REQUIRE(cls && pos && x && Nimg > 0 && T > 0 && D > 0, "cg_vit_set_cls_rows: bad arguments");
  set_cls_kernel<<<Nimg, 256, 0, cg_stream(stream)>>>(cls, pos, T, D, x);
  CG_LAUNCH_CHECK();
  return 0;
}

extern "C" int cg_vit_proj_fwd(const float* y, const float* proj, int N, int D, int E, float* emb, void* stream) {
  CG_REQUIRE(y && proj && emb && N > 0 && D > 0 && E > 0, "cg_vit_proj_fwd: bad arguments");
  proj_fwd_kernel<<<dim3((E + 127) / 128, N), 128, sizeof(float) * D, cg_stream(stream)>>>(y, proj, D, E, emb);
  CG_LAUNCH_CHECK();
  return 0;
}

extern "C" int cg_vit_proj_bwd(const float* demb, const float* proj, int N, int D, int E, float* dy, void* stream) {
  CG_REQUIRE(demb && proj && dy && N > 0 && D > 0 && E > 0, "cg_vit_proj_bwd: bad arguments");
  const long long warps = (long long)N * D;
  proj_bwd_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, cg_stream(stream)>>>(demb, proj, N, D, E, dy);
  CG_LAUNCH_CHECK();
  return 0;
}

extern "C" int cg_vit_tokens_to_bf16(const float* x, int Nimg, int T, int D, int drop_cls, void* out_bf16, void* stream) {
  CG_REQUIRE(x && out_bf16 && Nimg > 0 && T > 1 && D > 0 && D % 4 == 0, "cg_vit_tokens_to_bf16: bad arguments");
  const int drop = drop_cls ? 1 : 0;
  const long long total4 = (long long)Nimg * (T - drop) * (D / 4);
  long long blocks = (total4 + 255) / 256;
  if (blocks > CG_NUM_SMS * 8) blocks = CG_NUM_SMS * 8;
  tokens_to_bf16_kernel<<<(unsigned)blocks, 256, 0, cg_stream(stream)>>>(x, T, D, drop, total4, reinterpret_cast<__nv_bfloat16*>(out_bf16));
  CG_LAUNCH_CHECK();
  return 0;
}

extern "C" int cg_patchify_fwd(const float* img, int N, int cs, int patch, int kpad, int normalize, void* out_bf16, void* stream) {
  CG_REQUIRE(img && out_bf16 && N > 0 && cs > 0 && patch > 0 && cs % patch == 0 && kpad >= 3 * patch * patch, "cg_patchify_fwd: bad arguments");
  const int g = cs / patch;
  const long long total = (long long)N * g * g * kpad;
  long long blocks = (total + 255) / 256;
  if (blocks > CG_NUM_SMS * 16) blocks = CG_NUM_SMS * 16;
  patchify_kernel<false><<<(unsigned)blocks, 256, 0, cg_stream(stream)>>>(const_cast<float*>(img), reinterpret_cast<__nv_bfloat16*>(out_bf16), nullptr, cs,
                                                                         patch, kpad, normalize, total);
  CG_LAUNCH_CHECK();
  return 0;
}

extern "C" int cg_patchify_bwd(const void* dpatch, int dpatch_is_f32, int N, int cs, int patch, int kpad, int normalize, float* dimg, void* stream) {
  CG_REQUIRE(dpatch && dimg && N > 0 && cs > 0 && patch > 0 && cs % patch == 0 && kpad >= 3 * patch * patch, "cg_patchify_bwd: bad arguments");
  const int g = cs / patch;
  const long long total = (long long)N * g * g * kpad;
  long long blocks = (total + 255) / 256;
  if (blocks > CG_NUM_SMS * 16) blocks = CG_NUM_SMS * 16;
  patchify_kernel<true><<<(unsigned)blocks, 256, 0, cg_stream(stream)>>>(
      dimg, dpatch_is_f32 ? nullptr : const_cast<__nv_bfloat16*>(reinterpret_cast<const __nv_bfloat16*>(dpatch)),
      dpatch_is_f32 ? reinterpret_cast<const float*>(dpatch) : nullptr, cs, patch, kpad, normalize, total);
  CG_LAUNCH_CHECK();
  return 0;
}
