// The non-contraction kernels of CLIP's ModifiedResNet tower (OpenAI clip/model.py ModifiedResNet, Bottleneck, AttentionPool2d) on
// NHWC bf16 activations: explicit im2col for the 3x3 convolutions (forward, and the stride-1 input gradients as convolutions of the
// output gradient with flipped weights), the stem's stride-2 input gradient, 2x2 average pooling and its gradient, and the attention
// pool's token front end.  Every convolution itself is a cg_gemm_bf16_tn / cg_gemm_bf16_tn_relu call.  All HBM-bound, one pass, 128-bit
// accesses where the channel count allows; every sum is in a fixed order (no atomics), so results are bitwise reproducible.
#include "common.cuh"

namespace {

__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const __nv_bfloat162 p = *reinterpret_cast<const __nv_bfloat162*>(&w[j]);
    f[2 * j] = __low2float(p);
    f[2 * j + 1] = __high2float(p);
  }
}
__device__ __forceinline__ uint4 pack8(const float* f) {
  return make_uint4(pack2(f[0], f[1]), pack2(f[2], f[3]), pack2(f[4], f[5]), pack2(f[6], f[7]));
}
// ReLU derivative as torch's threshold_backward: zero where the saved output is <= 0 (a NaN output passes the gradient)
__device__ __forceinline__ float drelu(float g, float a) { return a <= 0.f ? 0.f : g; }

constexpr int THREADS = 256;

static inline int blocks_for(long long n) {
  long long b = (n + THREADS - 1) / THREADS;
  return (int)(b < 1 ? 1 : b);
}

// one thread per 8 output columns of one output row.  VEC: C % 8 == 0, so the 8 columns are 8 consecutive channels of one tap
template <bool VEC>
__global__ void __launch_bounds__(THREADS) im2col3x3_kernel(const __nv_bfloat16* __restrict__ x, int H, int W, int C, long long ldx, int stride,
                                                           int Ho, int Wo, int kpad, long long chunks, __nv_bfloat16* __restrict__ out) {
  const long long i = (long long)blockIdx.x * THREADS + threadIdx.x;
  if (i >= chunks) return;
  const int cpr = kpad >> 3;
  const long long r = i / cpr;
  const int j0 = (int)(i - r * cpr) * 8;
  const int ox = (int)(r % Wo);
  const long long t = r / Wo;
  const int oy = (int)(t % Ho);
  const long long n = t / Ho;
  const __nv_bfloat16* xn = x + n * H * W * ldx;
  uint4 v = make_uint4(0u, 0u, 0u, 0u);
  if (VEC) {
    const int tap = j0 / C;
    if (tap < 9) {
      const int iy = oy * stride + tap / 3 - 1, ix = ox * stride + tap % 3 - 1;
      if (iy >= 0 && iy < H && ix >= 0 && ix < W) v = __ldg(reinterpret_cast<const uint4*>(xn + ((long long)iy * W + ix) * ldx + (j0 - tap * C)));
    }
  } else {
    __nv_bfloat16 e[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int j = j0 + k, tap = j / C;
      e[k] = __float2bfloat16(0.f);
      if (tap < 9) {
        const int iy = oy * stride + tap / 3 - 1, ix = ox * stride + tap % 3 - 1;
        if (iy >= 0 && iy < H && ix >= 0 && ix < W) e[k] = xn[((long long)iy * W + ix) * ldx + (j - tap * C)];
      }
    }
    v = *reinterpret_cast<const uint4*>(e);
  }
  reinterpret_cast<uint4*>(out)[i] = v;
}

// one thread per input pixel: dx[n, iy, ix, ci] = sum over the (at most 4) output positions whose 3x3 stride-2 window covers (iy, ix), in
// the order ky, kx, co, of dy[n, oy, ox, co] * w[co, ci, ky, kx]
constexpr int S2_MAX_CIN = 8;
__global__ void __launch_bounds__(THREADS) conv3x3s2_dgrad_kernel(const __nv_bfloat16* __restrict__ dy, int Ho, int Wo, int Cout, long long lddy,
                                                                 const float* __restrict__ w, int Cin, int H, int W, int kpad, long long pixels,
                                                                 float* __restrict__ dx) {
  extern __shared__ float ws[];  // [Cout][Cin][9]
  for (int k = threadIdx.x; k < Cout * Cin * 9; k += THREADS) ws[k] = w[k];
  __syncthreads();
  const long long p = (long long)blockIdx.x * THREADS + threadIdx.x;
  if (p >= pixels) return;
  const int ix = (int)(p % W);
  const long long t = p / W;
  const int iy = (int)(t % H);
  const long long n = t / H;
  float acc[S2_MAX_CIN];
#pragma unroll
  for (int c = 0; c < S2_MAX_CIN; ++c) acc[c] = 0.f;
  for (int ky = 0; ky < 3; ++ky) {
    const int ty = iy + 1 - ky;
    if (ty < 0 || (ty & 1) || (ty >> 1) >= Ho) continue;
    for (int kx = 0; kx < 3; ++kx) {
      const int tx = ix + 1 - kx;
      if (tx < 0 || (tx & 1) || (tx >> 1) >= Wo) continue;
      const __nv_bfloat16* d = dy + ((n * Ho + (ty >> 1)) * Wo + (tx >> 1)) * lddy;
      const float* wk = ws + ky * 3 + kx;
      for (int co = 0; co < Cout; ++co) {
        const float g = __bfloat162float(d[co]);
#pragma unroll
        for (int c = 0; c < S2_MAX_CIN; ++c)
          if (c < Cin) acc[c] = fmaf(g, wk[(co * Cin + c) * 9], acc[c]);
      }
    }
  }
  float* o = dx + p * kpad;
#pragma unroll
  for (int c = 0; c < S2_MAX_CIN; ++c)
    if (c < kpad) o[c] = c < Cin ? acc[c] : 0.f;
  for (int c = S2_MAX_CIN; c < kpad; ++c) o[c] = 0.f;
}

// one thread per 8 channels of one output pixel
__global__ void __launch_bounds__(THREADS) avgpool2x2_fwd_kernel(const __nv_bfloat16* __restrict__ x, int H, int W, int C, long long chunks,
                                                                __nv_bfloat16* __restrict__ y) {
  const long long i = (long long)blockIdx.x * THREADS + threadIdx.x;
  if (i >= chunks) return;
  const int cpp = C >> 3, Ho = H >> 1, Wo = W >> 1;
  const long long r = i / cpp;
  const int c0 = (int)(i - r * cpp) * 8;
  const int ox = (int)(r % Wo);
  const long long t = r / Wo;
  const int oy = (int)(t % Ho);
  const long long n = t / Ho;
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int dy = 0; dy < 2; ++dy)
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      float f[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(x + ((n * H + 2 * oy + dy) * W + 2 * ox + dx) * C + c0)), f);
#pragma unroll
      for (int k = 0; k < 8; ++k) s[k] += f[k];
    }
#pragma unroll
  for (int k = 0; k < 8; ++k) s[k] *= 0.25f;
  reinterpret_cast<uint4*>(y)[i] = pack8(s);
}

// one thread per 8 channels of one INPUT pixel: dx = 0.25 dy[n, iy/2, ix/2] (* [mask > 0])
__global__ void __launch_bounds__(THREADS) avgpool2x2_bwd_kernel(const void* __restrict__ dy, int dy_f32, const __nv_bfloat16* __restrict__ mask,
                                                                int H, int W, int C, long long chunks, void* __restrict__ dx, int dx_f32) {
  const long long i = (long long)blockIdx.x * THREADS + threadIdx.x;
  if (i >= chunks) return;
  const int cpp = C >> 3, Ho = H >> 1, Wo = W >> 1;
  const long long r = i / cpp;
  const int c0 = (int)(i - r * cpp) * 8;
  const int ix = (int)(r % W);
  const long long t = r / W;
  const int iy = (int)(t % H);
  const long long n = t / H;
  const long long src = ((n * Ho + (iy >> 1)) * Wo + (ix >> 1)) * C + c0;
  float g[8];
  if (dy_f32) {
    const float4* p = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(dy) + src);
    const float4 a = __ldg(p), b = __ldg(p + 1);
    g[0] = a.x; g[1] = a.y; g[2] = a.z; g[3] = a.w; g[4] = b.x; g[5] = b.y; g[6] = b.z; g[7] = b.w;
  } else {
    unpack8(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(dy) + src)), g);
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) g[k] *= 0.25f;
  if (mask) {
    float m[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(mask) + i), m);
#pragma unroll
    for (int k = 0; k < 8; ++k) g[k] = drelu(g[k], m[k]);
  }
  if (dx_f32) {
    float4* o = reinterpret_cast<float4*>(dx) + 2 * i;
    o[0] = make_float4(g[0], g[1], g[2], g[3]);
    o[1] = make_float4(g[4], g[5], g[6], g[7]);
  } else {
    reinterpret_cast<uint4*>(dx)[i] = pack8(g);
  }
}

// AttentionPool2d front end.  One thread per (image, 8 channels): tok[n, 0] = mean_s x[n, s] + pos[0], tok[n, 1 + s] = x[n, s] + pos[1 + s]
__global__ void __launch_bounds__(THREADS) attnpool_fwd_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ pos, int N, int S,
                                                              int C, __nv_bfloat16* __restrict__ tok) {
  const long long i = (long long)blockIdx.x * THREADS + threadIdx.x;
  const int cpp = C >> 3;
  if (i >= (long long)N * cpp) return;
  const long long n = i / cpp;
  const int c0 = (int)(i - n * cpp) * 8;
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int j = 0; j < S; ++j) {
    float f[8], o[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(x + (n * S + j) * C + c0)), f);
    const float* p = pos + (long long)(1 + j) * C + c0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { s[k] += f[k]; o[k] = f[k] + __ldg(p + k); }
    *reinterpret_cast<uint4*>(tok + (n * (S + 1) + 1 + j) * C + c0) = pack8(o);
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) s[k] = s[k] / (float)S + __ldg(pos + c0 + k);
  *reinterpret_cast<uint4*>(tok + n * (S + 1) * C + c0) = pack8(s);
}

// g[n, s] = (dtok[n, 1 + s] + dtok[n, 0] / S) * [x[n, s] > 0]: the gradient of the tokens' front end, masked by the last block's ReLU
__global__ void __launch_bounds__(THREADS) attnpool_bwd_kernel(const float* __restrict__ dtok, const __nv_bfloat16* __restrict__ x, int N, int S,
                                                              int C, float* __restrict__ g, __nv_bfloat16* __restrict__ gb) {
  const long long i = (long long)blockIdx.x * THREADS + threadIdx.x;  // over N * S * C / 8
  const int cpp = C >> 3;
  if (i >= (long long)N * S * cpp) return;
  const long long r = i / cpp;
  const int c0 = (int)(i - r * cpp) * 8;
  const long long n = r / S, j = r - n * S;
  const float* d0 = dtok + n * (S + 1) * C + c0;
  const float* d = dtok + (n * (S + 1) + 1 + j) * C + c0;
  float m[8], v[8];
  unpack8(__ldg(reinterpret_cast<const uint4*>(x) + i), m);
#pragma unroll
  for (int k = 0; k < 8; ++k) v[k] = drelu(__ldg(d + k) + __ldg(d0 + k) / (float)S, m[k]);
  float4* o = reinterpret_cast<float4*>(g) + 2 * i;
  o[0] = make_float4(v[0], v[1], v[2], v[3]);
  o[1] = make_float4(v[4], v[5], v[6], v[7]);
  reinterpret_cast<uint4*>(gb)[i] = pack8(v);
}

// dctx[n*T + t, :] = t == 0 ? bf16(dy[n, :]) : 0 -- the attention output gradient of a pool that keeps only the query row 0
__global__ void __launch_bounds__(THREADS) attnpool_dctx_kernel(const float* __restrict__ dy, int N, int T, int C, __nv_bfloat16* __restrict__ dctx) {
  const long long i = (long long)blockIdx.x * THREADS + threadIdx.x;  // over N * T * C / 8
  const int cpp = C >> 3;
  if (i >= (long long)N * T * cpp) return;
  const long long r = i / cpp;
  const int c0 = (int)(i - r * cpp) * 8;
  const long long n = r / T;
  float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (r == n * T) {
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = __ldg(dy + n * C + c0 + k);
  }
  reinterpret_cast<uint4*>(dctx)[i] = pack8(v);
}

bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

}  // namespace

extern "C" int cg_im2col3x3_nhwc(const void* x, int N, int H, int W, int C, int64_t ldx, int stride, int kpad, void* out, void* stream) {
  CG_REQUIRE(x && out && N > 0 && H > 0 && W > 0 && C > 0, "cg_im2col3x3_nhwc: bad arguments");
  CG_REQUIRE(stride == 1 || stride == 2, "cg_im2col3x3_nhwc: stride %d must be 1 or 2", stride);
  CG_REQUIRE(ldx >= C && ldx % 8 == 0, "cg_im2col3x3_nhwc: ldx=%lld must be >= C=%d and a multiple of 8", (long long)ldx, C);
  CG_REQUIRE(kpad % 64 == 0 && kpad >= 9 * C, "cg_im2col3x3_nhwc: kpad=%d must be a multiple of 64 and >= 9C=%d", kpad, 9 * C);
  CG_REQUIRE(aligned16(x) && aligned16(out), "cg_im2col3x3_nhwc: pointers must be 16-byte aligned");
  const int Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
  const long long chunks = (long long)N * Ho * Wo * (kpad / 8);
  cudaStream_t s = cg_stream(stream);
  const auto* xb = reinterpret_cast<const __nv_bfloat16*>(x);
  auto* ob = reinterpret_cast<__nv_bfloat16*>(out);
  if (C % 8 == 0) im2col3x3_kernel<true><<<blocks_for(chunks), THREADS, 0, s>>>(xb, H, W, C, ldx, stride, Ho, Wo, kpad, chunks, ob);
  else im2col3x3_kernel<false><<<blocks_for(chunks), THREADS, 0, s>>>(xb, H, W, C, ldx, stride, Ho, Wo, kpad, chunks, ob);
  CG_LAUNCH_CHECK();
  return 0;
}

extern "C" int cg_conv3x3s2_dgrad(const void* dy, int N, int H, int W, int Cout, int64_t lddy, const float* w, int Cin, int kpad, float* dx,
                                  void* stream) {
  CG_REQUIRE(dy && w && dx && N > 0 && H > 0 && W > 0, "cg_conv3x3s2_dgrad: bad arguments");
  CG_REQUIRE(Cin > 0 && Cin <= S2_MAX_CIN && kpad >= Cin && kpad % 4 == 0, "cg_conv3x3s2_dgrad: Cin=%d must lie in [1, %d], kpad=%d >= Cin and a multiple of 4",
             Cin, S2_MAX_CIN, kpad);
  CG_REQUIRE(Cout > 0 && Cout <= 256 && lddy >= Cout, "cg_conv3x3s2_dgrad: Cout=%d must lie in [1, 256] and lddy >= Cout", Cout);
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  const long long pixels = (long long)N * H * W;
  const size_t smem = sizeof(float) * Cout * Cin * 9;
  conv3x3s2_dgrad_kernel<<<blocks_for(pixels), THREADS, smem, cg_stream(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(dy), Ho, Wo, Cout, lddy,
                                                                                    w, Cin, H, W, kpad, pixels, dx);
  CG_LAUNCH_CHECK();
  return 0;
}

extern "C" int cg_avgpool2x2_nhwc_fwd(const void* x, int N, int H, int W, int C, void* y, void* stream) {
  CG_REQUIRE(x && y && N > 0 && H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0 && C > 0 && C % 8 == 0,
             "cg_avgpool2x2_nhwc_fwd: bad sizes N=%d H=%d W=%d C=%d (H, W even, C %% 8 == 0)", N, H, W, C);
  CG_REQUIRE(aligned16(x) && aligned16(y), "cg_avgpool2x2_nhwc_fwd: pointers must be 16-byte aligned");
  const long long chunks = (long long)N * (H / 2) * (W / 2) * (C / 8);
  avgpool2x2_fwd_kernel<<<blocks_for(chunks), THREADS, 0, cg_stream(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(x), H, W, C, chunks,
                                                                               reinterpret_cast<__nv_bfloat16*>(y));
  CG_LAUNCH_CHECK();
  return 0;
}

extern "C" int cg_avgpool2x2_nhwc_bwd(const void* dy, int dy_f32, const void* mask, int N, int H, int W, int C, void* dx, int dx_f32, void* stream) {
  CG_REQUIRE(dy && dx && N > 0 && H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0 && C > 0 && C % 8 == 0,
             "cg_avgpool2x2_nhwc_bwd: bad sizes N=%d H=%d W=%d C=%d (H, W even, C %% 8 == 0)", N, H, W, C);
  CG_REQUIRE(aligned16(dy) && aligned16(dx) && aligned16(mask), "cg_avgpool2x2_nhwc_bwd: pointers must be 16-byte aligned");
  const long long chunks = (long long)N * H * W * (C / 8);
  avgpool2x2_bwd_kernel<<<blocks_for(chunks), THREADS, 0, cg_stream(stream)>>>(dy, dy_f32, reinterpret_cast<const __nv_bfloat16*>(mask), H, W, C,
                                                                               chunks, dx, dx_f32);
  CG_LAUNCH_CHECK();
  return 0;
}

extern "C" int cg_resnet_attnpool_fwd(const void* x, const float* pos, int N, int S, int C, void* tok, void* stream) {
  CG_REQUIRE(x && pos && tok && N > 0 && S > 0 && C > 0 && C % 8 == 0, "cg_resnet_attnpool_fwd: bad arguments N=%d S=%d C=%d", N, S, C);
  CG_REQUIRE(aligned16(x) && aligned16(tok), "cg_resnet_attnpool_fwd: pointers must be 16-byte aligned");
  attnpool_fwd_kernel<<<blocks_for((long long)N * C / 8), THREADS, 0, cg_stream(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(x), pos, N, S, C,
                                                                                          reinterpret_cast<__nv_bfloat16*>(tok));
  CG_LAUNCH_CHECK();
  return 0;
}

extern "C" int cg_resnet_attnpool_bwd(const float* dtok, const void* x, int N, int S, int C, float* g, void* g_bf16, void* stream) {
  CG_REQUIRE(dtok && x && g && g_bf16 && N > 0 && S > 0 && C > 0 && C % 8 == 0, "cg_resnet_attnpool_bwd: bad arguments N=%d S=%d C=%d", N, S, C);
  CG_REQUIRE(aligned16(x) && aligned16(g) && aligned16(g_bf16), "cg_resnet_attnpool_bwd: pointers must be 16-byte aligned");
  attnpool_bwd_kernel<<<blocks_for((long long)N * S * C / 8), THREADS, 0, cg_stream(stream)>>>(dtok, reinterpret_cast<const __nv_bfloat16*>(x), N, S,
                                                                                              C, g, reinterpret_cast<__nv_bfloat16*>(g_bf16));
  CG_LAUNCH_CHECK();
  return 0;
}

extern "C" int cg_resnet_attnpool_dctx(const float* dy, int N, int T, int C, void* dctx, void* stream) {
  CG_REQUIRE(dy && dctx && N > 0 && T > 0 && C > 0 && C % 8 == 0, "cg_resnet_attnpool_dctx: bad arguments N=%d T=%d C=%d", N, T, C);
  CG_REQUIRE(aligned16(dctx), "cg_resnet_attnpool_dctx: dctx must be 16-byte aligned");
  attnpool_dctx_kernel<<<blocks_for((long long)N * T * C / 8), THREADS, 0, cg_stream(stream)>>>(dy, N, T, C, reinterpret_cast<__nv_bfloat16*>(dctx));
  CG_LAUNCH_CHECK();
  return 0;
}
