// The two non-transformer steps of OpenAI CLIP's encode_text (utils/functional.py:91-94 calls it once per prompt list):
//   cg_text_embed_fwd   x[n*T + t, :] = token_embedding[tokens[n, t], :] + positional_embedding[t, :]   (fp32 residual stream)
//   cg_text_pool_fwd    y[n, :] = ln_final(x[n*T + argmax_t tokens[n, t], :])                          (end-of-text pooling)
// The transformer in between is the ViT's kernels (GEMMs, LayerNorm) plus the causal attention of vit_attention_tc.cu; the final
// projection is cg_vit_proj_fwd.  Both kernels are HBM / latency bound and tiny next to the transformer.
#include <limits.h>
#include "common.cuh"

namespace {

constexpr float LN_EPS = 1e-5f;

// one block per token row, one float4 per thread and step; an id outside [0, V) yields a NaN row (never a read outside the table)
__global__ void __launch_bounds__(128) text_embed_kernel(const int* __restrict__ tokens, const float* __restrict__ table, const float* __restrict__ pos,
                                                         int T, int D, int V, float* __restrict__ x) {
  const long long row = blockIdx.x;
  const int t = (int)(row % T);
  const int id = tokens[row];
  const bool ok = id >= 0 && id < V;
  const float4* e4 = reinterpret_cast<const float4*>(table + (long long)(ok ? id : 0) * D);
  const float4* p4 = reinterpret_cast<const float4*>(pos + (long long)t * D);
  float4* x4 = reinterpret_cast<float4*>(x + row * D);
  for (int c = threadIdx.x; c < (D >> 2); c += blockDim.x) {
    float4 v;
    if (ok) {
      const float4 e = __ldg(e4 + c), p = __ldg(p4 + c);
      v = make_float4(e.x + p.x, e.y + p.y, e.z + p.z, e.w + p.w);
    } else {
      v = make_float4(NAN, NAN, NAN, NAN);
    }
    x4[c] = v;
  }
}

// one warp per sequence: the position of the FIRST maximal token id (torch.argmax; the end-of-text token 49407 is the largest id of
// the vocabulary), then LayerNorm of that row of x (two passes over D floats read from L2)
__global__ void __launch_bounds__(256) text_pool_kernel(const float* __restrict__ x, const int* __restrict__ tokens, int N, int T, int D,
                                                        const float* __restrict__ gamma, const float* __restrict__ beta, float* __restrict__ y) {
  const int n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (n >= N) return;
  int best = INT_MIN, pos = 0;
  for (int t = lane; t < T; t += 32) {
    const int v = tokens[(long long)n * T + t];
    if (v > best) { best = v; pos = t; }  // ascending t per lane: the first maximum of this lane's share
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const int ob = __shfl_xor_sync(0xffffffffu, best, o), op = __shfl_xor_sync(0xffffffffu, pos, o);
    if (ob > best || (ob == best && op < pos)) { best = ob; pos = op; }
  }
  const float4* xr = reinterpret_cast<const float4*>(x + ((long long)n * T + pos) * D);
  const int D4 = D >> 2;
  float s = 0.f;
  for (int c = lane; c < D4; c += 32) {
    const float4 v = xr[c];
    s += (v.x + v.y) + (v.z + v.w);
  }
  const float mean = warp_sum(s) / (float)D;
  float q = 0.f;
  for (int c = lane; c < D4; c += 32) {
    const float4 v = xr[c];
    const float a = v.x - mean, b = v.y - mean, cc = v.z - mean, d = v.w - mean;
    q += a * a + b * b + cc * cc + d * d;
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)D + LN_EPS);
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  const float4* b4 = reinterpret_cast<const float4*>(beta);
  float4* yr = reinterpret_cast<float4*>(y + (long long)n * D);
  for (int c = lane; c < D4; c += 32) {
    const float4 v = xr[c], g = __ldg(g4 + c), b = __ldg(b4 + c);
    yr[c] = make_float4((v.x - mean) * rstd * g.x + b.x, (v.y - mean) * rstd * g.y + b.y, (v.z - mean) * rstd * g.z + b.z,
                        (v.w - mean) * rstd * g.w + b.w);
  }
}

}  // namespace

extern "C" int cg_text_embed_fwd(const int* tokens, const float* token_embedding, const float* pos, int N, int T, int D, int V, float* x, void* stream) {
  CG_REQUIRE(tokens && token_embedding && pos && x && N > 0 && T > 0 && V > 0, "cg_text_embed_fwd: bad arguments");
  CG_REQUIRE(D > 0 && D % 4 == 0, "cg_text_embed_fwd: D=%d must be a positive multiple of 4", D);
  text_embed_kernel<<<(unsigned)((long long)N * T), 128, 0, cg_stream(stream)>>>(tokens, token_embedding, pos, T, D, V, x);
  CG_LAUNCH_CHECK();
  return 0;
}

extern "C" int cg_text_pool_fwd(const float* x, const int* tokens, int N, int T, int D, const float* gamma, const float* beta, float* y, void* stream) {
  CG_REQUIRE(x && tokens && gamma && beta && y && N > 0 && T > 0, "cg_text_pool_fwd: bad arguments");
  CG_REQUIRE(D > 0 && D % 4 == 0, "cg_text_pool_fwd: D=%d must be a positive multiple of 4", D);
  text_pool_kernel<<<(unsigned)((N + 7) / 8), 256, 0, cg_stream(stream)>>>(x, tokens, N, T, D, gamma, beta, y);
  CG_LAUNCH_CHECK();
  return 0;
}
