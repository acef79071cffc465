// C-ABI plumbing shared by every entry point: thread-local error text, ABI version, device check,
// and the small cond_fn tail kernels (sample.py:228-238).
#include <stdarg.h>
#include <stdlib.h>
#include "common.cuh"

static thread_local char g_err[512] = "";

void cg_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" const char* cg_last_error(void) { return g_err; }
extern "C" int cg_abi_version(void) { return 5; }  // 5: cg_gemm_tile_variant; 4: cg_image_losses_fwd_bwd, deterministic loss values; 3: producer-side GroupNorm partials (input_partial); 2: + UNet NHWC ops (cg_groupnorm_nhwc_*, cg_bias_residual_add_nhwc, cg_resample2x_nhwc, cg_concat2_nhwc)

extern "C" int cg_check_device(void) {
  int dev = 0;
  CG_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp p;
  CG_CUDA(cudaGetDeviceProperties(&p, dev));
  if (p.major != 10) {
    cg_set_error("clipguide_b200 is built for sm_100a only; device %d is sm_%d%d", dev, p.major, p.minor);
    return CG_EARCH;
  }
  return 0;
}

int cg_get_scratch(CgScratch* out) {
  static CgScratch per_device[64] = {};
  int dev = 0;
  CG_CUDA(cudaGetDevice(&dev));
  CG_REQUIRE(dev >= 0 && dev < 64, "device ordinal %d out of range", dev);
  if (!per_device[dev].partials) {
    void* p = nullptr;
    CG_CUDA(cudaMalloc(&p, sizeof(float) * CG_SCRATCH_FLOATS + sizeof(unsigned) * CG_SCRATCH_COUNTERS));
    CG_CUDA(cudaMemset(p, 0, sizeof(float) * CG_SCRATCH_FLOATS + sizeof(unsigned) * CG_SCRATCH_COUNTERS));
    per_device[dev].partials = reinterpret_cast<float*>(p);
    per_device[dev].counters = reinterpret_cast<unsigned*>(per_device[dev].partials + CG_SCRATCH_FLOATS);
  }
  *out = per_device[dev];
  return 0;
}

namespace {

// scratch[0] = sum g^2 (deterministic: per-block partials summed in index order by the last block), scratch[1] = NaN count (> 0 or not:
// order independent)
__global__ void __launch_bounds__(256) sumsq_nan_kernel(const float* __restrict__ g, int64_t n, float* __restrict__ scratch, CgScratch ws) {
  __shared__ float red[32];
  float s = 0.f, bad = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = g[i];
    s += v * v;
    if (v != v) bad += 1.f;
  }
  const float ts = block_sum(s, red);
  const float tb = block_sum(bad, red);
  if (threadIdx.x == 0 && tb > 0.f) scratch[1] = tb;  // any positive value: racing writers all store "bad"
  if (cg_last_block(ts, ws.partials, ws.counters + 0, blockIdx.x, gridDim.x)) {
    const float total = cg_sum_partials(ws.partials, 0, gridDim.x, red);
    if (threadIdx.x == 0) scratch[0] = total;
  }
}

__global__ void __launch_bounds__(256) finalize_kernel(const float* __restrict__ g, int64_t n, float sign, float thr,
                                                       const float* __restrict__ scratch, const float* __restrict__ bad_flag,
                                                       float* __restrict__ out) {
  const bool bad = bad_flag ? (bad_flag[0] != 0.f) : (scratch[1] > 0.f);
  const float mag = sqrtf(scratch[0] / (float)n);
  // grad * clamp(mag, -thr, thr) / mag   (sample.py:236-238); mag == 0 gives NaN there as well (0/0)
  const float k = sign * fminf(fmaxf(mag, -thr), thr) / mag;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = bad ? 0.f : g[i] * k;
}

__global__ void nanflag_kernel(float* flag) { flag[0] = flag[1] > 0.f ? 1.f : 0.f; }

}  // namespace

static int blocks_for(int64_t n) {
  int64_t b = (n + 255) / 256;
  if (b > CG_NUM_SMS * 4) b = CG_NUM_SMS * 4;
  return (int)(b < 1 ? 1 : b);
}

extern "C" int cg_grad_finalize(const float* g, int64_t n, float sign, float thr, const float* bad_flag, float* out, float* scratch,
                                void* stream) {
  CG_REQUIRE(g && out && scratch && n > 0, "cg_grad_finalize: bad arguments");
  cudaStream_t s = cg_stream(stream);
  CgScratch ws;
  int rc = cg_get_scratch(&ws);
  if (rc) return rc;
  CG_CUDA(cudaMemsetAsync(scratch, 0, 2 * sizeof(float), s));
  sumsq_nan_kernel<<<blocks_for(n), 256, 0, s>>>(g, n, scratch, ws);
  CG_LAUNCH_CHECK();
  finalize_kernel<<<blocks_for(n), 256, 0, s>>>(g, n, sign, thr, scratch, bad_flag, out);
  CG_LAUNCH_CHECK();
  return 0;
}

extern "C" int cg_any_nan(const float* g, int64_t n, float* flag, void* stream) {
  CG_REQUIRE(g && flag && n > 0, "cg_any_nan: bad arguments");
  cudaStream_t s = cg_stream(stream);
  CgScratch ws;
  int rc = cg_get_scratch(&ws);
  if (rc) return rc;
  // flag doubles as scratch: needs 2 floats
  CG_CUDA(cudaMemsetAsync(flag, 0, 2 * sizeof(float), s));
  sumsq_nan_kernel<<<blocks_for(n), 256, 0, s>>>(g, n, flag, ws);
  CG_LAUNCH_CHECK();
  nanflag_kernel<<<1, 1, 0, s>>>(flag);
  CG_LAUNCH_CHECK();
  return 0;
}

bool cg_pdl_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("CG_PDL");
    v = (e && atoi(e) == 0) ? 0 : 1;
  }
  return v != 0;
}
