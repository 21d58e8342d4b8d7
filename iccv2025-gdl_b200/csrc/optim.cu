// optim.cu — gradient clipping statistics, DGL gradient diagnostics and the parameter updates over
// the flat fp32 parameter arena (reference main_dgl.py:129 clip_grad_norm_(40, L2),
// :132-143 sum_p mean|grad_p| per encoder, :154/:249-256 torch.optim.SGD(momentum, weight_decay),
// Adagrad and Adam).  One pass over the gradients produces the global L2 norm and both diagnostics;
// the clip coefficient stays on the device and is folded into the update kernel, which also writes
// the clipped gradient back (clip_grad_norm_ is in-place in the reference).
#include "common.cuh"
#include "api_version.h"

namespace gdl {

constexpr int kChunk = 8192;  // elements per block: fixed => deterministic partials
constexpr int kOptThreads = 256;

__device__ __forceinline__ int find_segment(const int64_t* __restrict__ seg_end, int nseg, int64_t i) {
  int lo = 0, hi = nseg - 1;
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (i < seg_end[mid]) hi = mid; else lo = mid + 1;
  }
  return lo;
}

__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
  if (threadIdx.x < 32) {
    t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    t = warp_sum(t);
  }
  return t;  // valid in warp 0
}

__global__ void __launch_bounds__(kOptThreads) grad_stats_kernel(
    const float* __restrict__ grad, int64_t numel, const int64_t* __restrict__ seg_end,
    const int32_t* __restrict__ seg_group, const float* __restrict__ seg_inv_numel, int nseg,
    float* __restrict__ partial) {
  pdl_enter();
  __shared__ float red[32];
  __shared__ int s_lo, s_hi;
  const int64_t start = (int64_t)blockIdx.x * kChunk;
  const int64_t end = start + kChunk < numel ? start + kChunk : numel;
  if (threadIdx.x == 0) {
    s_lo = find_segment(seg_end, nseg, start);
    s_hi = find_segment(seg_end, nseg, end - 1);
  }
  __syncthreads();
  const int lo = s_lo, hi = s_hi;
  float sq = 0.f, wa = 0.f, wv = 0.f;
  for (int64_t i = start + threadIdx.x; i < end; i += kOptThreads) {
    float g = grad[i];
    sq = fmaf(g, g, sq);
    int sgm = lo;
    if (lo != hi) {
      while (sgm < hi && i >= seg_end[sgm]) ++sgm;
    }
    int grp = seg_group[sgm];
    float w = fabsf(g) * seg_inv_numel[sgm];
    if (grp == 0) wa += w;
    else if (grp == 1) wv += w;
  }
  float t0 = block_sum(sq, red);
  float t1 = block_sum(wa, red);
  float t2 = block_sum(wv, red);
  if (threadIdx.x == 0) {
    partial[(int64_t)blockIdx.x * 3 + 0] = t0;
    partial[(int64_t)blockIdx.x * 3 + 1] = t1;
    partial[(int64_t)blockIdx.x * 3 + 2] = t2;
  }
}

__global__ void grad_stats_finalize_kernel(const float* __restrict__ partial, int nblk, float max_norm,
                                           float* __restrict__ stats) {
  pdl_enter();
  // single block; fixed-order strided accumulation in double, then a fixed tree
  __shared__ double red[3][256];
  double a0 = 0, a1 = 0, a2 = 0;
  for (int b = threadIdx.x; b < nblk; b += 256) {
    a0 += partial[(int64_t)b * 3 + 0];
    a1 += partial[(int64_t)b * 3 + 1];
    a2 += partial[(int64_t)b * 3 + 2];
  }
  red[0][threadIdx.x] = a0; red[1][threadIdx.x] = a1; red[2][threadIdx.x] = a2;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      red[0][threadIdx.x] += red[0][threadIdx.x + s];
      red[1][threadIdx.x] += red[1][threadIdx.x + s];
      red[2][threadIdx.x] += red[2][threadIdx.x + s];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    float norm = (float)sqrt(red[0][0]);
    float coef = max_norm / (norm + 1e-6f);  // torch.nn.utils.clip_grad_norm_ formula
    if (coef > 1.f) coef = 1.f;
    stats[0] = norm;
    stats[1] = coef;
    stats[2] = (float)red[1][0] * coef;
    stats[3] = (float)red[2][0] * coef;
  }
}

// lr_dev (may be NULL => lr): the learning rate as one float64 in device memory, cast to float here as ctypes casts
// a Python float passed as lr, so a captured update follows a per-iteration lr schedule without re-capture.
__global__ void __launch_bounds__(256) sgd_momentum_kernel(float* __restrict__ param,
                                                           float* __restrict__ grad,
                                                           float* __restrict__ buf, int64_t n4,
                                                           int64_t numel, float lr_host,
                                                           const double* __restrict__ lr_dev, float mu,
                                                           float wd, int first,
                                                           const float* __restrict__ stats) {
  pdl_enter();
  const float coef = stats ? stats[1] : 1.f;
  const float lr = lr_dev ? (float)*lr_dev : lr_host;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
       i += (int64_t)gridDim.x * blockDim.x) {
    float4 p = reinterpret_cast<float4*>(param)[i];
    float4 g = reinterpret_cast<float4*>(grad)[i];
    float4 m = first ? make_float4(0.f, 0.f, 0.f, 0.f) : reinterpret_cast<float4*>(buf)[i];
    float* pp = &p.x; float* gg = &g.x; float* mm = &m.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float gc = gg[k] * coef;
      gg[k] = gc;
      float d = fmaf(wd, pp[k], gc);
      mm[k] = first ? d : fmaf(mu, mm[k], d);
      pp[k] = fmaf(-lr, mm[k], pp[k]);
    }
    reinterpret_cast<float4*>(param)[i] = p;
    reinterpret_cast<float4*>(grad)[i] = g;
    reinterpret_cast<float4*>(buf)[i] = m;
  }
  // tail (numel not a multiple of 4)
  if (blockIdx.x == 0 && threadIdx.x < (numel & 3)) {
    int64_t i = n4 * 4 + threadIdx.x;
    float gc = grad[i] * coef;
    grad[i] = gc;
    float d = fmaf(wd, param[i], gc);
    float m = first ? d : fmaf(mu, buf[i], d);
    buf[i] = m;
    param[i] = fmaf(-lr, m, param[i]);
  }
}

// ---- Adam / Adagrad (torch.optim.Adam / Adagrad, non-capturable single-tensor and foreach formulas) ----
// The update runs inside a CUDA graph captured once, so the step count cannot be a kernel argument: it lives in
// step_state[0] on the device, and so may the lr (lr_dev, one float64; NULL => lr_host).  One thread advances the
// count and writes the step's scalars into step_state[1..2] before the element kernel reads them (stream order), so
// every block of the element kernel sees the same step.
enum { kRuleAdam = 0, kRuleAdagrad = 1 };

__global__ void optim_step_prologue_kernel(int32_t* __restrict__ step_state, int rule, double lr_host,
                                           const double* __restrict__ lr_dev, double a, double b) {
  pdl_enter();
  const double lr = lr_dev ? *lr_dev : lr_host;
  const int32_t step = step_state[0] + 1;
  step_state[0] = step;
  float* f = reinterpret_cast<float*>(step_state + 1);
  const double s = (double)step;  // torch: the step is a Python float here
  if (rule == kRuleAdam) {        // a = beta1, b = beta2
    const double bc1 = 1.0 - pow(a, s), bc2 = 1.0 - pow(b, s);
    f[0] = (float)(lr / bc1);  // step_size, cast where addcdiv_(value=-step_size) casts it
    f[1] = (float)sqrt(bc2);   // bias_correction2_sqrt, cast where the tensor division casts it
  } else {                     // a = lr_decay
    f[0] = (float)(lr / (1.0 + (s - 1.0) * a));  // clr
  }
}

__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ param, float* __restrict__ grad,
                                                   float* __restrict__ exp_avg, float* __restrict__ exp_avg_sq,
                                                   int64_t n4, int64_t numel, float w1, float beta2, float w2,
                                                   float eps, float wd, const float* __restrict__ stats,
                                                   const int32_t* __restrict__ step_state) {
  pdl_enter();
  const float coef = stats ? stats[1] : 1.f;
  const float* sc = reinterpret_cast<const float*>(step_state + 1);
  const float step_size = sc[0], bc2s = sc[1];
  // m = lerp(m, g, w1) (torch's small-weight branch), v = beta2*v + w2*g*g, p -= step_size * m / (sqrt(v)/bc2s + eps)
  auto upd = [&](float& p, float& g, float& m, float& v) {
    const float gc = g * coef;
    g = gc;
    const float d = fmaf(wd, p, gc);
    m = fmaf(w1, d - m, m);
    v = fmaf(w2, d * d, v * beta2);
    const float denom = sqrtf(v) / bc2s + eps;
    p = fmaf(-step_size, m / denom, p);
  };
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
       i += (int64_t)gridDim.x * blockDim.x) {
    float4 p = reinterpret_cast<float4*>(param)[i];
    float4 g = reinterpret_cast<float4*>(grad)[i];
    float4 m = reinterpret_cast<float4*>(exp_avg)[i];
    float4 v = reinterpret_cast<float4*>(exp_avg_sq)[i];
    upd(p.x, g.x, m.x, v.x);
    upd(p.y, g.y, m.y, v.y);
    upd(p.z, g.z, m.z, v.z);
    upd(p.w, g.w, m.w, v.w);
    reinterpret_cast<float4*>(param)[i] = p;
    reinterpret_cast<float4*>(grad)[i] = g;
    reinterpret_cast<float4*>(exp_avg)[i] = m;
    reinterpret_cast<float4*>(exp_avg_sq)[i] = v;
  }
  // tail (numel not a multiple of 4)
  if (blockIdx.x == 0 && threadIdx.x < (numel & 3)) {
    int64_t i = n4 * 4 + threadIdx.x;
    upd(param[i], grad[i], exp_avg[i], exp_avg_sq[i]);
  }
}

__global__ void __launch_bounds__(256) adagrad_kernel(float* __restrict__ param, float* __restrict__ grad,
                                                      float* __restrict__ sum, int64_t n4, int64_t numel, float eps,
                                                      float wd, const float* __restrict__ stats,
                                                      const int32_t* __restrict__ step_state) {
  pdl_enter();
  const float coef = stats ? stats[1] : 1.f;
  const float clr = reinterpret_cast<const float*>(step_state + 1)[0];
  // s += g*g, p -= clr * g / (sqrt(s) + eps)
  auto upd = [&](float& p, float& g, float& s) {
    const float gc = g * coef;
    g = gc;
    const float d = fmaf(wd, p, gc);
    s = fmaf(d, d, s);
    p = fmaf(-clr, d / (sqrtf(s) + eps), p);
  };
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
       i += (int64_t)gridDim.x * blockDim.x) {
    float4 p = reinterpret_cast<float4*>(param)[i];
    float4 g = reinterpret_cast<float4*>(grad)[i];
    float4 s = reinterpret_cast<float4*>(sum)[i];
    upd(p.x, g.x, s.x);
    upd(p.y, g.y, s.y);
    upd(p.z, g.z, s.z);
    upd(p.w, g.w, s.w);
    reinterpret_cast<float4*>(param)[i] = p;
    reinterpret_cast<float4*>(grad)[i] = g;
    reinterpret_cast<float4*>(sum)[i] = s;
  }
  if (blockIdx.x == 0 && threadIdx.x < (numel & 3)) {
    int64_t i = n4 * 4 + threadIdx.x;
    upd(param[i], grad[i], sum[i]);
  }
}

// dst = src or dst = dst + src: the gradient sum over replicas run one after another (DGLStep replicas > 1)
__global__ void __launch_bounds__(256) grad_accumulate_kernel(float* __restrict__ dst, const float* __restrict__ src,
                                                              int64_t n4, int64_t numel, int accumulate) {
  pdl_enter();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
       i += (int64_t)gridDim.x * blockDim.x) {
    float4 s = reinterpret_cast<const float4*>(src)[i];
    if (accumulate) {
      const float4 d = reinterpret_cast<const float4*>(dst)[i];
      s.x = d.x + s.x; s.y = d.y + s.y; s.z = d.z + s.z; s.w = d.w + s.w;
    }
    reinterpret_cast<float4*>(dst)[i] = s;
  }
  // tail (numel not a multiple of 4)
  if (blockIdx.x == 0 && threadIdx.x < (numel & 3)) {
    int64_t i = n4 * 4 + threadIdx.x;
    dst[i] = accumulate ? dst[i] + src[i] : src[i];
  }
}

static unsigned elementwise_blocks(int64_t numel) {
  int64_t n4 = numel / 4;
  int64_t blocks = ceil_div64(n4 > 0 ? n4 : 1, 256);
  if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
  return (unsigned)blocks;
}

static char g_last_error[512] = "";

void set_last_error(const char* msg) { snprintf(g_last_error, sizeof(g_last_error), "%s", msg); }
int cuda_fail(cudaError_t e, const char* where) {
  snprintf(g_last_error, sizeof(g_last_error), "%s: %s", where, cudaGetErrorString(e));
  return GDL_ECUDA;
}

}  // namespace gdl

using namespace gdl;

extern "C" int gdl_version(void) { return GDL_B200_VERSION; }
extern "C" const char* gdl_last_error_string(void) { return g_last_error; }

extern "C" int gdl_init(int device) {
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceProperties");
  if (prop.major != 10) {
    snprintf(g_last_error, sizeof(g_last_error),
             "gdl_b200 needs an sm_100 (B200) device; device %d is sm_%d%d", device, prop.major, prop.minor);
    return GDL_EARCH;
  }
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
  return GDL_OK;
}

extern "C" int64_t gdl_optim_scratch_floats(int64_t numel, int nseg) {
  (void)nseg;
  return ceil_div64(numel, kChunk) * 3;
}

extern "C" int gdl_grad_stats(const float* grad, int64_t numel, const int64_t* seg_end,
                              const int32_t* seg_group, const float* seg_inv_numel, int nseg,
                              float max_norm, float* scratch, float* stats_out, gdl_stream_t s) {
  GDL_REQUIRE(grad && seg_end && seg_group && seg_inv_numel && scratch && stats_out, "gdl_grad_stats: null pointer");
  GDL_REQUIRE(numel > 0 && nseg > 0, "gdl_grad_stats: bad shape");
  int nblk = (int)ceil_div64(numel, kChunk);
  launch_pdl(grad_stats_kernel, nblk, kOptThreads, 0, (cudaStream_t)s, grad, numel, seg_end, seg_group,
                                                              seg_inv_numel, nseg, scratch);
  GDL_CHECK_LAUNCH("grad_stats_kernel");
  launch_pdl(grad_stats_finalize_kernel, 1, 256, 0, (cudaStream_t)s, scratch, nblk, max_norm, stats_out);
  GDL_CHECK_LAUNCH("grad_stats_finalize_kernel");
  return GDL_OK;
}

// The host-lr entries and the device-lr entries (*_lr_dev) launch the same kernels: lr_dev NULL selects lr_host.
static int sgd_momentum_launch(float* param, float* grad, float* momentum_buf, int64_t numel, float lr,
                               const double* lr_dev, float mu, float wd, int first_step, const float* stats,
                               gdl_stream_t s) {
  GDL_REQUIRE(param && grad && momentum_buf && numel > 0, "gdl_sgd_momentum: bad arguments");
  GDL_REQUIRE((((uintptr_t)param | (uintptr_t)grad | (uintptr_t)momentum_buf) & 15) == 0,
              "gdl_sgd_momentum: arenas must be 16-byte aligned");
  launch_pdl(sgd_momentum_kernel, elementwise_blocks(numel), 256, 0, (cudaStream_t)s, param, grad, momentum_buf,
             numel / 4, numel, lr, lr_dev, mu, wd, first_step, stats);
  GDL_CHECK_LAUNCH("sgd_momentum_kernel");
  return GDL_OK;
}

static int adam_launch(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int32_t* step_state,
                       int64_t numel, double lr, const double* lr_dev, double beta1, double beta2, double eps,
                       double wd, const float* stats, gdl_stream_t s) {
  GDL_REQUIRE(param && grad && exp_avg && exp_avg_sq && step_state && numel > 0, "gdl_adam: bad arguments");
  GDL_REQUIRE((((uintptr_t)param | (uintptr_t)grad | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) & 15) == 0,
              "gdl_adam: arenas must be 16-byte aligned");
  GDL_REQUIRE(beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0, "gdl_adam: betas must lie in [0, 1)");
  launch_pdl(optim_step_prologue_kernel, 1, 1, 0, (cudaStream_t)s, step_state, (int)kRuleAdam, lr, lr_dev, beta1,
             beta2);
  GDL_CHECK_LAUNCH("optim_step_prologue_kernel");
  launch_pdl(adam_kernel, elementwise_blocks(numel), 256, 0, (cudaStream_t)s, param, grad, exp_avg, exp_avg_sq,
             numel / 4, numel, (float)(1.0 - beta1), (float)beta2, (float)(1.0 - beta2), (float)eps, (float)wd,
             stats, (const int32_t*)step_state);
  GDL_CHECK_LAUNCH("adam_kernel");
  return GDL_OK;
}

static int adagrad_launch(float* param, float* grad, float* sum, int32_t* step_state, int64_t numel, double lr,
                          const double* lr_dev, double lr_decay, double eps, double wd, const float* stats,
                          gdl_stream_t s) {
  GDL_REQUIRE(param && grad && sum && step_state && numel > 0, "gdl_adagrad: bad arguments");
  GDL_REQUIRE((((uintptr_t)param | (uintptr_t)grad | (uintptr_t)sum) & 15) == 0,
              "gdl_adagrad: arenas must be 16-byte aligned");
  launch_pdl(optim_step_prologue_kernel, 1, 1, 0, (cudaStream_t)s, step_state, (int)kRuleAdagrad, lr, lr_dev,
             lr_decay, 0.0);
  GDL_CHECK_LAUNCH("optim_step_prologue_kernel");
  launch_pdl(adagrad_kernel, elementwise_blocks(numel), 256, 0, (cudaStream_t)s, param, grad, sum, numel / 4, numel,
             (float)eps, (float)wd, stats, (const int32_t*)step_state);
  GDL_CHECK_LAUNCH("adagrad_kernel");
  return GDL_OK;
}

extern "C" int gdl_sgd_momentum(float* param, float* grad, float* momentum_buf, int64_t numel,
                                float lr, float mu, float wd, int first_step, const float* stats,
                                gdl_stream_t s) {
  return sgd_momentum_launch(param, grad, momentum_buf, numel, lr, nullptr, mu, wd, first_step, stats, s);
}

extern "C" int gdl_sgd_momentum_lr_dev(float* param, float* grad, float* momentum_buf, int64_t numel,
                                       const double* lr, float mu, float wd, int first_step, const float* stats,
                                       gdl_stream_t s) {
  GDL_REQUIRE(lr, "gdl_sgd_momentum_lr_dev: null lr");
  return sgd_momentum_launch(param, grad, momentum_buf, numel, 0.f, lr, mu, wd, first_step, stats, s);
}

extern "C" int gdl_adam(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int32_t* step_state,
                        int64_t numel, double lr, double beta1, double beta2, double eps, double wd,
                        const float* stats, gdl_stream_t s) {
  return adam_launch(param, grad, exp_avg, exp_avg_sq, step_state, numel, lr, nullptr, beta1, beta2, eps, wd, stats,
                     s);
}

extern "C" int gdl_adam_lr_dev(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int32_t* step_state,
                               int64_t numel, const double* lr, double beta1, double beta2, double eps, double wd,
                               const float* stats, gdl_stream_t s) {
  GDL_REQUIRE(lr, "gdl_adam_lr_dev: null lr");
  return adam_launch(param, grad, exp_avg, exp_avg_sq, step_state, numel, 0.0, lr, beta1, beta2, eps, wd, stats, s);
}

extern "C" int gdl_adagrad(float* param, float* grad, float* sum, int32_t* step_state, int64_t numel, double lr,
                           double lr_decay, double eps, double wd, const float* stats, gdl_stream_t s) {
  return adagrad_launch(param, grad, sum, step_state, numel, lr, nullptr, lr_decay, eps, wd, stats, s);
}

extern "C" int gdl_adagrad_lr_dev(float* param, float* grad, float* sum, int32_t* step_state, int64_t numel,
                                  const double* lr, double lr_decay, double eps, double wd, const float* stats,
                                  gdl_stream_t s) {
  GDL_REQUIRE(lr, "gdl_adagrad_lr_dev: null lr");
  return adagrad_launch(param, grad, sum, step_state, numel, 0.0, lr, lr_decay, eps, wd, stats, s);
}

extern "C" int gdl_grad_accumulate(float* dst, const float* src, int64_t numel, int accumulate, gdl_stream_t s) {
  GDL_REQUIRE(dst && src && numel > 0, "gdl_grad_accumulate: bad arguments");
  GDL_REQUIRE((((uintptr_t)dst | (uintptr_t)src) & 15) == 0, "gdl_grad_accumulate: arenas must be 16-byte aligned");
  launch_pdl(grad_accumulate_kernel, elementwise_blocks(numel), 256, 0, (cudaStream_t)s, dst, src, numel / 4, numel,
             accumulate);
  GDL_CHECK_LAUNCH("grad_accumulate_kernel");
  return GDL_OK;
}
