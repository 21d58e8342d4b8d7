// elementwise.cu — the HBM-bound kernels of the DGL step: input layout conversion,
// BatchNorm (training mode) statistics / apply / backward, ReLU and residual add fused into
// the BN passes, MaxPool 3x3/s2, global average pooling.  All activations NHWC bf16, 16-byte
// vector accesses, fp32 math, deterministic fixed-order reductions (per-block partials reduced
// by a finalize kernel; no float atomics — reference utils/utils.py:12 asks for determinism).
#include <stdlib.h>
#include "common.cuh"

namespace gdl {

// ------------------------------------------------------------------------------------------
// layout: f32 [B,C,T,H,W] -> bf16 [B*T,H,W,8]      (reference models/backbone.py:162-164)
// ------------------------------------------------------------------------------------------
__global__ void layout_kernel(const float* __restrict__ src, bf16* __restrict__ dst, int B, int C,
                              int T, int H, int W) {
  const int64_t HW = (int64_t)H * W;
  const int64_t total = (int64_t)B * T * HW;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int64_t bt = i / HW;
    int64_t hw = i - bt * HW;
    int b = int(bt / T), t = int(bt - (int64_t)b * T);
    float f[8];
#pragma unroll
    for (int c = 0; c < 8; ++c)
      f[c] = c < C ? src[(((int64_t)b * C + c) * T + t) * HW + hw] : 0.f;
    *reinterpret_cast<uint4*>(dst + i * 8) = pack8(f);
  }
}

// ------------------------------------------------------------------------------------------
// BatchNorm statistics
// ------------------------------------------------------------------------------------------
constexpr int kBnThreads = 256;
constexpr int kBnMaxBlocks = 4 * kNumSMs;

// Sweep direction hint (gdl_set_sweep, include/gdl_b200.h): the grid-stride kernels below walk their pixel /
// vector range in ascending order, or descending when the hint is set.  A pass that runs opposite to the pass
// that last touched a tensor starts on the part of it that is still in the 126 MB L2 (the producer's tail)
// instead of on the part that was evicted first.  Two-pass operations (reduce + apply) run their second pass
// opposite to the first.  Element-wise results do not depend on it; reductions keep a fixed order per setting.
thread_local int g_sweep_rev = 0;
__device__ __forceinline__ int64_t sweep_idx(int64_t i, int64_t n, int rev) { return rev ? n - 1 - i : i; }

// Grid-stride kernels are launched with exactly one wave of co-resident CTAs (occupancy x 148 SMs): a fixed
// 4 x 148 grid left a 33 % partial second wave whenever register use allowed only 3 CTAs per SM.
template <typename K>
static int resident_blocks(K kernel, int threads) {
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
  return per_sm * kNumSMs;
}
#define GDL_RESIDENT(kernel, threads)                           \
  ([]() {                                                       \
    static const int v = resident_blocks(kernel, threads);      \
    return v;                                                   \
  }())

static int bn_blocks_cap(int64_t P, int C, int cap) {
  int lanes = kBnThreads / (C / 8);
  int64_t want = ceil_div64(P, (int64_t)lanes * 8);
  if (want < 1) want = 1;
  if (cap > kBnMaxBlocks) cap = kBnMaxBlocks;
  return int(want < cap ? want : cap);
}

// Reduce the 8-channel accumulators of all pixel lanes of a block; thread layout is
// tid = lane * (C/8) + cg.  Result (2 x C floats) is written to partial[block].
template <int NACC>
__device__ __forceinline__ void block_channel_reduce(float (&acc)[NACC][8], int C,
                                                     float* __restrict__ partial_blk) {
  __shared__ float red[kBnThreads * 8];
  const int groups = C / 8;
  const int lanes = kBnThreads / groups;
  const int cg = threadIdx.x % groups;
  const int lane = threadIdx.x / groups;
#pragma unroll
  for (int a = 0; a < NACC; ++a) {
    __syncthreads();
#pragma unroll
    for (int c = 0; c < 8; ++c) red[(lane * groups + cg) * 8 + c] = acc[a][c];
    __syncthreads();
    // fixed-order tree over lanes
    for (int stride = lanes / 2; stride > 0; stride >>= 1) {
      if (lane < stride) {
#pragma unroll
        for (int c = 0; c < 8; ++c)
          red[(lane * groups + cg) * 8 + c] += red[((lane + stride) * groups + cg) * 8 + c];
      }
      __syncthreads();
    }
    if (lane == 0) {
#pragma unroll
      for (int c = 0; c < 8; ++c) partial_blk[a * C + cg * 8 + c] = red[cg * 8 + c];
    }
  }
}

__global__ void __launch_bounds__(kBnThreads) bn_stats_kernel(const bf16* __restrict__ x, int64_t P,
                                                              int C, float* __restrict__ partial, int rev) {
  const int groups = C / 8;
  const int lanes = kBnThreads / groups;
  const int cg = threadIdx.x % groups;
  const int lane = threadIdx.x / groups;
  float acc[2][8];
#pragma unroll
  for (int c = 0; c < 8; ++c) acc[0][c] = acc[1][c] = 0.f;
  // four pixels in flight per thread (memory-level parallelism); the per-thread order stays fixed
  const int64_t stride = (int64_t)gridDim.x * lanes;
  int64_t pix = (int64_t)blockIdx.x * lanes + lane;
  for (; pix + 3 * stride < P; pix += 4 * stride) {
    uint4 u[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) u[k] = ld_stream16(x + sweep_idx(pix + k * stride, P, rev) * C + cg * 8);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float f[8];
      unpack8(u[k], f);
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        acc[0][c] += f[c];
        acc[1][c] = fmaf(f[c], f[c], acc[1][c]);
      }
    }
  }
  for (; pix < P; pix += stride) {
    float f[8];
    unpack8(ld_stream16(x + sweep_idx(pix, P, rev) * C + cg * 8), f);
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      acc[0][c] += f[c];
      acc[1][c] = fmaf(f[c], f[c], acc[1][c]);
    }
  }
  block_channel_reduce<2>(acc, C, partial + (size_t)blockIdx.x * 2 * C);
}

// One warp per channel: lanes stride over the per-block partials (fixed order), double
// accumulation, fixed shuffle tree => deterministic and ~100x shorter than a serial loop.
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void bn_stats_finalize_kernel(const float* __restrict__ partial, int nblk, int64_t P, int C,
                                         const float* __restrict__ gamma,
                                         const float* __restrict__ beta, float eps, float momentum,
                                         float* running_mean, float* running_var, float* mean_out,
                                         float* invstd_out, float* scale, float* shift) {
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (c >= C) return;
  double s1 = 0.0, s2 = 0.0;
  for (int b = lane; b < nblk; b += 32) {
    s1 += (double)partial[(size_t)b * 2 * C + c];
    s2 += (double)partial[(size_t)b * 2 * C + C + c];
  }
  s1 = warp_sum_d(s1);
  s2 = warp_sum_d(s2);
  if (lane != 0) return;
  double mean = s1 / (double)P;
  double var = s2 / (double)P - mean * mean;
  if (var < 0.0) var = 0.0;
  float invstd = (float)(1.0 / sqrt(var + (double)eps));
  float m = (float)mean;
  mean_out[c] = m;
  invstd_out[c] = invstd;
  float sc = gamma[c] * invstd;
  scale[c] = sc;
  shift[c] = beta[c] - m * sc;
  if (running_mean != nullptr) {
    double unbiased = P > 1 ? var * (double)P / (double)(P - 1) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * m;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
  }
}

// eval mode: fused affine from the running statistics (reference model.eval(), main_dgl.py:186)
__global__ void bn_eval_affine_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                                      const float* __restrict__ rm, const float* __restrict__ rv, float eps,
                                      float* __restrict__ scale, float* __restrict__ shift, int C) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float sc = gamma[c] * rsqrtf(rv[c] + eps);
  scale[c] = sc;
  shift[c] = beta[c] - rm[c] * sc;
}

// Per-channel coefficients of the element-wise passes live in REGISTERS: the grid stride (gridDim.x * blockDim.x) and the
// vector count are multiples of C/8, so a thread meets the same 8-channel group in every iteration.  (Shared-memory
// coefficient tables cost 2-5 LDS.128 per 16-byte vector, each 4-8 wavefronts because neighbouring lanes read different
// groups: ncu showed the L1/shared pipe at 80-94 % and DRAM at 50-68 % in bn_bwd_apply / bn_bwd_nores_apply.)
__device__ __forceinline__ int fixed_channel_group(int64_t first_vec, int64_t nvec, int groups, int rev) {
  const int cg = int(first_vec % groups);
  return rev ? groups - 1 - cg : cg;  // nvec % groups == 0: vector nvec-1-i belongs to group groups-1-(i % groups)
}

// y = [relu](x*scale + shift [+ res])
__global__ void __launch_bounds__(256) bn_apply_kernel(const bf16* __restrict__ x,
                                                       const bf16* __restrict__ res,
                                                       bf16* __restrict__ y, int64_t nvec, int C,
                                                       const float* __restrict__ scale,
                                                       const float* __restrict__ shift, int relu, int rev) {
  const int groups = C / 8;
  const int64_t first = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int cg = fixed_channel_group(first, nvec, groups, rev);
  float sc[8], sh[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    sc[c] = scale[cg * 8 + c];
    sh[c] = shift[cg * 8 + c];
  }
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  auto body = [&](int64_t i, const uint4& ux, const uint4& ur) {
    float f[8];
    unpack8(ux, f);
#pragma unroll
    for (int c = 0; c < 8; ++c) f[c] = fmaf(f[c], sc[c], sh[c]);
    if (res != nullptr) {
      float r[8];
      unpack8(ur, r);
#pragma unroll
      for (int c = 0; c < 8; ++c) f[c] += r[c];
    }
    if (relu) {
#pragma unroll
      for (int c = 0; c < 8; ++c) f[c] = fmaxf(f[c], 0.f);
    }
    *reinterpret_cast<uint4*>(y + i * 8) = pack8(f);
  };
  const uint4 zero4 = make_uint4(0, 0, 0, 0);
  int64_t i0 = first;
  for (; i0 + stride < nvec; i0 += 2 * stride) {  // two vectors (up to four loads) in flight per thread
    const int64_t j0 = sweep_idx(i0, nvec, rev), j1 = sweep_idx(i0 + stride, nvec, rev);
    const uint4 x0 = ld_stream16(x + j0 * 8), x1 = ld_stream16(x + j1 * 8);
    const uint4 r0 = res ? ld_stream16(res + j0 * 8) : zero4, r1 = res ? ld_stream16(res + j1 * 8) : zero4;
    body(j0, x0, r0);
    body(j1, x1, r1);
  }
  for (; i0 < nvec; i0 += stride) {
    const int64_t j = sweep_idx(i0, nvec, rev);
    body(j, ld_stream16(x + j * 8), res ? ld_stream16(res + j * 8) : zero4);
  }
}

// backward pass 1: dz = dy * (y > 0); partial sums of dz and dz * x (bn_bwd_finalize_raw_kernel forms sum(dz * xhat))
__global__ void __launch_bounds__(kBnThreads) bn_bwd_reduce_kernel(
    const bf16* dy, const bf16* __restrict__ y, const bf16* __restrict__ x, bf16* dz, int64_t P, int C,
    float* __restrict__ partial, int relu, int rev) {
  const int groups = C / 8;
  const int lanes = kBnThreads / groups;
  const int cg = threadIdx.x % groups;
  const int lane = threadIdx.x / groups;
  float acc[2][8];
#pragma unroll
  for (int c = 0; c < 8; ++c) acc[0][c] = acc[1][c] = 0.f;
  const int64_t stride = (int64_t)gridDim.x * lanes;
  int64_t pix = (int64_t)blockIdx.x * lanes + lane;
  auto body = [&](int64_t off, const uint4& ug, const uint4& ux, const uint4& uy) {
    float g[8], xv[8];
    unpack8(ug, g);
    unpack8(ux, xv);
    if (relu) {
      float yv[8];
      unpack8(uy, yv);
#pragma unroll
      for (int c = 0; c < 8; ++c) g[c] = yv[c] > 0.f ? g[c] : 0.f;
      *reinterpret_cast<uint4*>(dz + off) = pack8(g);
    }
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      acc[0][c] += g[c];
      acc[1][c] = fmaf(g[c], xv[c], acc[1][c]);
    }
  };
  const uint4 zero4 = make_uint4(0, 0, 0, 0);
  for (; pix + stride < P; pix += 2 * stride) {  // two pixels in flight; dz may alias dy: no .nc path for dy
    const int64_t o0 = sweep_idx(pix, P, rev) * C + cg * 8, o1 = sweep_idx(pix + stride, P, rev) * C + cg * 8;
    const uint4 g0 = *reinterpret_cast<const uint4*>(dy + o0), x0 = ld_stream16(x + o0);
    const uint4 g1 = *reinterpret_cast<const uint4*>(dy + o1), x1 = ld_stream16(x + o1);
    const uint4 y0 = relu ? ld_stream16(y + o0) : zero4, y1 = relu ? ld_stream16(y + o1) : zero4;
    body(o0, g0, x0, y0);
    body(o1, g1, x1, y1);
  }
  for (; pix < P; pix += stride) {
    const int64_t off = sweep_idx(pix, P, rev) * C + cg * 8;
    body(off, *reinterpret_cast<const uint4*>(dy + off), ld_stream16(x + off), relu ? ld_stream16(y + off) : zero4);
  }
  block_channel_reduce<2>(acc, C, partial + (size_t)blockIdx.x * 2 * C);
}

__global__ void bn_bwd_finalize_kernel(const float* __restrict__ partial, int nblk, int C,
                                       float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (c >= C) return;
  double s1 = 0.0, s2 = 0.0;
  for (int b = lane; b < nblk; b += 32) {
    s1 += (double)partial[(size_t)b * 2 * C + c];
    s2 += (double)partial[(size_t)b * 2 * C + C + c];
  }
  s1 = warp_sum_d(s1);
  s2 = warp_sum_d(s2);
  if (lane == 0) {
    dbeta[c] = (float)s1;
    dgamma[c] = (float)s2;
  }
}

// backward pass 2: dx = gamma*invstd*(dz - dbeta/P - xhat*dgamma/P)
__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(
    const bf16* __restrict__ dz, const bf16* __restrict__ x, bf16* __restrict__ dx, int64_t nvec,
    int C, float invP, const float* __restrict__ gamma, const float* __restrict__ mean,
    const float* __restrict__ invstd, const float* __restrict__ dgamma,
    const float* __restrict__ dbeta, int rev) {
  // dx = a*dz + b*x + c  with  a = gamma*invstd,  b = -a*invstd*dgamma/P,
  //                            c = -a*dbeta/P - b*mean          (per channel, in registers: see fixed_channel_group)
  const int groups = C / 8;
  const int64_t first = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int cg = fixed_channel_group(first, nvec, groups, rev);
  float ka[8], kb[8], kc[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int ch = cg * 8 + c;
    const float a = gamma[ch] * invstd[ch];
    const float b = -a * invstd[ch] * dgamma[ch] * invP;
    ka[c] = a;
    kb[c] = b;
    kc[c] = -a * dbeta[ch] * invP - b * mean[ch];
  }
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  auto body = [&](int64_t i, const uint4& ug, const uint4& ux) {
    float g[8], xv[8];
    unpack8(ug, g);
    unpack8(ux, xv);
#pragma unroll
    for (int c = 0; c < 8; ++c) g[c] = fmaf(ka[c], g[c], fmaf(kb[c], xv[c], kc[c]));
    *reinterpret_cast<uint4*>(dx + i * 8) = pack8(g);
  };
  int64_t i = first;
  for (; i + stride < nvec; i += 2 * stride) {
    const int64_t j0 = sweep_idx(i, nvec, rev), j1 = sweep_idx(i + stride, nvec, rev);
    const uint4 g0 = ld_stream16(dz + j0 * 8), x0 = ld_stream16(x + j0 * 8);
    const uint4 g1 = ld_stream16(dz + j1 * 8), x1 = ld_stream16(x + j1 * 8);
    body(j0, g0, x0);
    body(j1, g1, x1);
  }
  for (; i < nvec; i += stride) {
    const int64_t j = sweep_idx(i, nvec, rev);
    body(j, ld_stream16(dz + j * 8), ld_stream16(x + j * 8));
  }
}

// ------------------------------------------------------------------------------------------
// MaxPool2d(kernel 3, stride 2, pad 1)       (reference models/backbone.py:106)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) maxpool_fwd_kernel(const bf16* __restrict__ x,
                                                          bf16* __restrict__ y,
                                                          uint8_t* __restrict__ amax, int N, int H,
                                                          int W, int C, int Ho, int Wo) {
  const int groups = C / 8;
  const int64_t total = (int64_t)N * Ho * Wo * groups;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int cg = int(i % groups);
    int64_t pix = i / groups;
    int wo = int(pix % Wo);
    int64_t t = pix / Wo;
    int ho = int(t % Ho);
    int n = int(t / Ho);
    float best[8];
    int bi[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      best[c] = -INFINITY;
      bi[c] = 0;
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      int h = ho * 2 - 1 + r;
      if (h < 0 || h >= H) continue;
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        int w = wo * 2 - 1 + s;
        if (w < 0 || w >= W) continue;
        float f[8];
        unpack8(*reinterpret_cast<const uint4*>(x + (((int64_t)n * H + h) * W + w) * C + cg * 8), f);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          if (f[c] > best[c]) {  // strict: the first maximum in scan order wins (ATen rule)
            best[c] = f[c];
            bi[c] = r * 3 + s;
          }
        }
      }
    }
    *reinterpret_cast<uint4*>(y + pix * C + cg * 8) = pack8(best);
    uint2 packed;
    packed.x = uint32_t(bi[0]) | (uint32_t(bi[1]) << 8) | (uint32_t(bi[2]) << 16) | (uint32_t(bi[3]) << 24);
    packed.y = uint32_t(bi[4]) | (uint32_t(bi[5]) << 8) | (uint32_t(bi[6]) << 16) | (uint32_t(bi[7]) << 24);
    *reinterpret_cast<uint2*>(amax + pix * C + cg * 8) = packed;
  }
}

__global__ void __launch_bounds__(256) maxpool_bwd_kernel(const bf16* __restrict__ dy,
                                                          const uint8_t* __restrict__ amax,
                                                          bf16* __restrict__ dx, int N, int H, int W,
                                                          int C, int Ho, int Wo) {
  const int groups = C / 8;
  const int64_t total = (int64_t)N * H * W * groups;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int cg = int(i % groups);
    int64_t pix = i / groups;
    int w = int(pix % W);
    int64_t t = pix / W;
    int h = int(t % H);
    int n = int(t / H);
    float acc[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] = 0.f;
    int ho_lo = h >> 1, ho_hi = (h + 1) >> 1;  // windows ho with 2*ho-1 <= h <= 2*ho+1
    int wo_lo = w >> 1, wo_hi = (w + 1) >> 1;
    for (int ho = ho_lo; ho <= ho_hi; ++ho) {
      if (ho >= Ho) continue;
      int r = h - (ho * 2 - 1);
      for (int wo = wo_lo; wo <= wo_hi; ++wo) {
        if (wo >= Wo) continue;
        int s = w - (wo * 2 - 1);
        int idx = r * 3 + s;
        int64_t o = (((int64_t)n * Ho + ho) * Wo + wo) * C + cg * 8;
        uint2 am = *reinterpret_cast<const uint2*>(amax + o);
        float g[8];
        unpack8(*reinterpret_cast<const uint4*>(dy + o), g);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          uint32_t word = c < 4 ? am.x : am.y;
          int a = (word >> ((c & 3) * 8)) & 0xff;
          if (a == idx) acc[c] += g[c];
        }
      }
    }
    *reinterpret_cast<uint4*>(dx + pix * C + cg * 8) = pack8(acc);
  }
}

// ------------------------------------------------------------------------------------------
// BatchNorm backward for units WITHOUT a residual input (conv1 of a BasicBlock, reference
// models/backbone.py:44-46): the ReLU mask is recomputed from x (y > 0  <=>  x*scale+shift > 0), so
// neither y is read nor the masked gradient written: 10 B/element instead of 14.
// ------------------------------------------------------------------------------------------
// The reduce pass accumulates sum(dz) and sum(dz * x); the finalize kernel turns the second into
// sum(dz * xhat) = invstd * (sum(dz * x) - mean * sum(dz)) in double precision (5 instead of 8 instructions per
// element and 16 registers fewer: three CTAs per SM instead of two — the kernel was latency bound at 25 % occupancy).
__global__ void __launch_bounds__(kBnThreads, 3) bn_bwd_nores_reduce_kernel(
    const bf16* __restrict__ dy, const bf16* __restrict__ x, int64_t P, int C, const float* __restrict__ scale,
    const float* __restrict__ shift, float* __restrict__ partial, int rev) {
  const int groups = C / 8;
  const int lanes = kBnThreads / groups;
  const int cg = threadIdx.x % groups;
  const int lane = threadIdx.x / groups;
  float sc[8], sh[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    sc[c] = scale[cg * 8 + c];
    sh[c] = shift[cg * 8 + c];
  }
  float acc[2][8];
#pragma unroll
  for (int c = 0; c < 8; ++c) acc[0][c] = acc[1][c] = 0.f;
  const int64_t stride = (int64_t)gridDim.x * lanes;
  int64_t pix = (int64_t)blockIdx.x * lanes + lane;
  auto body = [&](const uint4& ug, const uint4& ux) {
    float g[8], xv[8];
    unpack8(ug, g);
    unpack8(ux, xv);
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const float gz = fmaf(xv[c], sc[c], sh[c]) > 0.f ? g[c] : 0.f;
      acc[0][c] += gz;
      acc[1][c] = fmaf(gz, xv[c], acc[1][c]);
    }
  };
  for (; pix + 3 * stride < P; pix += 4 * stride) {  // four pixels (eight 16-byte loads) in flight per thread
    uint4 g[4], xx[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int64_t o = sweep_idx(pix + k * stride, P, rev) * C + cg * 8;
      g[k] = ld_stream16(dy + o);
      xx[k] = ld_stream16(x + o);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) body(g[k], xx[k]);
  }
  for (; pix < P; pix += stride) {
    const int64_t off = sweep_idx(pix, P, rev) * C + cg * 8;
    body(ld_stream16(dy + off), ld_stream16(x + off));
  }
  block_channel_reduce<2>(acc, C, partial + (size_t)blockIdx.x * 2 * C);
}

// partials hold (sum dz, sum dz*x): dbeta = s1, dgamma = invstd * (s2 - mean * s1)
__global__ void bn_bwd_finalize_raw_kernel(const float* __restrict__ partial, int nblk, int C,
                                           const float* __restrict__ mean, const float* __restrict__ invstd,
                                           float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (c >= C) return;
  double s1 = 0.0, s2 = 0.0;
  for (int b = lane; b < nblk; b += 32) {
    s1 += (double)partial[(size_t)b * 2 * C + c];
    s2 += (double)partial[(size_t)b * 2 * C + C + c];
  }
  s1 = warp_sum_d(s1);
  s2 = warp_sum_d(s2);
  if (lane == 0) {
    dbeta[c] = (float)s1;
    dgamma[c] = (float)((double)invstd[c] * (s2 - (double)mean[c] * s1));
  }
}

__global__ void __launch_bounds__(256) bn_bwd_nores_apply_kernel(
    const bf16* __restrict__ dy, const bf16* __restrict__ x, bf16* __restrict__ dx, int64_t nvec, int C,
    float invP, const float* __restrict__ gamma, const float* __restrict__ mean,
    const float* __restrict__ invstd, const float* __restrict__ scale, const float* __restrict__ shift,
    const float* __restrict__ dgamma, const float* __restrict__ dbeta, int rev) {
  const int groups = C / 8;
  const int64_t first = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int cg = fixed_channel_group(first, nvec, groups, rev);
  float ka[8], kb[8], kc[8], sc[8], sh[8];  // per-channel coefficients in registers (see fixed_channel_group)
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int ch = cg * 8 + c;
    const float a = gamma[ch] * invstd[ch];
    const float b = -a * invstd[ch] * dgamma[ch] * invP;
    ka[c] = a;
    kb[c] = b;
    kc[c] = -a * dbeta[ch] * invP - b * mean[ch];
    sc[c] = scale[ch];
    sh[c] = shift[ch];
  }
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  auto body = [&](int64_t i, const uint4& ug, const uint4& ux) {
    float g[8], xv[8];
    unpack8(ug, g);
    unpack8(ux, xv);
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const float gz = fmaf(xv[c], sc[c], sh[c]) > 0.f ? g[c] : 0.f;
      g[c] = fmaf(ka[c], gz, fmaf(kb[c], xv[c], kc[c]));
    }
    *reinterpret_cast<uint4*>(dx + i * 8) = pack8(g);
  };
  int64_t i = first;
  for (; i + stride < nvec; i += 2 * stride) {  // two vectors (four loads) in flight per thread
    const int64_t j0 = sweep_idx(i, nvec, rev), j1 = sweep_idx(i + stride, nvec, rev);
    const uint4 g0 = ld_stream16(dy + j0 * 8), x0 = ld_stream16(x + j0 * 8);
    const uint4 g1 = ld_stream16(dy + j1 * 8), x1 = ld_stream16(x + j1 * 8);
    body(j0, g0, x0);
    body(j1, g1, x1);
  }
  for (; i < nvec; i += stride) {
    const int64_t j = sweep_idx(i, nvec, rev);
    body(j, ld_stream16(dy + j * 8), ld_stream16(x + j * 8));
  }
}

// ------------------------------------------------------------------------------------------
// Stem tail fused: BN-apply + ReLU + MaxPool(3, s2, p1) forward (reference models/backbone.py:104-106)
// and its backward (max-pool scatter + ReLU mask + BN backward).  The stem activation
// y0 = relu(bn(x0)) — the largest tensor of the step — and its gradient are never materialised:
// forward reads x0 and writes the pooled map + 1-byte arg-max; backward gathers the pooled gradient
// through the arg-max and recomputes the ReLU mask from x0.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float bf16_round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

__global__ void __launch_bounds__(256) bn_relu_maxpool_fwd_kernel(
    const bf16* __restrict__ x, const float* __restrict__ scale, const float* __restrict__ shift,
    bf16* __restrict__ y, uint8_t* __restrict__ amax, bf16* __restrict__ xmax, int N, int H, int W, int C, int Ho,
    int Wo) {
  __shared__ float s_scale[512], s_shift[512];
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    s_scale[c] = scale[c];
    s_shift[c] = shift[c];
  }
  __syncthreads();
  const int groups = C / 8;
  const int64_t total = (int64_t)N * Ho * Wo * groups;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int cg = int(i % groups);
    int64_t pix = i / groups;
    int wo = int(pix % Wo);
    int64_t t = pix / Wo;
    int ho = int(t % Ho);
    int n = int(t / Ho);
    float sc[8], sh[8], best[8], bx[8];
    int bi[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      sc[c] = s_scale[cg * 8 + c];
      sh[c] = s_shift[cg * 8 + c];
      best[c] = -INFINITY;
      bx[c] = 0.f;
      bi[c] = 0;
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      int h = ho * 2 - 1 + r;
      if (h < 0 || h >= H) continue;
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        int w = wo * 2 - 1 + s;
        if (w < 0 || w >= W) continue;
        float f[8];
        unpack8(*reinterpret_cast<const uint4*>(x + (((int64_t)n * H + h) * W + w) * C + cg * 8), f);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          // the value the unfused path would have stored: bf16(relu(x*scale+shift))
          const float v = bf16_round(fmaxf(fmaf(f[c], sc[c], sh[c]), 0.f));
          if (v > best[c]) {  // strict: the first maximum in scan order wins (ATen rule)
            best[c] = v;
            bx[c] = f[c];
            bi[c] = r * 3 + s;
          }
        }
      }
    }
    *reinterpret_cast<uint4*>(y + pix * C + cg * 8) = pack8(best);
    // the conv output AT the arg-max (exact: f came from bf16): lets the backward form the BN sums on the
    // pooled grid (4x fewer elements) instead of a pass over the whole stem output
    if (xmax != nullptr) *reinterpret_cast<uint4*>(xmax + pix * C + cg * 8) = pack8(bx);
    uint2 packed;
    packed.x = uint32_t(bi[0]) | (uint32_t(bi[1]) << 8) | (uint32_t(bi[2]) << 16) | (uint32_t(bi[3]) << 24);
    packed.y = uint32_t(bi[4]) | (uint32_t(bi[5]) << 8) | (uint32_t(bi[6]) << 16) | (uint32_t(bi[7]) << 24);
    *reinterpret_cast<uint2*>(amax + pix * C + cg * 8) = packed;
  }
}

// BN+ReLU+rounding of two channels in one cvt.rn.relu.bf16x2: the rounded activation is a non-negative bf16, so its
// fp32 bit pattern orders like the value and has 16 free low bits for an arg-max tag (the keys below).
__device__ __forceinline__ uint32_t relu_pack_bf16x2(float hi, float lo) {
  uint32_t r;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r & 0x7fff7fffu;  // -0 -> +0: the keys below compare as unsigned integers
}

// Column sweep.  One thread per (image, segment of kTailSeg output rows, output column, 8-channel group) walks
// down its column: every input row is loaded and BN+ReLU-evaluated ONCE per thread (3 pixels: 1.5 evaluations per
// output-row pixel instead of 6.25 per 2x2 block), the max is separable — horizontal max of a row with the column tag
// (2 - s) in the key's low bits, then vertical max with the row tag 3*(2 - r) added — and the bottom row of one window
// is the top row of the next.  Key = bf16 bits of the activation << 16 | (8 - tap): one unsigned max per candidate gives
// the value and the FIRST arg-max in scan order (ATen's rule).  ~330 instructions per output pixel and 8 channels
// (~640 for one thread per 2x2 output block), all six loads of an iteration issued before any is consumed.
constexpr int kTailSeg = 14;

__device__ __forceinline__ void tail_row_keys(const uint4& u, const float (&sc)[8], const float (&sh)[8], uint32_t tag,
                                              uint32_t (&k)[8]) {
  const uint32_t wd[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float f0 = __uint_as_float(wd[j] << 16), f1 = __uint_as_float(wd[j] & 0xffff0000u);
    const uint32_t pk = relu_pack_bf16x2(fmaf(f1, sc[2 * j + 1], sh[2 * j + 1]), fmaf(f0, sc[2 * j], sh[2 * j]));
    k[2 * j] = __byte_perm(pk, tag, 0x1054);      // (low half of pk) << 16 | tag
    k[2 * j + 1] = __byte_perm(pk, tag, 0x3254);  // (high half of pk) << 16 | tag
  }
}

__global__ void __launch_bounds__(256, 3) bn_relu_maxpool_fwd3_kernel(
    const bf16* __restrict__ x, const float* __restrict__ scale, const float* __restrict__ shift,
    bf16* __restrict__ y, uint8_t* __restrict__ amax, bf16* __restrict__ xmax, int N, int H, int W, int C, int Ho,
    int Wo, int nseg, int seglen, int rev) {
  __shared__ int s_tapoff[16];  // element offset of tap (r,s) from the window's top-left pixel
  if (threadIdx.x < 9) s_tapoff[threadIdx.x] = ((threadIdx.x / 3) * W + threadIdx.x % 3) * C;
  __syncthreads();
  const int groups = C / 8;
  const int total = N * nseg * Wo * groups;  // 32-bit index arithmetic: the launcher checks the element count of x
  for (int i0 = blockIdx.x * blockDim.x + threadIdx.x; i0 < total; i0 += gridDim.x * blockDim.x) {
    const int i = rev ? total - 1 - i0 : i0;
    const int cg = i % groups;
    int t = i / groups;
    const int wo = t % Wo;
    t /= Wo;
    const int seg = t % nseg;
    const int n = t / nseg;
    float sc[8], sh[8];
    {
      const float4 a0 = __ldg(reinterpret_cast<const float4*>(scale + cg * 8)), a1 = __ldg(reinterpret_cast<const float4*>(scale + cg * 8 + 4));
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(shift + cg * 8)), b1 = __ldg(reinterpret_cast<const float4*>(shift + cg * 8 + 4));
      sc[0] = a0.x; sc[1] = a0.y; sc[2] = a0.z; sc[3] = a0.w; sc[4] = a1.x; sc[5] = a1.y; sc[6] = a1.z; sc[7] = a1.w;
      sh[0] = b0.x; sh[1] = b0.y; sh[2] = b0.z; sh[3] = b0.w; sh[4] = b1.x; sh[5] = b1.y; sh[6] = b1.z; sh[7] = b1.w;
    }
    const bf16* xn = x + (int64_t)n * H * W * C + cg * 8;
    const int w0 = 2 * wo - 1;
    const bool lv = w0 >= 0, rv = w0 + 2 < W;
    const int e0 = (lv ? w0 : 0) * C, e1 = (w0 + 1) * C, e2 = (rv ? w0 + 2 : w0 + 1) * C;  // clamped column offsets
    const int rowe = W * C;
    auto hmax = [&](const uint4& u0, const uint4& u1, const uint4& u2, uint32_t (&hm)[8]) {
      tail_row_keys(u1, sc, sh, 1u, hm);
      uint32_t k[8];
      if (lv) {
        tail_row_keys(u0, sc, sh, 2u, k);
#pragma unroll
        for (int c = 0; c < 8; ++c) hm[c] = max(hm[c], k[c]);
      }
      if (rv) {
        tail_row_keys(u2, sc, sh, 0u, k);
#pragma unroll
        for (int c = 0; c < 8; ++c) hm[c] = max(hm[c], k[c]);
      }
    };
    const int ho0 = seg * seglen, ho1 = min(ho0 + seglen, Ho);
    uint32_t carry[8];
    uint32_t carry_tag = 0u;  // 6 once the carried row exists (it is row r = 0 of the next window)
    if (ho0 > 0) {
      const bf16* xr = xn + (2 * ho0 - 1) * rowe;
      const uint4 u0 = ld_keep16(xr + e0), u1 = ld_keep16(xr + e1), u2 = ld_keep16(xr + e2);
      hmax(u0, u1, u2, carry);
      carry_tag = 6u;
    } else {
#pragma unroll
      for (int c = 0; c < 8; ++c) carry[c] = 0u;
    }
    for (int ho = ho0; ho < ho1; ++ho) {
      const bool dv = 2 * ho + 1 < H;
      const bf16* xa = xn + (2 * ho) * rowe;
      const bf16* xb = xa + (dv ? rowe : 0);
      const uint4 a0 = ld_keep16(xa + e0), a1 = ld_keep16(xa + e1), a2 = ld_keep16(xa + e2);
      const uint4 b0 = ld_keep16(xb + e0), b1 = ld_keep16(xb + e1), b2 = ld_keep16(xb + e2);
      uint32_t mid[8], bot[8], key[8];
      hmax(a0, a1, a2, mid);
      if (dv) {
        hmax(b0, b1, b2, bot);
      } else {
#pragma unroll
        for (int c = 0; c < 8; ++c) bot[c] = 0u;
      }
#pragma unroll
      for (int c = 0; c < 8; ++c) key[c] = max(max(carry[c] + carry_tag, mid[c] + 3u), bot[c]);
      const int64_t off = (int64_t)((n * Ho + ho) * Wo + wo) * C + cg * 8;
      uint4 yv;
      uint32_t* yw = reinterpret_cast<uint32_t*>(&yv);
      uint32_t tap[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) tap[c] = 8u - (key[c] & 15u);
#pragma unroll
      for (int j = 0; j < 4; ++j) yw[j] = __byte_perm(key[2 * j], key[2 * j + 1], 0x7632);
      *reinterpret_cast<uint4*>(y + off) = yv;
      uint2 packed;
      packed.x = tap[0] | (tap[1] << 8) | (tap[2] << 16) | (tap[3] << 24);
      packed.y = tap[4] | (tap[5] << 8) | (tap[6] << 16) | (tap[7] << 24);
      *reinterpret_cast<uint2*>(amax + off) = packed;
      if (xmax != nullptr) {
        // conv output at the arg-max: re-read (L1 hit) through the tap-offset table
        const unsigned short* xw = reinterpret_cast<const unsigned short*>(xn) + ((2 * ho - 1) * W + w0) * C;
        uint32_t xb16[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) xb16[c] = xw[s_tapoff[tap[c]] + c];
        uint4 xv;
        xv.x = xb16[0] | (xb16[1] << 16);
        xv.y = xb16[2] | (xb16[3] << 16);
        xv.z = xb16[4] | (xb16[5] << 16);
        xv.w = xb16[6] | (xb16[7] << 16);
        *reinterpret_cast<uint4*>(xmax + off) = xv;
      }
#pragma unroll
      for (int c = 0; c < 8; ++c) carry[c] = bot[c];
      carry_tag = 6u;
    }
  }
}

// Backward works on 2x2 blocks of stem pixels (rows 2i,2i+1 x cols 2j,2j+1; 8 channels per thread): the
// block is covered by the four pooling windows (i,j), (i,j+1), (i+1,j), (i+1,j+1), and which tap of which
// window each of the four pixels is follows from the parities alone, so one thread loads 4 windows for 4
// pixels (a per-pixel gather loads 9) with compile-time tap indices.
struct PoolWin {
  float g[8];
  uint32_t a0, a1;  // 8 one-byte arg-max indices
};
__device__ __forceinline__ float win_pick(const PoolWin& w, int c, int tap) {
  const uint32_t word = c < 4 ? w.a0 : w.a1;
  return ((word >> ((c & 3) * 8)) & 0xffu) == (uint32_t)tap ? w.g[c] : 0.f;
}
// dy (gradient wrt relu output) of the four pixels of block (i,j): p[0]=(2i,2j) p[1]=(2i,2j+1) p[2]=(2i+1,2j) p[3]=(2i+1,2j+1).
// Summation order per pixel = ascending (ho, wo), the order of the unfused max-pool backward.
// All loads of a block — four pooling windows (gradient + arg-max bytes) and the four stem pixels — are issued
// UNCONDITIONALLY on clamped addresses before anything is consumed (a window / pixel outside the map is masked
// afterwards): with a branch around each load the kernel had one request in flight per thread (2.6 TB/s).
struct PoolBlock {
  PoolWin w00, w01, w10, w11;
  uint4 xq[4];
  bool okq[4];
  int64_t offq[4];
};
__device__ __forceinline__ void set_win(PoolWin& w, const uint4& g, const uint2& am, bool ok) {
  unpack8(g, w.g);
  w.a0 = ok ? am.x : 0xffffffffu;  // 0xff matches no tap
  w.a1 = ok ? am.y : 0xffffffffu;
}
__device__ __forceinline__ void load_block(const bf16* __restrict__ gpool, const uint8_t* __restrict__ amax,
                                           const bf16* __restrict__ x, int n, int i, int j, int cg, int C, int H,
                                           int W, int Ho, int Wo, PoolBlock& b) {
  const int64_t base = (((int64_t)n * Ho + i) * Wo + j) * C + cg * 8;
  const bool okj = j + 1 < Wo, oki = i + 1 < Ho;
  const int64_t dj = okj ? C : 0, di = oki ? (int64_t)Wo * C : 0;
  const uint4 g00 = ld_keep16(gpool + base), g01 = ld_keep16(gpool + base + dj);
  const uint4 g10 = ld_keep16(gpool + base + di), g11 = ld_keep16(gpool + base + di + dj);
  const uint2 a00 = ld_keep8(amax + base), a01 = ld_keep8(amax + base + dj);
  const uint2 a10 = ld_keep8(amax + base + di), a11 = ld_keep8(amax + base + di + dj);
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int h = 2 * i + (q >> 1), w = 2 * j + (q & 1);
    b.okq[q] = h < H && w < W;
    b.offq[q] = (((int64_t)n * H + min(h, H - 1)) * W + min(w, W - 1)) * C + cg * 8;
    b.xq[q] = ld_stream16(x + b.offq[q]);
  }
  set_win(b.w00, g00, a00, true);
  set_win(b.w01, g01, a01, okj);
  set_win(b.w10, g10, a10, oki);
  set_win(b.w11, g11, a11, oki && okj);
}
__device__ __forceinline__ void block_pool_grad(const PoolBlock& b, float (&p)[4][8]) {
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    p[0][c] = win_pick(b.w00, c, 4);
    p[1][c] = win_pick(b.w00, c, 5) + win_pick(b.w01, c, 3);
    p[2][c] = win_pick(b.w00, c, 7) + win_pick(b.w10, c, 1);
    p[3][c] = ((win_pick(b.w00, c, 8) + win_pick(b.w01, c, 6)) + win_pick(b.w10, c, 2)) + win_pick(b.w11, c, 0);
  }
}

__global__ void __launch_bounds__(kBnThreads) bn_relu_maxpool_bwd_reduce_kernel(
    const bf16* __restrict__ gpool, const uint8_t* __restrict__ amax, const bf16* __restrict__ x, int N, int H,
    int W, int C, int Ho, int Wo, const float* __restrict__ mean, const float* __restrict__ invstd,
    const float* __restrict__ scale, const float* __restrict__ shift, float* __restrict__ partial) {
  const int groups = C / 8;
  const int lanes = kBnThreads / groups;
  const int cg = threadIdx.x % groups;
  const int lane = threadIdx.x / groups;
  float mu[8], is[8], sc[8], sh[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    mu[c] = mean[cg * 8 + c];
    is[c] = invstd[cg * 8 + c];
    sc[c] = scale[cg * 8 + c];
    sh[c] = shift[cg * 8 + c];
  }
  float acc[2][8];
#pragma unroll
  for (int c = 0; c < 8; ++c) acc[0][c] = acc[1][c] = 0.f;
  const int64_t nblk = (int64_t)N * Ho * Wo;  // one 2x2 block per pooling-window origin
  for (int64_t b = (int64_t)blockIdx.x * lanes + lane; b < nblk; b += (int64_t)gridDim.x * lanes) {
    const int j = int(b % Wo);
    const int64_t t = b / Wo;
    const int i = int(t % Ho), n = int(t / Ho);
    PoolBlock blk;
    load_block(gpool, amax, x, n, i, j, cg, C, H, W, Ho, Wo, blk);
    float p[4][8];
    block_pool_grad(blk, p);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float xv[8];
      unpack8(blk.xq[q], xv);
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        // the pooled gradient was stored in bf16 by the unfused path; keep that rounding point
        const float gz = (blk.okq[q] && fmaf(xv[c], sc[c], sh[c]) > 0.f) ? bf16_round(p[q][c]) : 0.f;
        acc[0][c] += gz;
        acc[1][c] = fmaf(gz, (xv[c] - mu[c]) * is[c], acc[1][c]);
      }
    }
  }
  block_channel_reduce<2>(acc, C, partial + (size_t)blockIdx.x * 2 * C);
}

__global__ void __launch_bounds__(256, 2) bn_relu_maxpool_bwd_apply_kernel(
    const bf16* __restrict__ gpool, const uint8_t* __restrict__ amax, const bf16* __restrict__ x,
    bf16* __restrict__ dx, int N, int H, int W, int C, int Ho, int Wo, float invP,
    const float* __restrict__ gamma, const float* __restrict__ mean, const float* __restrict__ invstd,
    const float* __restrict__ scale, const float* __restrict__ shift, const float* __restrict__ dgamma,
    const float* __restrict__ dbeta) {
  // per-channel coefficients in registers: the grid stride is a multiple of C/8, so a thread keeps its channel group
  // (the shared-memory tables cost 40 LDS.128 per block); block indices are 32-bit (the launcher checks the range)
  const int groups = C / 8;
  const int first = blockIdx.x * blockDim.x + threadIdx.x;
  const int cg = first % groups;
  float ka[8], kb[8], kc[8], sc[8], sh[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int ch = cg * 8 + c;
    const float a = gamma[ch] * invstd[ch];
    const float b = -a * invstd[ch] * dgamma[ch] * invP;
    ka[c] = a;
    kb[c] = b;
    kc[c] = -a * dbeta[ch] * invP - b * mean[ch];
    sc[c] = scale[ch];
    sh[c] = shift[ch];
  }
  const int total = N * Ho * Wo * groups;
  const int stride = gridDim.x * blockDim.x;
  for (int idx = first; idx < total; idx += stride) {
    {  // L2 prefetch of the four stem pixels of this thread's NEXT iteration (ptxas sinks three of the four
       // x loads of load_block behind the stores; a full iteration of lead hides their DRAM latency)
      const int idx2 = idx + stride;
      if (idx2 < total) {
        const int b2 = idx2 / groups;
        const int j2 = b2 % Wo;
        const int t2 = b2 / Wo;
        const int i2 = t2 % Ho;
        const bf16* xb = x + (((int64_t)(t2 / Ho) * H + min(2 * i2, H - 1)) * W + min(2 * j2, W - 1)) * C + cg * 8;
        const int dw = 2 * j2 + 1 < W ? C : 0, dh = 2 * i2 + 1 < H ? W * C : 0;
        prefetch_l2(xb);
        prefetch_l2(xb + dw);
        prefetch_l2(xb + dh);
        prefetch_l2(xb + dh + dw);
      }
    }
    const int b = idx / groups;
    const int j = b % Wo;
    const int t = b / Wo;
    const int i = t % Ho, n = t / Ho;
    PoolBlock blk;
    load_block(gpool, amax, x, n, i, j, cg, C, H, W, Ho, Wo, blk);
    float p[4][8];
    block_pool_grad(blk, p);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int64_t off = blk.offq[q];
      float xv[8], o[8];
      unpack8(blk.xq[q], xv);
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const float gz = fmaf(xv[c], sc[c], sh[c]) > 0.f ? bf16_round(p[q][c]) : 0.f;
        o[c] = fmaf(ka[c], gz, fmaf(kb[c], xv[c], kc[c]));
      }
      if (blk.okq[q]) *reinterpret_cast<uint4*>(dx + off) = pack8(o);
    }
  }
}

// ------------------------------------------------------------------------------------------
// global average pool   (reference models/basic_model.py:73-82)
// ------------------------------------------------------------------------------------------
__global__ void gap_fwd_kernel(const bf16* __restrict__ x, float* __restrict__ out, int B, int G,
                               int C) {
  const int groups = C / 8;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * groups) return;
  int cg = int(i % groups);
  int b = int(i / groups);
  float acc[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) acc[c] = 0.f;
  const bf16* p = x + (int64_t)b * G * C + cg * 8;
  for (int g = 0; g < G; ++g) {
    float f[8];
    unpack8(*reinterpret_cast<const uint4*>(p + (int64_t)g * C), f);
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] += f[c];
  }
  const float inv = 1.f / (float)G;
#pragma unroll
  for (int c = 0; c < 8; ++c) out[(int64_t)b * C + cg * 8 + c] = acc[c] * inv;
}

__global__ void gap_bwd_kernel(const float* __restrict__ dout, bf16* __restrict__ dx, int B, int G,
                               int C) {
  const int groups = C / 8;
  const int64_t total = (int64_t)B * G * groups;
  const float inv = 1.f / (float)G;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int cg = int(i % groups);
    int b = int(i / ((int64_t)G * groups));
    float f[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) f[c] = dout[(int64_t)b * C + cg * 8 + c] * inv;
    *reinterpret_cast<uint4*>(dx + i * 8) = pack8(f);
  }
}

static unsigned ew_grid(int64_t work_items, int threads, int cap = kNumSMs * 16) {
  int64_t blocks = ceil_div64(work_items, threads);
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (unsigned)blocks;
}

static bool chan_ok(int C) { return C >= 64 && C <= 512 && (C & (C - 1)) == 0; }

}  // namespace gdl

using namespace gdl;

extern "C" int gdl_layout_ncthw_to_nhwc8(const float* src, void* dst, int B, int C, int T, int H,
                                         int W, gdl_stream_t s) {
  GDL_REQUIRE(src && dst, "gdl_layout_ncthw_to_nhwc8: null pointer");
  GDL_REQUIRE(B > 0 && C > 0 && C <= 8 && T > 0 && H > 0 && W > 0, "gdl_layout_ncthw_to_nhwc8: bad shape");
  int64_t total = (int64_t)B * T * H * W;
  layout_kernel<<<ew_grid(total, 256), 256, 0, (cudaStream_t)s>>>(src, (bf16*)dst, B, C, T, H, W);
  GDL_CHECK_LAUNCH("layout_kernel");
  return GDL_OK;
}

extern "C" int64_t gdl_bn_partial_floats(int64_t P, int C) {
  (void)P;
  return (int64_t)kBnMaxBlocks * 2 * C;
}

extern "C" int gdl_bn_stats(const void* x, int64_t P, int C, float* partial, const float* gamma,
                            const float* beta, float eps, float momentum, float* running_mean,
                            float* running_var, float* mean, float* invstd, float* scale,
                            float* shift, gdl_stream_t s) {
  GDL_REQUIRE(chan_ok(C) && P > 0, "gdl_bn_stats: bad shape");
  GDL_REQUIRE(x && partial && gamma && beta && mean && invstd && scale && shift, "gdl_bn_stats: null pointer");
  int nblk = bn_blocks_cap(P, C, GDL_RESIDENT(bn_stats_kernel, kBnThreads));
  bn_stats_kernel<<<nblk, kBnThreads, 0, (cudaStream_t)s>>>((const bf16*)x, P, C, partial, g_sweep_rev);
  GDL_CHECK_LAUNCH("bn_stats_kernel");
  bn_stats_finalize_kernel<<<(C * 32 + 255) / 256, 256, 0, (cudaStream_t)s>>>(partial, nblk, P, C, gamma, beta, eps, momentum, running_mean, running_var, mean, invstd, scale, shift);
  GDL_CHECK_LAUNCH("bn_stats_finalize_kernel");
  return GDL_OK;
}

extern "C" int gdl_bn_stats_finalize(const float* partial, int rows, int64_t P, int C, const float* gamma,
                                     const float* beta, float eps, float momentum, float* running_mean,
                                     float* running_var, float* mean, float* invstd, float* scale, float* shift,
                                     gdl_stream_t s) {
  GDL_REQUIRE(chan_ok(C) && P > 0 && rows > 0, "gdl_bn_stats_finalize: bad shape");
  GDL_REQUIRE(partial && gamma && beta && mean && invstd && scale && shift, "gdl_bn_stats_finalize: null pointer");
  bn_stats_finalize_kernel<<<(C * 32 + 255) / 256, 256, 0, (cudaStream_t)s>>>(partial, rows, P, C, gamma, beta, eps, momentum, running_mean, running_var, mean, invstd, scale, shift);
  GDL_CHECK_LAUNCH("bn_stats_finalize_kernel");
  return GDL_OK;
}

extern "C" int gdl_bn_eval_affine(const float* gamma, const float* beta, const float* running_mean,
                                  const float* running_var, float eps, float* scale, float* shift, int C,
                                  gdl_stream_t s) {
  GDL_REQUIRE(gamma && beta && running_mean && running_var && scale && shift && C > 0, "gdl_bn_eval_affine: bad arguments");
  bn_eval_affine_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)s>>>(gamma, beta, running_mean, running_var, eps,
                                                                     scale, shift, C);
  GDL_CHECK_LAUNCH("bn_eval_affine_kernel");
  return GDL_OK;
}

extern "C" int gdl_bn_apply(const void* x, const void* res, void* y, int64_t P, int C,
                            const float* scale, const float* shift, int relu, gdl_stream_t s) {
  GDL_REQUIRE(chan_ok(C) && P > 0, "gdl_bn_apply: bad shape");
  GDL_REQUIRE(x && y && scale && shift, "gdl_bn_apply: null pointer");
  int64_t nvec = P * C / 8;
  bn_apply_kernel<<<ew_grid(nvec, 256, GDL_RESIDENT(bn_apply_kernel, 256)), 256, 0, (cudaStream_t)s>>>((const bf16*)x, (const bf16*)res,
                                                                  (bf16*)y, nvec, C, scale, shift, relu, g_sweep_rev);
  GDL_CHECK_LAUNCH("bn_apply_kernel");
  return GDL_OK;
}

extern "C" int gdl_bn_bwd(const void* dy, const void* y, const void* x, void* dz, void* dx,
                          int64_t P, int C, const float* gamma, const float* mean,
                          const float* invstd, float* partial, float* dgamma, float* dbeta,
                          int relu, gdl_stream_t s) {
  GDL_REQUIRE(chan_ok(C) && P > 0, "gdl_bn_bwd: bad shape");
  GDL_REQUIRE(dy && x && dx && gamma && mean && invstd && partial && dgamma && dbeta, "gdl_bn_bwd: null pointer");
  GDL_REQUIRE(!relu || (y && dz), "gdl_bn_bwd: relu needs y and dz");
  int nblk = bn_blocks_cap(P, C, GDL_RESIDENT(bn_bwd_reduce_kernel, kBnThreads));
  bn_bwd_reduce_kernel<<<nblk, kBnThreads, 0, (cudaStream_t)s>>>((const bf16*)dy, (const bf16*)y, (const bf16*)x, (bf16*)dz, P, C, partial, relu, g_sweep_rev);
  GDL_CHECK_LAUNCH("bn_bwd_reduce_kernel");
  bn_bwd_finalize_raw_kernel<<<(C * 32 + 255) / 256, 256, 0, (cudaStream_t)s>>>(partial, nblk, C, mean, invstd, dgamma,
                                                                               dbeta);
  GDL_CHECK_LAUNCH("bn_bwd_finalize_raw_kernel");
  int64_t nvec = P * C / 8;
  const bf16* dzp = relu ? (const bf16*)dz : (const bf16*)dy;
  bn_bwd_apply_kernel<<<ew_grid(nvec, 256, GDL_RESIDENT(bn_bwd_apply_kernel, 256)), 256, 0, (cudaStream_t)s>>>(dzp, (const bf16*)x, (bf16*)dx, nvec, C, 1.f / (float)P, gamma, mean, invstd, dgamma, dbeta, !g_sweep_rev);
  GDL_CHECK_LAUNCH("bn_bwd_apply_kernel");
  return GDL_OK;
}

extern "C" int gdl_bn_bwd_nores(const void* dy, const void* x, void* dx, int64_t P, int C, const float* gamma,
                                const float* mean, const float* invstd, const float* scale, const float* shift,
                                float* partial, float* dgamma, float* dbeta, gdl_stream_t s) {
  GDL_REQUIRE(chan_ok(C) && P > 0, "gdl_bn_bwd_nores: bad shape");
  GDL_REQUIRE(dy && x && dx && gamma && mean && invstd && scale && shift && partial && dgamma && dbeta,
              "gdl_bn_bwd_nores: null pointer");
  int nblk = bn_blocks_cap(P, C, GDL_RESIDENT(bn_bwd_nores_reduce_kernel, kBnThreads));
  bn_bwd_nores_reduce_kernel<<<nblk, kBnThreads, 0, (cudaStream_t)s>>>((const bf16*)dy, (const bf16*)x, P, C, scale,
                                                                      shift, partial, g_sweep_rev);
  GDL_CHECK_LAUNCH("bn_bwd_nores_reduce_kernel");
  bn_bwd_finalize_raw_kernel<<<(C * 32 + 255) / 256, 256, 0, (cudaStream_t)s>>>(partial, nblk, C, mean, invstd, dgamma,
                                                                               dbeta);
  GDL_CHECK_LAUNCH("bn_bwd_finalize_raw_kernel");
  int64_t nvec = P * C / 8;
  bn_bwd_nores_apply_kernel<<<ew_grid(nvec, 256, GDL_RESIDENT(bn_bwd_nores_apply_kernel, 256)), 256, 0, (cudaStream_t)s>>>((const bf16*)dy, (const bf16*)x, (bf16*)dx, nvec, C, 1.f / (float)P, gamma, mean, invstd, scale, shift, dgamma,
      dbeta, !g_sweep_rev);
  GDL_CHECK_LAUNCH("bn_bwd_nores_apply_kernel");
  return GDL_OK;
}

extern "C" int gdl_bn_relu_maxpool_fwd(const void* x, const float* scale, const float* shift, void* y,
                                       uint8_t* argmax, void* xmax, int N, int H, int W, int C, int Ho, int Wo,
                                       gdl_stream_t s) {
  GDL_REQUIRE(x && scale && shift && y && argmax, "gdl_bn_relu_maxpool_fwd: null pointer");
  GDL_REQUIRE(chan_ok(C) && Ho == (H - 1) / 2 + 1 && Wo == (W - 1) / 2 + 1, "gdl_bn_relu_maxpool_fwd: bad shape");
  if ((int64_t)N * H * W * C < ((int64_t)1 << 31)) {  // 32-bit indexing inside the kernel
    const int nseg = (Ho + kTailSeg - 1) / kTailSeg;
    int64_t total3 = (int64_t)N * nseg * Wo * (C / 8);
    bn_relu_maxpool_fwd3_kernel<<<ew_grid(total3, 256, GDL_RESIDENT(bn_relu_maxpool_fwd3_kernel, 256)), 256, 0,
                                  (cudaStream_t)s>>>((const bf16*)x, scale, shift, (bf16*)y, argmax, (bf16*)xmax, N, H,
                                                     W, C, Ho, Wo, nseg, kTailSeg, g_sweep_rev);
    GDL_CHECK_LAUNCH("bn_relu_maxpool_fwd3_kernel");
    return GDL_OK;
  }
  int64_t total = (int64_t)N * Ho * Wo * (C / 8);
  bn_relu_maxpool_fwd_kernel<<<ew_grid(total, 256, GDL_RESIDENT(bn_relu_maxpool_fwd_kernel, 256)), 256, 0, (cudaStream_t)s>>>(
      (const bf16*)x, scale, shift, (bf16*)y, argmax, (bf16*)xmax, N, H, W, C, Ho, Wo);
  GDL_CHECK_LAUNCH("bn_relu_maxpool_fwd_kernel");
  return GDL_OK;
}

extern "C" int gdl_bn_relu_maxpool_bwd(const void* gpool, const uint8_t* argmax, const void* xmax, const void* x,
                                       void* dx, int N, int H, int W, int C, int Ho, int Wo, const float* gamma,
                                       const float* mean,
                                       const float* invstd, const float* scale, const float* shift, float* partial,
                                       float* dgamma, float* dbeta, gdl_stream_t s) {
  GDL_REQUIRE(gpool && argmax && x && dx && gamma && mean && invstd && scale && shift && partial && dgamma && dbeta,
              "gdl_bn_relu_maxpool_bwd: null pointer");
  GDL_REQUIRE(chan_ok(C) && Ho == (H - 1) / 2 + 1 && Wo == (W - 1) / 2 + 1, "gdl_bn_relu_maxpool_bwd: bad shape");
  const int64_t P = (int64_t)N * H * W;
  int nblk;
  if (xmax != nullptr) {
    // sums of dz and dz*xhat over the POOLED grid: each window contributes its gradient at its arg-max pixel,
    // whose conv output the forward saved — the no-residual BN reduce kernel on (gpool, xmax)
    const int64_t Pp = (int64_t)N * Ho * Wo;
    nblk = bn_blocks_cap(Pp, C, GDL_RESIDENT(bn_bwd_nores_reduce_kernel, kBnThreads));
    bn_bwd_nores_reduce_kernel<<<nblk, kBnThreads, 0, (cudaStream_t)s>>>((const bf16*)gpool, (const bf16*)xmax, Pp, C,
                                                                        scale, shift, partial, g_sweep_rev);
    GDL_CHECK_LAUNCH("bn_bwd_nores_reduce_kernel(stem tail)");
    bn_bwd_finalize_raw_kernel<<<(C * 32 + 255) / 256, 256, 0, (cudaStream_t)s>>>(partial, nblk, C, mean, invstd, dgamma,
                                                                                 dbeta);
  } else {
    nblk = bn_blocks_cap((int64_t)N * Ho * Wo * 4, C, GDL_RESIDENT(bn_relu_maxpool_bwd_reduce_kernel, kBnThreads));
    bn_relu_maxpool_bwd_reduce_kernel<<<nblk, kBnThreads, 0, (cudaStream_t)s>>>(
        (const bf16*)gpool, argmax, (const bf16*)x, N, H, W, C, Ho, Wo, mean, invstd, scale, shift, partial);
    GDL_CHECK_LAUNCH("bn_relu_maxpool_bwd_reduce_kernel");
    bn_bwd_finalize_kernel<<<(C * 32 + 255) / 256, 256, 0, (cudaStream_t)s>>>(partial, nblk, C, dgamma, dbeta);
  }
  GDL_CHECK_LAUNCH("bn_bwd_finalize_kernel");
  int64_t total = (int64_t)N * Ho * Wo * (C / 8);
  GDL_REQUIRE(total < ((int64_t)1 << 30), "gdl_bn_relu_maxpool_bwd: too many pooled pixels for 32-bit block indices");
  bn_relu_maxpool_bwd_apply_kernel<<<ew_grid(total, 256, GDL_RESIDENT(bn_relu_maxpool_bwd_apply_kernel, 256)), 256, 0, (cudaStream_t)s>>>((const bf16*)gpool, argmax, (const bf16*)x, (bf16*)dx, N, H, W, C, Ho, Wo, 1.f / (float)P, gamma, mean, invstd,
      scale, shift, dgamma, dbeta);
  GDL_CHECK_LAUNCH("bn_relu_maxpool_bwd_apply_kernel");
  return GDL_OK;
}

extern "C" int gdl_maxpool_fwd(const void* x, void* y, uint8_t* argmax, int N, int H, int W, int C,
                               int Ho, int Wo, gdl_stream_t s) {
  GDL_REQUIRE(x && y && argmax, "gdl_maxpool_fwd: null pointer");
  GDL_REQUIRE(C % 8 == 0 && Ho == (H - 1) / 2 + 1 && Wo == (W - 1) / 2 + 1, "gdl_maxpool_fwd: bad shape");
  int64_t total = (int64_t)N * Ho * Wo * (C / 8);
  maxpool_fwd_kernel<<<ew_grid(total, 256), 256, 0, (cudaStream_t)s>>>((const bf16*)x, (bf16*)y, argmax,
                                                                      N, H, W, C, Ho, Wo);
  GDL_CHECK_LAUNCH("maxpool_fwd_kernel");
  return GDL_OK;
}

extern "C" int gdl_maxpool_bwd(const void* dy, const uint8_t* argmax, void* dx, int N, int H, int W,
                               int C, int Ho, int Wo, gdl_stream_t s) {
  GDL_REQUIRE(dy && dx && argmax, "gdl_maxpool_bwd: null pointer");
  GDL_REQUIRE(C % 8 == 0 && Ho == (H - 1) / 2 + 1 && Wo == (W - 1) / 2 + 1, "gdl_maxpool_bwd: bad shape");
  int64_t total = (int64_t)N * H * W * (C / 8);
  maxpool_bwd_kernel<<<ew_grid(total, 256), 256, 0, (cudaStream_t)s>>>((const bf16*)dy, argmax, (bf16*)dx,
                                                                      N, H, W, C, Ho, Wo);
  GDL_CHECK_LAUNCH("maxpool_bwd_kernel");
  return GDL_OK;
}

extern "C" int gdl_gap_fwd(const void* x, float* out, int B, int G, int C, gdl_stream_t s) {
  GDL_REQUIRE(x && out && B > 0 && G > 0 && C % 8 == 0, "gdl_gap_fwd: bad arguments");
  int64_t total = (int64_t)B * (C / 8);
  gap_fwd_kernel<<<(unsigned)ceil_div64(total, 128), 128, 0, (cudaStream_t)s>>>((const bf16*)x, out, B, G, C);
  GDL_CHECK_LAUNCH("gap_fwd_kernel");
  return GDL_OK;
}

extern "C" int gdl_gap_bwd(const float* dout, void* dx, int B, int G, int C, gdl_stream_t s) {
  GDL_REQUIRE(dout && dx && B > 0 && G > 0 && C % 8 == 0, "gdl_gap_bwd: bad arguments");
  int64_t total = (int64_t)B * G * (C / 8);
  gap_bwd_kernel<<<ew_grid(total, 256), 256, 0, (cudaStream_t)s>>>(dout, (bf16*)dx, B, G, C);
  GDL_CHECK_LAUNCH("gap_bwd_kernel");
  return GDL_OK;
}

extern "C" int gdl_set_sweep(int reverse) {
  const int old = gdl::g_sweep_rev;
  gdl::g_sweep_rev = reverse != 0;
  return old;
}
