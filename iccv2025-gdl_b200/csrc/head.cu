// head.cu — fusion heads of the DGL step.
//
//  * gdl_dgl_head_linear : the fused ConcatFusion_DGL / SumFusion_DGL head (reference
//    models/fusion_modules.py:51-59, :22-30).  With W = [Wx | Wy] the three logit sets are
//    x_out = Wx a + bx, y_out = Wy v + by, out = Wx a + Wy v + bo, so ONE pass over the two
//    half-products yields all three; the kernel then does the three softmax-cross-entropies
//    (main_dgl.py:102-104) and applies the DGL gradient routing in registers
//    (main_dgl.py:108-122): da <- alpha*dLa only, dv <- alpha*dLv only (the multimodal head saw
//    detached features), dW/db <- dLf only (the unimodal gradient of the head is wiped).
//  * gdl_linear_fwd/bwd, gdl_softmax_ce, gdl_gated_fwd/bwd : generic pieces used by the
//    GatedFusion_DGL / FiLM_DGL heads and by the autograd-compatible module path.
// Everything is fp32 and deterministic (fixed-order loops over the batch).
#include "common.cuh"

namespace gdl {

// ------------------------------------------------------------------------------------------
// generic linear
// ------------------------------------------------------------------------------------------
__global__ void linear_fwd_kernel(const float* __restrict__ x, const float* __restrict__ W, int ldw,
                                  const float* __restrict__ b, float* __restrict__ y, int B, int In,
                                  int Out) {
  int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;  // one warp per (b, o)
  int lane = threadIdx.x & 31;
  if (gw >= (int64_t)B * Out) return;
  int bi = int(gw / Out), o = int(gw - (int64_t)bi * Out);
  const float* xr = x + (int64_t)bi * In;
  const float* wr = W + (int64_t)o * ldw;
  float acc = 0.f;
  for (int i = lane; i < In; i += 32) acc = fmaf(xr[i], wr[i], acc);
  acc = warp_sum(acc);
  if (lane == 0) y[gw] = acc + (b ? b[o] : 0.f);
}

__global__ void linear_bwd_dx_kernel(const float* __restrict__ dy, const float* __restrict__ W, int ldw,
                                     float* __restrict__ dx, int B, int In, int Out) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // (b, i), i fastest
  if (idx >= (int64_t)B * In) return;
  int bi = int(idx / In), i = int(idx - (int64_t)bi * In);
  const float* g = dy + (int64_t)bi * Out;
  float acc = 0.f;
  for (int o = 0; o < Out; ++o) acc = fmaf(g[o], W[(int64_t)o * ldw + i], acc);
  dx[idx] = acc;
}

__global__ void linear_bwd_dw_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                     float* __restrict__ dW, int lddw, float* __restrict__ db, int B,
                                     int In, int Out, int accumulate) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // (o, i), i fastest; i == In -> bias
  int64_t total = (int64_t)Out * (In + 1);
  if (idx >= total) return;
  int o = int(idx / (In + 1)), i = int(idx - (int64_t)o * (In + 1));
  float acc = 0.f;
  if (i < In) {
    for (int bi = 0; bi < B; ++bi) acc = fmaf(dy[(int64_t)bi * Out + o], x[(int64_t)bi * In + i], acc);
    float* dst = dW + (int64_t)o * lddw + i;
    *dst = accumulate ? *dst + acc : acc;
  } else if (db != nullptr) {
    for (int bi = 0; bi < B; ++bi) acc += dy[(int64_t)bi * Out + o];
    db[o] = accumulate ? db[o] + acc : acc;
  }
}

// ------------------------------------------------------------------------------------------
// softmax cross-entropy of one row held in shared memory, computed by one warp.
// Returns the loss (valid in all lanes); writes grad[j] = gscale*(softmax_j - onehot_j).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_softmax_ce(const float* z, int n, int label, float gscale,
                                                 float* grad) {
  const int lane = threadIdx.x & 31;
  float m = -INFINITY;
  for (int j = lane; j < n; j += 32) m = fmaxf(m, z[j]);
  m = warp_max(m);
  float sum = 0.f;
  for (int j = lane; j < n; j += 32) sum += expf(z[j] - m);
  sum = warp_sum(sum);
  const float lse = m + logf(sum);
  const float inv = 1.f / sum;
  if (grad != nullptr) {
    for (int j = lane; j < n; j += 32) {
      float pj = expf(z[j] - m) * inv;
      grad[j] = gscale * (pj - (j == label ? 1.f : 0.f));
    }
  }
  return lse - z[label];
}

// ------------------------------------------------------------------------------------------
// fused concat / sum head, phase A: one CTA per sample
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

constexpr int kHeadThreads = 256;
constexpr int kHeadMaxN = 512;
constexpr int kHeadMaxD = 1024;

__global__ void __launch_bounds__(kHeadThreads) dgl_head_sample_kernel(
    int kind, const float* __restrict__ a, const float* __restrict__ v, const float* __restrict__ Wx,
    const float* __restrict__ Wy, int ldw, const float* __restrict__ bx, const float* __restrict__ by,
    const int64_t* __restrict__ labels, float alpha, float inv_batch, float* __restrict__ logits,
    float* __restrict__ da, float* __restrict__ dv, float* __restrict__ g_out_all,
    float* __restrict__ loss_rows, int B, int D, int n) {
  __shared__ float s_a[kHeadMaxD], s_v[kHeadMaxD];
  __shared__ float s_z[3][kHeadMaxN];  // out, x_out, y_out
  __shared__ float s_g[3][kHeadMaxN];
  const int b = blockIdx.x;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < D; i += kHeadThreads) {
    s_a[i] = a[(int64_t)b * D + i];
    s_v[i] = v[(int64_t)b * D + i];
  }
  __syncthreads();
  for (int j = warp; j < n; j += kHeadThreads / 32) {
    const float* wx = Wx + (int64_t)j * ldw;
    const float* wy = Wy + (int64_t)j * ldw;
    float pa = 0.f, pv = 0.f;
    for (int i = lane; i < D; i += 32) {
      pa = fmaf(wx[i], s_a[i], pa);
      pv = fmaf(wy[i], s_v[i], pv);
    }
    pa = warp_sum(pa);
    pv = warp_sum(pv);
    if (lane == 0) {
      float bxj = bx[j];
      float byj = kind == 0 ? bxj : by[j];
      float boj = kind == 0 ? bxj : bxj + byj;
      // same association order as the reference: (Wx a + Wy v) + b for concat,
      // (Wx a + bx) + (Wy v + by) for sum
      s_z[0][j] = kind == 0 ? (pa + pv) + boj : (pa + bxj) + (pv + byj);
      s_z[1][j] = pa + bxj;
      s_z[2][j] = pv + byj;
    }
  }
  __syncthreads();
  const int label = int(labels[b]);
  if (warp < 3) {
    const float gs = warp == 0 ? inv_batch : alpha * inv_batch;
    float loss = warp_softmax_ce(s_z[warp], n, label, gs, s_g[warp]);
    if (lane == 0) loss_rows[(int64_t)b * 3 + warp] = loss;
  }
  __syncthreads();
  for (int j = tid; j < n; j += kHeadThreads) {
    logits[((int64_t)0 * B + b) * n + j] = s_z[0][j];
    logits[((int64_t)1 * B + b) * n + j] = s_z[1][j];
    logits[((int64_t)2 * B + b) * n + j] = s_z[2][j];
    g_out_all[(int64_t)b * n + j] = s_g[0][j];
  }
  // encoder-facing gradients: ONLY the unimodal losses reach a and v
  for (int i = tid; i < D; i += kHeadThreads) {
    float ga = 0.f, gv = 0.f;
    for (int j = 0; j < n; ++j) {
      ga = fmaf(s_g[1][j], Wx[(int64_t)j * ldw + i], ga);
      gv = fmaf(s_g[2][j], Wy[(int64_t)j * ldw + i], gv);
    }
    da[(int64_t)b * D + i] = ga;
    dv[(int64_t)b * D + i] = gv;
  }
}

// phase B: head-parameter gradients from Lf only + loss reduction (fixed order over the batch)
__global__ void dgl_head_param_kernel(int kind, const float* __restrict__ a,
                                      const float* __restrict__ v, const float* __restrict__ g_out,
                                      const float* __restrict__ loss_rows, float inv_batch,
                                      float* __restrict__ dWx, float* __restrict__ dWy, int lddw,
                                      float* __restrict__ dbx, float* __restrict__ dby,
                                      float* __restrict__ losses, int B, int D, int n) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nW = (int64_t)n * 2 * D;
  if (idx < nW) {
    int j = int(idx / (2 * D)), i = int(idx - (int64_t)j * 2 * D);
    const float* f = i < D ? a : v;
    int ii = i < D ? i : i - D;
    float acc = 0.f;
    for (int b = 0; b < B; ++b) acc = fmaf(g_out[(int64_t)b * n + j], f[(int64_t)b * D + ii], acc);
    if (i < D)
      dWx[(int64_t)j * lddw + ii] = acc;
    else
      dWy[(int64_t)j * lddw + ii] = acc;
  } else if (idx < nW + n) {
    int j = int(idx - nW);
    float acc = 0.f;
    for (int b = 0; b < B; ++b) acc += g_out[(int64_t)b * n + j];
    dbx[j] = acc;
    if (kind == 1) dby[j] = acc;
  } else if (idx < nW + n + 3) {
    int h = int(idx - nW - n);
    float acc = 0.f;
    for (int b = 0; b < B; ++b) acc += loss_rows[(int64_t)b * 3 + h];
    losses[h] = acc * inv_batch;
  }
}

// ------------------------------------------------------------------------------------------
// stand-alone softmax-CE (gated / film heads)
// ------------------------------------------------------------------------------------------
__global__ void softmax_ce_rows_kernel(const float* __restrict__ logits,
                                       const int64_t* __restrict__ labels, float grad_scale,
                                       float* __restrict__ dlogits, float* __restrict__ loss_rows,
                                       int B, int n) {
  extern __shared__ float s_row[];
  int warps = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int b = blockIdx.x * warps + warp;
  if (b >= B) return;
  float* z = s_row + (size_t)warp * n;
  for (int j = lane; j < n; j += 32) z[j] = logits[(int64_t)b * n + j];
  __syncwarp();
  float loss = warp_softmax_ce(z, n, int(labels[b]), grad_scale, dlogits ? dlogits + (int64_t)b * n : nullptr);
  if (lane == 0) loss_rows[b] = loss;
}
__global__ void loss_rows_sum_kernel(const float* __restrict__ loss_rows, float scale,
                                     float* __restrict__ out, int B) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    float acc = 0.f;
    for (int b = 0; b < B; ++b) acc += loss_rows[b];
    out[0] = acc * scale;
  }
}

// ------------------------------------------------------------------------------------------
// gated head elementwise pieces
// ------------------------------------------------------------------------------------------
__global__ void gated_fwd_kernel(const float* __restrict__ hx, const float* __restrict__ hy,
                                 float* __restrict__ m_out, float* __restrict__ m_x,
                                 float* __restrict__ m_y, int64_t numel) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= numel) return;
  float x = hx[i], y = hy[i];
  float sx = sigmoidf_(x), sy = sigmoidf_(y);
  m_out[i] = sx * y;  // x_gate=True: gate from (detached) hx applied to (detached) hy
  m_x[i] = sx * x;
  m_y[i] = sy * y;
}
__global__ void gated_bwd_kernel(const float* __restrict__ hx, const float* __restrict__ hy,
                                 const float* __restrict__ dm_x, const float* __restrict__ dm_y,
                                 float* __restrict__ dhx, float* __restrict__ dhy, int64_t numel) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= numel) return;
  float x = hx[i], y = hy[i];
  float sx = sigmoidf_(x), sy = sigmoidf_(y);
  dhx[i] = dm_x[i] * (sx + x * sx * (1.f - sx));
  dhy[i] = dm_y[i] * (sy + y * sy * (1.f - sy));
}


// ------------------------------------------------------------------------------------------
// fused GatedFusion_DGL head (reference models/fusion_modules.py:230-250 + main_dgl.py:102-122), one CTA per sample:
//   hx = fc_x(a), hy = fc_y(v);  out = fc_out(sig(hx.detach()) * hy.detach()),
//   out_x = fc_out(sig(hx) * hx), out_y = fc_out(sig(hy) * hy);  three softmax-CE;
//   routing in registers: a <- alpha*dLa through fc_out, the gate and fc_x;  v <- alpha*dLv likewise;
//   fc_out <- dLf only (phase B: dgl_gated_param_kernel);  fc_x / fc_y receive NO gradient (their unimodal
//   gradient is wiped, and Lf sees them detached — SURVEY.md §8a quirk 2).
// Replaces the chain of 15 generic launches (2 linear, gate, 3 x (linear + CE), 5 linear_bwd, gate_bwd).
// ------------------------------------------------------------------------------------------
constexpr int kGatedD = 512;

__global__ void __launch_bounds__(kHeadThreads) dgl_gated_sample_kernel(
    const float* __restrict__ a, const float* __restrict__ v, const float* __restrict__ Wx, const float* __restrict__ bx,
    const float* __restrict__ Wy, const float* __restrict__ by, const float* __restrict__ Wo, const float* __restrict__ bo,
    const int64_t* __restrict__ labels, float alpha, float inv_batch, float* __restrict__ logits, float* __restrict__ da,
    float* __restrict__ dv, float* __restrict__ m_out_all, float* __restrict__ g_out_all, float* __restrict__ loss_rows,
    int B, int n) {
  constexpr int D = kGatedD;
  __shared__ float s_a[D], s_v[D], s_hx[D], s_hy[D];
  __shared__ float s_m[3][D];            // m_out, m_x, m_y; later reused for dhx (row 1) and dhy (row 2)
  __shared__ float s_z[3][kHeadMaxN];
  __shared__ float s_g[3][kHeadMaxN];
  const int b = blockIdx.x;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < D; i += kHeadThreads) {
    s_a[i] = a[(int64_t)b * D + i];
    s_v[i] = v[(int64_t)b * D + i];
  }
  __syncthreads();
  for (int j = warp; j < D; j += kHeadThreads / 32) {  // hx, hy: one warp per output row
    const float* wx = Wx + (int64_t)j * D;
    const float* wy = Wy + (int64_t)j * D;
    float px = 0.f, py = 0.f;
    for (int i = lane; i < D; i += 32) {
      px = fmaf(wx[i], s_a[i], px);
      py = fmaf(wy[i], s_v[i], py);
    }
    px = warp_sum(px);
    py = warp_sum(py);
    if (lane == 0) {
      s_hx[j] = px + bx[j];
      s_hy[j] = py + by[j];
    }
  }
  __syncthreads();
  for (int i = tid; i < D; i += kHeadThreads) {
    const float x = s_hx[i], y = s_hy[i];
    const float sx = sigmoidf_(x), sy = sigmoidf_(y);
    s_m[0][i] = sx * y;
    s_m[1][i] = sx * x;
    s_m[2][i] = sy * y;
    m_out_all[(int64_t)b * D + i] = sx * y;
  }
  __syncthreads();
  for (int j = warp; j < n; j += kHeadThreads / 32) {  // three logit sets share every row of fc_out
    const float* wo = Wo + (int64_t)j * D;
    float p0 = 0.f, p1 = 0.f, p2 = 0.f;
    for (int i = lane; i < D; i += 32) {
      const float w = wo[i];
      p0 = fmaf(w, s_m[0][i], p0);
      p1 = fmaf(w, s_m[1][i], p1);
      p2 = fmaf(w, s_m[2][i], p2);
    }
    p0 = warp_sum(p0);
    p1 = warp_sum(p1);
    p2 = warp_sum(p2);
    if (lane == 0) {
      s_z[0][j] = p0 + bo[j];
      s_z[1][j] = p1 + bo[j];
      s_z[2][j] = p2 + bo[j];
    }
  }
  __syncthreads();
  const int label = int(labels[b]);
  if (warp < 3) {
    const float gs = warp == 0 ? inv_batch : alpha * inv_batch;
    float loss = warp_softmax_ce(s_z[warp], n, label, gs, s_g[warp]);
    if (lane == 0) loss_rows[(int64_t)b * 3 + warp] = loss;
  }
  __syncthreads();
  for (int j = tid; j < n; j += kHeadThreads) {
    logits[((int64_t)0 * B + b) * n + j] = s_z[0][j];
    logits[((int64_t)1 * B + b) * n + j] = s_z[1][j];
    logits[((int64_t)2 * B + b) * n + j] = s_z[2][j];
    g_out_all[(int64_t)b * n + j] = s_g[0][j];
  }
  // unimodal gradients back through fc_out and the gates: dh = (Wo^T g) * d(sig(h) h)/dh
  for (int i = tid; i < D; i += kHeadThreads) {
    float gx = 0.f, gy = 0.f;
    for (int j = 0; j < n; ++j) {
      const float w = Wo[(int64_t)j * D + i];
      gx = fmaf(s_g[1][j], w, gx);
      gy = fmaf(s_g[2][j], w, gy);
    }
    const float x = s_hx[i], y = s_hy[i];
    const float sx = sigmoidf_(x), sy = sigmoidf_(y);
    s_m[1][i] = gx * (sx + x * sx * (1.f - sx));
    s_m[2][i] = gy * (sy + y * sy * (1.f - sy));
  }
  __syncthreads();
  // ... and through fc_x / fc_y to the pooled features (column access: consecutive threads, consecutive i)
  for (int i = tid; i < D; i += kHeadThreads) {
    float ga = 0.f, gv = 0.f;
    for (int k = 0; k < D; ++k) {
      ga = fmaf(s_m[1][k], Wx[(int64_t)k * D + i], ga);
      gv = fmaf(s_m[2][k], Wy[(int64_t)k * D + i], gv);
    }
    da[(int64_t)b * D + i] = ga;
    dv[(int64_t)b * D + i] = gv;
  }
}

// phase B: dWo = sum_b g_out[b] (x) m_out[b], dbo = sum_b g_out[b]  (Lf only), losses; fixed order over the batch
__global__ void dgl_gated_param_kernel(const float* __restrict__ m_out, const float* __restrict__ g_out,
                                       const float* __restrict__ loss_rows, float inv_batch, float* __restrict__ dWo,
                                       float* __restrict__ dbo, float* __restrict__ losses, int B, int n) {
  constexpr int D = kGatedD;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nW = (int64_t)n * D;
  if (idx < nW) {
    const int j = int(idx / D), i = int(idx - (int64_t)j * D);
    float acc = 0.f;
    for (int b = 0; b < B; ++b) acc = fmaf(g_out[(int64_t)b * n + j], m_out[(int64_t)b * D + i], acc);
    dWo[idx] = acc;
  } else if (idx < nW + n) {
    const int j = int(idx - nW);
    float acc = 0.f;
    for (int b = 0; b < B; ++b) acc += g_out[(int64_t)b * n + j];
    dbo[j] = acc;
  } else if (idx < nW + n + 3) {
    const int h = int(idx - nW - n);
    float acc = 0.f;
    for (int b = 0; b < B; ++b) acc += loss_rows[(int64_t)b * 3 + h];
    losses[h] = acc * inv_batch;
  }
}

}  // namespace gdl

using namespace gdl;

extern "C" int gdl_linear_fwd(const float* x, const float* W, int ldw, const float* b, float* y, int B,
                              int In, int Out, gdl_stream_t s) {
  GDL_REQUIRE(x && W && y && B > 0 && In > 0 && Out > 0 && ldw >= In, "gdl_linear_fwd: bad arguments");
  int64_t threads = (int64_t)B * Out * 32;
  linear_fwd_kernel<<<(unsigned)ceil_div64(threads, 256), 256, 0, (cudaStream_t)s>>>(x, W, ldw, b, y, B, In, Out);
  GDL_CHECK_LAUNCH("linear_fwd_kernel");
  return GDL_OK;
}

extern "C" int gdl_linear_bwd(const float* dy, const float* x, const float* W, int ldw, float* dx,
                              float* dW, int lddw, float* db, int B, int In, int Out, int accumulate,
                              gdl_stream_t s) {
  GDL_REQUIRE(dy && B > 0 && In > 0 && Out > 0, "gdl_linear_bwd: bad arguments");
  if (dx != nullptr) {
    GDL_REQUIRE(W != nullptr, "gdl_linear_bwd: dx needs W");
    linear_bwd_dx_kernel<<<(unsigned)ceil_div64((int64_t)B * In, 256), 256, 0, (cudaStream_t)s>>>(dy, W, ldw, dx, B, In, Out);
    GDL_CHECK_LAUNCH("linear_bwd_dx_kernel");
  }
  if (dW != nullptr) {
    GDL_REQUIRE(x != nullptr, "gdl_linear_bwd: dW needs x");
    linear_bwd_dw_kernel<<<(unsigned)ceil_div64((int64_t)Out * (In + 1), 256), 256, 0, (cudaStream_t)s>>>(
        dy, x, dW, lddw, db, B, In, Out, accumulate);
    GDL_CHECK_LAUNCH("linear_bwd_dw_kernel");
  }
  return GDL_OK;
}

extern "C" int64_t gdl_head_scratch_floats(int B, int n) { return (int64_t)B * n + (int64_t)B * 3; }

extern "C" int gdl_dgl_head_linear(int kind, const float* a, const float* v, const float* Wx,
                                   const float* Wy, int ldw, const float* bx, const float* by,
                                   const int64_t* labels, float alpha, float inv_batch,
                                   float* logits, float* losses, float* da, float* dv, float* dWx,
                                   float* dWy, int lddw, float* dbx, float* dby, float* scratch,
                                   int B, int D, int n, gdl_stream_t s) {
  GDL_REQUIRE(kind == 0 || kind == 1, "gdl_dgl_head_linear: kind must be 0 (concat) or 1 (sum)");
  GDL_REQUIRE(a && v && Wx && Wy && bx && labels && logits && losses && da && dv && dWx && dWy && dbx && scratch,
              "gdl_dgl_head_linear: null pointer");
  GDL_REQUIRE(kind == 0 || (by && dby), "gdl_dgl_head_linear: sum head needs by/dby");
  GDL_REQUIRE(B > 0 && D > 0 && D <= kHeadMaxD && n > 0 && n <= kHeadMaxN, "gdl_dgl_head_linear: bad shape");
  float* g_out = scratch;
  float* loss_rows = scratch + (int64_t)B * n;
  dgl_head_sample_kernel<<<B, kHeadThreads, 0, (cudaStream_t)s>>>(kind, a, v, Wx, Wy, ldw, bx, by, labels,
                                                                  alpha, inv_batch, logits, da, dv, g_out,
                                                                  loss_rows, B, D, n);
  GDL_CHECK_LAUNCH("dgl_head_sample_kernel");
  int64_t total = (int64_t)n * 2 * D + n + 3;
  dgl_head_param_kernel<<<(unsigned)ceil_div64(total, 256), 256, 0, (cudaStream_t)s>>>(kind, a, v, g_out, loss_rows, inv_batch, dWx, dWy, lddw, dbx, dby, losses, B, D, n);
  GDL_CHECK_LAUNCH("dgl_head_param_kernel");
  return GDL_OK;
}

extern "C" int gdl_softmax_ce(const float* logits, const int64_t* labels, float loss_scale,
                              float grad_scale, float* loss_out, float* dlogits, float* scratch,
                              int B, int n, gdl_stream_t s) {
  GDL_REQUIRE(logits && labels && loss_out && scratch && B > 0 && n > 0 && n <= 4096, "gdl_softmax_ce: bad arguments");
  const int warps = 4;
  softmax_ce_rows_kernel<<<(B + warps - 1) / warps, warps * 32, (size_t)warps * n * sizeof(float), (cudaStream_t)s>>>(
      logits, labels, grad_scale, dlogits, scratch, B, n);
  GDL_CHECK_LAUNCH("softmax_ce_rows_kernel");
  loss_rows_sum_kernel<<<1, 32, 0, (cudaStream_t)s>>>(scratch, loss_scale, loss_out, B);
  GDL_CHECK_LAUNCH("loss_rows_sum_kernel");
  return GDL_OK;
}

extern "C" int gdl_gated_fwd(const float* hx, const float* hy, float* m_out, float* m_x, float* m_y,
                             int64_t numel, gdl_stream_t s) {
  GDL_REQUIRE(hx && hy && m_out && m_x && m_y && numel > 0, "gdl_gated_fwd: bad arguments");
  gated_fwd_kernel<<<(unsigned)ceil_div64(numel, 256), 256, 0, (cudaStream_t)s>>>(hx, hy, m_out, m_x, m_y, numel);
  GDL_CHECK_LAUNCH("gated_fwd_kernel");
  return GDL_OK;
}

extern "C" int gdl_gated_bwd(const float* hx, const float* hy, const float* dm_x, const float* dm_y,
                             float* dhx, float* dhy, int64_t numel, gdl_stream_t s) {
  GDL_REQUIRE(hx && hy && dm_x && dm_y && dhx && dhy && numel > 0, "gdl_gated_bwd: bad arguments");
  gated_bwd_kernel<<<(unsigned)ceil_div64(numel, 256), 256, 0, (cudaStream_t)s>>>(hx, hy, dm_x, dm_y, dhx, dhy, numel);
  GDL_CHECK_LAUNCH("gated_bwd_kernel");
  return GDL_OK;
}

extern "C" int64_t gdl_gated_head_scratch_floats(int B, int n) { return (int64_t)B * 512 + (int64_t)B * n + (int64_t)B * 3; }

extern "C" int gdl_dgl_head_gated(const float* a, const float* v, const float* Wx, const float* bx, const float* Wy,
                                  const float* by, const float* Wo, const float* bo, const int64_t* labels, float alpha,
                                  float inv_batch, float* logits, float* losses, float* da, float* dv, float* dWo,
                                  float* dbo, float* scratch, int B, int D, int n, gdl_stream_t s) {
  GDL_REQUIRE(a && v && Wx && bx && Wy && by && Wo && bo && labels && logits && losses && da && dv && dWo && dbo && scratch,
              "gdl_dgl_head_gated: null pointer");
  GDL_REQUIRE(B > 0 && D == kGatedD && n > 0 && n <= kHeadMaxN, "gdl_dgl_head_gated: bad shape (D must be 512, n <= 512)");
  float* m_out = scratch;
  float* g_out = m_out + (int64_t)B * D;
  float* loss_rows = g_out + (int64_t)B * n;
  dgl_gated_sample_kernel<<<B, kHeadThreads, 0, (cudaStream_t)s>>>(a, v, Wx, bx, Wy, by, Wo, bo, labels, alpha, inv_batch,
                                                                   logits, da, dv, m_out, g_out, loss_rows, B, n);
  GDL_CHECK_LAUNCH("dgl_gated_sample_kernel");
  const int64_t total = (int64_t)n * D + n + 3;
  dgl_gated_param_kernel<<<(unsigned)ceil_div64(total, 256), 256, 0, (cudaStream_t)s>>>(m_out, g_out, loss_rows, inv_batch,
                                                                                       dWo, dbo, losses, B, n);
  GDL_CHECK_LAUNCH("dgl_gated_param_kernel");
  return GDL_OK;
}
