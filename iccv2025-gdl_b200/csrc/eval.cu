// eval.cu — the eval-mode head of valid() / model(...) in eval mode (reference main_dgl.py:168-222,
// models/basic_model.py:65-86, models/fusion_modules.py).
//
//  * gdl_eval_head : one CTA per sample, starting from the two bf16 NHWC layer-4 maps the eval encoders write:
//    global average pooling (audio over h*w, visual over T*h*w per sample = adaptive_avg_pool3d), the three logit
//    sets of the concat / sum / gated head (gated honours x_gate), the arg-max of each row and the per-head correct
//    counts, added into an int64 device counter.  kind 3 only pools (the FiLM head runs its GEMMs next).
//  * gdl_eval_count : arg-max + counts over given logits [3,B,n] (the FiLM head's count step).
//  * gdl_eval_confusion : arg-max over given logits [3,B,n] + per-head confusion matrices conf[h][label][pred]
//    (the per-class report of valid_report(); a separate launch, paid only when a report is asked for).
// Every reduction runs in a fixed order and the counts are integers, so the results are deterministic.
#include "common.cuh"

namespace gdl {

constexpr int kEvalThreads = 256;
constexpr int kEvalD = 512;
constexpr int kEvalMaxN = 512;

__device__ __forceinline__ float eval_sigmoid(float x) { return 1.f / (1.f + expf(-x)); }

// (v, i) beats (bv, bi): torch.argmax order — NaN is the largest value, ties go to the lowest index
__device__ __forceinline__ bool argmax_better(float v, int i, float bv, int bi) {
  if (bi < 0) return true;
  const bool nv = v != v, nb = bv != bv;
  if (nv || nb) return nv && (!nb || i < bi);
  return v > bv || (v == bv && i < bi);
}

// arg-max of z[0..n) by one warp (result valid in every lane)
__device__ __forceinline__ int warp_argmax(const float* z, int n) {
  const int lane = threadIdx.x & 31;
  float bv = 0.f;
  int bi = -1;
  for (int j = lane; j < n; j += 32)
    if (argmax_better(z[j], j, bv, bi)) {
      bv = z[j];
      bi = j;
    }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (oi >= 0 && argmax_better(ov, oi, bv, bi)) {
      bv = ov;
      bi = oi;
    }
  }
  return bi;
}

// mean over G positions of one sample's [G][512] bf16 map -> out[512]; part[4][512] is shared scratch.
// Thread t sums channel group t % 64 over positions t / 64, t / 64 + 4, ...; the four partials are added in order.
__device__ __forceinline__ void eval_pool(const bf16* __restrict__ x, int G, float* __restrict__ part,
                                          float* __restrict__ out) {
  const int tid = threadIdx.x, cg = tid & 63, q = tid >> 6;
  float acc[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) acc[c] = 0.f;
  const bf16* p = x + cg * 8;
#pragma unroll 4
  for (int g = q; g < G; g += 4) {
    float f[8];
    unpack8(ld_stream16(p + (int64_t)g * kEvalD), f);
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] += f[c];
  }
#pragma unroll
  for (int c = 0; c < 8; ++c) part[q * kEvalD + cg * 8 + c] = acc[c];
  __syncthreads();
  const float inv = 1.f / (float)G;
  for (int i = tid; i < kEvalD; i += kEvalThreads)
    out[i] = (((part[i] + part[kEvalD + i]) + part[2 * kEvalD + i]) + part[3 * kEvalD + i]) * inv;
  __syncthreads();
}

__global__ void __launch_bounds__(kEvalThreads) eval_head_kernel(
    int kind, const bf16* __restrict__ fa, int Ga, const bf16* __restrict__ fv, int Gv, const float* __restrict__ Wx,
    const float* __restrict__ Wy, int ldw, const float* __restrict__ bx, const float* __restrict__ by,
    const float* __restrict__ Wo, const float* __restrict__ bo, int x_gate, const int64_t* __restrict__ labels,
    float* __restrict__ a_out, float* __restrict__ v_out, float* __restrict__ logits,
    unsigned long long* __restrict__ counts, int B, int n) {
  pdl_enter();
  constexpr int D = kEvalD;
  __shared__ float s_a[D], s_v[D];
  __shared__ float s_m[4][D];  // pooling partials, then the gated head's h_x, h_y and its three gated vectors
  __shared__ float s_z[3][kEvalMaxN];
  const int b = blockIdx.x;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  eval_pool(fa + (int64_t)b * Ga * D, Ga, &s_m[0][0], s_a);
  eval_pool(fv + (int64_t)b * Gv * D, Gv, &s_m[0][0], s_v);
  if (a_out != nullptr)
    for (int i = tid; i < D; i += kEvalThreads) {
      a_out[(int64_t)b * D + i] = s_a[i];
      v_out[(int64_t)b * D + i] = s_v[i];
    }
  if (kind == 3) return;
  if (kind == 2) {
    // gated: hx = fc_x(a), hy = fc_y(v) (one warp per output row), then the gate products
    for (int j = warp; j < D; j += kEvalThreads / 32) {
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
        s_m[0][j] = px + bx[j];
        s_m[1][j] = py + by[j];
      }
    }
    __syncthreads();
    // s_a <- the multimodal gated vector, s_v <- sig(hx) hx, s_m[2] <- sig(hy) hy
    for (int i = tid; i < D; i += kEvalThreads) {
      const float x = s_m[0][i], y = s_m[1][i];
      const float sx = eval_sigmoid(x), sy = eval_sigmoid(y);
      s_a[i] = x_gate ? sx * y : sy * x;
      s_v[i] = sx * x;
      s_m[2][i] = sy * y;
    }
    __syncthreads();
    for (int j = warp; j < n; j += kEvalThreads / 32) {  // the three logit sets share every row of fc_out
      const float* wo = Wo + (int64_t)j * D;
      float p0 = 0.f, p1 = 0.f, p2 = 0.f;
      for (int i = lane; i < D; i += 32) {
        const float w = wo[i];
        p0 = fmaf(w, s_a[i], p0);
        p1 = fmaf(w, s_v[i], p1);
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
  } else {
    // concat (kind 0: Wy = Wx + D inside fc_out, one bias) / sum (kind 1: two linears, two biases)
    for (int j = warp; j < n; j += kEvalThreads / 32) {
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
        const float bxj = bx[j];
        const float byj = kind == 0 ? bxj : by[j];
        // the module's association: (Wx a + Wy v) + b for concat, (Wx a + bx) + (Wy v + by) for sum
        s_z[0][j] = kind == 0 ? (pa + pv) + bxj : (pa + bxj) + (pv + byj);
        s_z[1][j] = pa + bxj;
        s_z[2][j] = pv + byj;
      }
    }
  }
  __syncthreads();
  if (logits != nullptr)
    for (int j = tid; j < n; j += kEvalThreads) {
      logits[((int64_t)0 * B + b) * n + j] = s_z[0][j];
      logits[((int64_t)1 * B + b) * n + j] = s_z[1][j];
      logits[((int64_t)2 * B + b) * n + j] = s_z[2][j];
    }
  if (warp < 3 && labels != nullptr) {
    const int pred = warp_argmax(s_z[warp], n);
    if (lane == 0 && (int64_t)pred == labels[b]) atomicAdd(counts + warp, 1ull);
  }
}

// one warp per (head, row) of logits [3][B][n]
__global__ void eval_count_kernel(const float* __restrict__ logits, const int64_t* __restrict__ labels,
                                  unsigned long long* __restrict__ counts, int B, int n) {
  pdl_enter();
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= 3 * (int64_t)B) return;
  const int h = int(w / B), b = int(w - (int64_t)h * B);
  const int pred = warp_argmax(logits + ((int64_t)h * B + b) * n, n);
  if ((threadIdx.x & 31) == 0 && (int64_t)pred == labels[b]) atomicAdd(counts + h, 1ull);
}

// one warp per (head, row) of logits [3][B][n]: conf[h][label][pred] += 1; a label < 0 is skipped, a label >= n is
// counted once per row (head 0) in *out_of_range and never indexes conf
__global__ void eval_confusion_kernel(const float* __restrict__ logits, const int64_t* __restrict__ labels,
                                      unsigned long long* __restrict__ conf,
                                      unsigned long long* __restrict__ out_of_range, int B, int n) {
  pdl_enter();
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= 3 * (int64_t)B) return;
  const int h = int(w / B), b = int(w - (int64_t)h * B);
  const int64_t label = labels[b];
  if (label < 0) return;
  if (label >= n) {
    if (h == 0 && (threadIdx.x & 31) == 0) atomicAdd(out_of_range, 1ull);
    return;
  }
  const int pred = warp_argmax(logits + ((int64_t)h * B + b) * n, n);
  if ((threadIdx.x & 31) == 0) atomicAdd(conf + ((int64_t)h * n + label) * n + pred, 1ull);
}

}  // namespace gdl

using namespace gdl;

extern "C" int gdl_eval_head(int kind, const void* fa, int Ga, const void* fv, int Gv, const float* Wx,
                             const float* Wy, int ldw, const float* bx, const float* by, const float* Wo,
                             const float* bo, int x_gate, const int64_t* labels, float* a_out, float* v_out,
                             float* logits, int64_t* counts, int B, int n, gdl_stream_t s) {
  GDL_REQUIRE(kind >= 0 && kind <= 3, "gdl_eval_head: kind must be 0 (concat), 1 (sum), 2 (gated) or 3 (pool only)");
  GDL_REQUIRE(fa && fv && B > 0 && Ga > 0 && Gv > 0, "gdl_eval_head: bad feature maps");
  GDL_REQUIRE(((uintptr_t)fa & 15) == 0 && ((uintptr_t)fv & 15) == 0, "gdl_eval_head: maps must be 16-byte aligned");
  GDL_REQUIRE((a_out == nullptr) == (v_out == nullptr), "gdl_eval_head: a_out and v_out go together");
  if (kind == 3) {
    GDL_REQUIRE(a_out != nullptr, "gdl_eval_head: pool-only needs a_out / v_out");
  } else {
    GDL_REQUIRE(n > 0 && n <= kEvalMaxN, "gdl_eval_head: n must be in 1..512");
    GDL_REQUIRE(Wx && Wy && bx, "gdl_eval_head: null weight");
    GDL_REQUIRE(kind == 0 ? ldw >= 2 * kEvalD : (kind == 1 ? ldw >= kEvalD && by != nullptr : (by && Wo && bo)),
                "gdl_eval_head: bad head weights");
    GDL_REQUIRE(labels == nullptr || counts != nullptr, "gdl_eval_head: labels need counts");
  }
  launch_pdl(eval_head_kernel, B, kEvalThreads, 0, (cudaStream_t)s, kind, (const bf16*)fa, Ga, (const bf16*)fv, Gv,
             Wx, Wy, ldw, bx, by, Wo, bo, x_gate, kind == 3 ? nullptr : labels, a_out, v_out, logits,
             (unsigned long long*)counts, B, n);
  GDL_CHECK_LAUNCH("eval_head_kernel");
  return GDL_OK;
}

extern "C" int gdl_eval_count(const float* logits, const int64_t* labels, int64_t* counts, int B, int n,
                              gdl_stream_t s) {
  GDL_REQUIRE(logits && labels && counts && B > 0 && n > 0, "gdl_eval_count: bad arguments");
  const int64_t threads = 3 * (int64_t)B * 32;
  launch_pdl(eval_count_kernel, (unsigned)ceil_div64(threads, 256), 256, 0, (cudaStream_t)s, logits, labels,
             (unsigned long long*)counts, B, n);
  GDL_CHECK_LAUNCH("eval_count_kernel");
  return GDL_OK;
}

extern "C" int gdl_eval_confusion(const float* logits, const int64_t* labels, int64_t* conf, int64_t* out_of_range,
                                  int B, int n, gdl_stream_t s) {
  GDL_REQUIRE(logits && labels && conf && out_of_range, "gdl_eval_confusion: null pointer");
  GDL_REQUIRE(B > 0, "gdl_eval_confusion: B must be positive");
  GDL_REQUIRE(n > 0 && n <= kEvalMaxN, "gdl_eval_confusion: n must be in 1..512");
  const int64_t threads = 3 * (int64_t)B * 32;
  launch_pdl(eval_confusion_kernel, (unsigned)ceil_div64(threads, 256), 256, 0, (cudaStream_t)s, logits, labels,
             (unsigned long long*)conf, (unsigned long long*)out_of_range, B, n);
  GDL_CHECK_LAUNCH("eval_confusion_kernel");
  return GDL_OK;
}
