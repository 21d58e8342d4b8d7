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
//  * gdl_eval_scores : softmax of given logits [3,B,n], appended class-major to a [3][n][cap] score store at a device
//    row cursor (one captured graph appends batch after batch), the labels to an int32 [cap] store, and the top-k hits
//    of every head added to an int64 counter (valid_report(ap=True)).
//  * gdl_eval_ap : the non-interpolated average precision of every (head, class) column of the score store: the column
//    sorted by score (bitonic, in shared memory or, for a long store, in a global workspace), then one pass over it.
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

// ---------------------------------------------------------------------------------------------- scores and AP
constexpr int kScoreRows = 32;          // rows of one head per CTA of eval_scores_kernel (one per lane when writing)
constexpr int kScoreThreads = 256;
constexpr int kApThreads = 1024;
constexpr int kApSmemKeys = 16384;      // 128 KB of 64-bit sort keys: columns up to 16384 rows sort in shared memory
constexpr int64_t kApMaxCap = 1 << 28;

// z_j ranks before z_y (label y): greater, or equal at a lower index; NaN is the largest value and ties with NaN
__device__ __forceinline__ bool ranks_before(float zj, int j, float zy, int y) {
  const bool nj = zj != zj, ny = zy != zy;
  if (ny) return nj && j < y;
  return nj || zj > zy || (zj == zy && j < y);
}

// CTA (row tile, head h): per row the max, the sum of exp(z - max) (lane-strided partial sums, then the xor butterfly)
// and the rank of the label's logit; then lane = row writes p = exp(z - max) / sum class by class, so consecutive
// lanes write consecutive rows of a class-major column.  Rows at store index >= cap are not written; head 0 stores the
// labels (-1 for a label outside 0..n-1) and counts the labelled rows that did not fit in *overflow.
__global__ void __launch_bounds__(kScoreThreads) eval_scores_kernel(
    const float* __restrict__ logits, const int64_t* __restrict__ labels, float* __restrict__ store,
    int* __restrict__ store_labels, const int64_t* __restrict__ cursor, unsigned long long* __restrict__ hits,
    unsigned long long* __restrict__ overflow, int64_t cap, int B, int n, int k) {
  __shared__ float s_max[kScoreRows], s_sum[kScoreRows];
  __shared__ unsigned s_hits;
  const int h = blockIdx.y, r0 = blockIdx.x * kScoreRows;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) s_hits = 0u;
  const int64_t base = *cursor;
  __syncthreads();
  for (int i = warp; i < kScoreRows && r0 + i < B; i += kScoreThreads / 32) {
    const int r = r0 + i;
    const float* z = logits + ((int64_t)h * B + r) * n;
    float m = -INFINITY;
    for (int j = lane; j < n; j += 32) m = fmaxf(m, z[j]);
    m = warp_max(m);
    float sum = 0.f;
    for (int j = lane; j < n; j += 32) sum += expf(z[j] - m);
    sum = warp_sum(sum);
    if (lane == 0) {
      s_max[i] = m;
      s_sum[i] = sum;
    }
    const int64_t y = labels[r];
    if (y >= 0 && y < n) {
      const float zy = z[y];
      unsigned before = 0;
      for (int j = lane; j < n; j += 32) before += ranks_before(z[j], j, zy, (int)y);
      before = __reduce_add_sync(0xffffffffu, before);
      if (lane == 0 && before < (unsigned)k) atomicAdd(&s_hits, 1u);
    }
  }
  __syncthreads();
  const int r = r0 + lane;
  const int64_t dst = base + r;
  if (r < B && dst < cap) {
    const float* z = logits + ((int64_t)h * B + r) * n;
    const float m = s_max[lane], sum = s_sum[lane];
    for (int c = warp; c < n; c += kScoreThreads / 32) store[((int64_t)h * n + c) * cap + dst] = expf(z[c] - m) / sum;
  }
  if (h == 0 && warp == 0 && r < B) {
    const int64_t y = labels[r];
    if (dst < cap)
      store_labels[dst] = (y >= 0 && y < n) ? (int)y : -1;
    else if (y >= 0)
      atomicAdd(overflow, 1ull);
  }
  if (tid == 0 && s_hits) atomicAdd(hits + h, (unsigned long long)s_hits);
}

// after every CTA of eval_scores_kernel has read the cursor (stream order)
__global__ void eval_scores_advance_kernel(int64_t* __restrict__ cursor, int B) {
  *cursor += B;
}

// 32-bit key whose unsigned order is the float order with NaN largest (every NaN the same key) and -0 == +0; every
// key of a number is >= 0x007fffff, so 0 sorts below all of them
__device__ __forceinline__ uint32_t ap_key(float x) {
  if (x != x) return 0xffffffffu;
  uint32_t u = __float_as_uint(x);
  if (u == 0x80000000u) u = 0u;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// exclusive prefix sum of v over the CTA (Hillis-Steele on buf[kApThreads]); *total gets the sum
__device__ __forceinline__ int ap_scan(int v, int* buf, int* total) {
  const int t = threadIdx.x;
  buf[t] = v;
  __syncthreads();
  for (int d = 1; d < kApThreads; d <<= 1) {
    const int o = t >= d ? buf[t - d] : 0;
    __syncthreads();
    buf[t] += o;
    __syncthreads();
  }
  const int incl = buf[t];
  *total = buf[kApThreads - 1];
  __syncthreads();
  return incl - v;
}

// One CTA per (head, class) column of the score store [3][n][cap].  Every row with a label in 0..n-1 becomes the key
// (ap_key(score) << 1 | positive); the keys (padded with 0 to a power of two) are sorted in descending order, so the
// sorted column depends only on the multiset of (score, positive) pairs, never on the row order.  Thread t then owns
// a contiguous chunk of the Nv sorted rows.  A group is a run of equal scores; N(>= s) of a row is its group's end
// index + 1 and TP(>= s) the positives up to that end.  Pass 1 counts each chunk's positives (scanned into the chunk's
// base) and finds its first group end; a suffix scan hands each chunk the nearest group end after it; pass 2 walks
// the chunk backwards and adds TP / N (double) for every positive.  The per-thread sums are added by a fixed tree.
__global__ void __launch_bounds__(kApThreads) eval_ap_kernel(const float* __restrict__ store,
                                                             const int* __restrict__ labels,
                                                             const int64_t* __restrict__ cursor, int64_t cap, int n,
                                                             double* __restrict__ ap, int64_t* __restrict__ support,
                                                             unsigned long long* work, int64_t work_stride) {
  extern __shared__ unsigned long long s_keys[];
  __shared__ int s_int[kApThreads];
  __shared__ int s_end[kApThreads], s_tp[kApThreads];
  __shared__ double s_sum[kApThreads];
  const int col = blockIdx.x, h = col / n, c = col - h * n;
  const int t = threadIdx.x;
  const int N = (int)min(*cursor, cap);
  int M = 1;
  while (M < N) M <<= 1;
  unsigned long long* a = work != nullptr ? work + (int64_t)col * work_stride : s_keys;
  const float* x = store + (int64_t)col * cap;
  int valid = 0;
  for (int i = t; i < M; i += kApThreads) {
    unsigned long long v = 0ull;
    if (i < N) {
      const int y = labels[i];
      if (y >= 0 && y < n) {
        v = ((unsigned long long)ap_key(x[i]) << 1) | (unsigned long long)(y == c);
        ++valid;
      }
    }
    a[i] = v;
  }
  int Nv;
  ap_scan(valid, s_int, &Nv);  // also a barrier: the keys are in place
  // bitonic sort, descending: M/2 compare-exchanges per pass
  for (int kk = 2; kk <= M; kk <<= 1)
    for (int j = kk >> 1; j > 0; j >>= 1) {
      for (int p = t; p < (M >> 1); p += kApThreads) {
        const int i = ((p & ~(j - 1)) << 1) | (p & (j - 1)), l = i + j;
        const unsigned long long u = a[i], w = a[l];
        if ((i & kk) == 0 ? u < w : u > w) {
          a[i] = w;
          a[l] = u;
        }
      }
      __syncthreads();
    }
  const int C = (Nv + kApThreads - 1) / kApThreads;
  const int lo = min(t * C, Nv), hi = min(lo + C, Nv);
  int pos = 0, first_end = -1, first_tp = 0;
  for (int i = lo; i < hi; ++i) {
    pos += (int)(a[i] & 1ull);
    if (first_end < 0 && (i == Nv - 1 || (a[i] >> 1) != (a[i + 1] >> 1))) {
      first_end = i;
      first_tp = pos;
    }
  }
  int P;
  const int base = ap_scan(pos, s_int, &P);
  s_end[t] = first_end;
  s_tp[t] = base + first_tp;
  __syncthreads();
  for (int d = 1; d < kApThreads; d <<= 1) {  // suffix scan: the nearest chunk at or after t with a group end
    int e = s_end[t], tp = s_tp[t];
    if (e < 0 && t + d < kApThreads) {
      e = s_end[t + d];
      tp = s_tp[t + d];
    }
    __syncthreads();
    s_end[t] = e;
    s_tp[t] = tp;
    __syncthreads();
  }
  int end = t + 1 < kApThreads ? s_end[t + 1] : -1, tp_end = t + 1 < kApThreads ? s_tp[t + 1] : 0;
  int cum = base + pos;  // TP(<= i) for i = hi - 1
  double sum = 0.0;
  for (int i = hi - 1; i >= lo; --i) {
    const int pi = (int)(a[i] & 1ull);
    if (i == Nv - 1 || (a[i] >> 1) != (a[i + 1] >> 1)) {
      end = i;
      tp_end = cum;
    }
    if (pi) sum += (double)tp_end / (double)(end + 1);
    cum -= pi;
  }
  s_sum[t] = sum;
  __syncthreads();
  for (int s = kApThreads / 2; s > 0; s >>= 1) {
    if (t < s) s_sum[t] += s_sum[t + s];
    __syncthreads();
  }
  if (t == 0) {
    ap[col] = P > 0 ? s_sum[0] / (double)P : __longlong_as_double(0x7ff8000000000000ll);
    if (h == 0) support[c] = P;
  }
}

// one thread per stored row with a label in 0..n-1: counts the rows with a non-finite score in any column
__global__ void eval_nonfinite_kernel(const float* __restrict__ store, const int* __restrict__ labels,
                                      const int64_t* __restrict__ cursor, int64_t cap, int n,
                                      unsigned long long* __restrict__ nonfinite) {
  const int64_t N = min(*cursor, cap);
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool bad = false;
  if (r < N) {
    const int y = labels[r];
    if (y >= 0 && y < n)
      for (int col = 0; col < 3 * n; ++col) bad |= !isfinite(store[(int64_t)col * cap + r]);
  }
  const unsigned m = __ballot_sync(0xffffffffu, bad);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd(nonfinite, (unsigned long long)__popc(m));
}

static int64_t ap_sort_len(int64_t cap) {
  int64_t M = 1;
  while (M < cap) M <<= 1;
  return M;
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
  eval_head_kernel<<<B, kEvalThreads, 0, (cudaStream_t)s>>>(kind, (const bf16*)fa, Ga, (const bf16*)fv, Gv,
             Wx, Wy, ldw, bx, by, Wo, bo, x_gate, kind == 3 ? nullptr : labels, a_out, v_out, logits,
             (unsigned long long*)counts, B, n);
  GDL_CHECK_LAUNCH("eval_head_kernel");
  return GDL_OK;
}

extern "C" int gdl_eval_count(const float* logits, const int64_t* labels, int64_t* counts, int B, int n,
                              gdl_stream_t s) {
  GDL_REQUIRE(logits && labels && counts && B > 0 && n > 0, "gdl_eval_count: bad arguments");
  const int64_t threads = 3 * (int64_t)B * 32;
  eval_count_kernel<<<(unsigned)ceil_div64(threads, 256), 256, 0, (cudaStream_t)s>>>(logits, labels,
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
  eval_confusion_kernel<<<(unsigned)ceil_div64(threads, 256), 256, 0, (cudaStream_t)s>>>(logits, labels,
             (unsigned long long*)conf, (unsigned long long*)out_of_range, B, n);
  GDL_CHECK_LAUNCH("eval_confusion_kernel");
  return GDL_OK;
}

extern "C" int gdl_eval_scores(const float* logits, const int64_t* labels, int B, int n, int k, float* store,
                               int32_t* store_labels, int64_t cap, int64_t* cursor, int64_t* hits, int64_t* overflow,
                               gdl_stream_t s) {
  GDL_REQUIRE(logits && labels && store && store_labels && cursor && hits && overflow, "gdl_eval_scores: null pointer");
  GDL_REQUIRE(B > 0, "gdl_eval_scores: B must be positive");
  GDL_REQUIRE(n > 0 && n <= kEvalMaxN, "gdl_eval_scores: n must be in 1..512");
  GDL_REQUIRE(k > 0 && k <= n, "gdl_eval_scores: k must be in 1..n");
  GDL_REQUIRE(cap > 0 && cap <= kApMaxCap, "gdl_eval_scores: cap must be in 1..2^28");
  const dim3 grid((unsigned)ceil_div64(B, kScoreRows), 3);
  eval_scores_kernel<<<grid, kScoreThreads, 0, (cudaStream_t)s>>>(logits, labels, store, (int*)store_labels,
             (const int64_t*)cursor, (unsigned long long*)hits, (unsigned long long*)overflow, cap, B, n, k);
  GDL_CHECK_LAUNCH("eval_scores_kernel");
  eval_scores_advance_kernel<<<1, 1, 0, (cudaStream_t)s>>>(cursor, B);
  GDL_CHECK_LAUNCH("eval_scores_advance_kernel");
  return GDL_OK;
}

extern "C" int64_t gdl_eval_ap_workspace_bytes(int64_t cap, int n) {
  if (cap <= 0 || n <= 0) return 0;
  const int64_t M = ap_sort_len(cap);
  return M <= kApSmemKeys ? 0 : 3 * (int64_t)n * M * (int64_t)sizeof(unsigned long long);
}

extern "C" int gdl_eval_ap(const float* store, const int32_t* store_labels, const int64_t* cursor, int64_t cap, int n,
                           double* ap, int64_t* support, int64_t* nonfinite, void* workspace, int64_t workspace_bytes,
                           gdl_stream_t s) {
  GDL_REQUIRE(store && store_labels && cursor && ap && support && nonfinite, "gdl_eval_ap: null pointer");
  GDL_REQUIRE(n > 0 && n <= kEvalMaxN, "gdl_eval_ap: n must be in 1..512");
  GDL_REQUIRE(cap > 0 && cap <= kApMaxCap, "gdl_eval_ap: cap must be in 1..2^28");
  const int64_t need = gdl_eval_ap_workspace_bytes(cap, n);
  GDL_REQUIRE(need == 0 || (workspace != nullptr && workspace_bytes >= need && ((uintptr_t)workspace & 7) == 0),
              "gdl_eval_ap: a store of more than 16384 rows needs gdl_eval_ap_workspace_bytes of workspace");
  const cudaStream_t st = (cudaStream_t)s;
  cudaError_t e = cudaMemsetAsync(nonfinite, 0, sizeof(int64_t), st);
  if (e != cudaSuccess) return cuda_fail(e, "gdl_eval_ap: cudaMemsetAsync");
  eval_nonfinite_kernel<<<(unsigned)ceil_div64(cap, 256), 256, 0, st>>>(store, (const int*)store_labels,
             cursor, cap, n, (unsigned long long*)nonfinite);
  GDL_CHECK_LAUNCH("eval_nonfinite_kernel");
  const int64_t M = ap_sort_len(cap);
  const size_t smem = need == 0 ? (size_t)M * sizeof(unsigned long long) : 0;
  e = cudaFuncSetAttribute(eval_ap_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           (int)(kApSmemKeys * sizeof(unsigned long long)));
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(eval_ap_kernel)");
  eval_ap_kernel<<<3 * n, kApThreads, smem, st>>>(store, (const int*)store_labels, cursor, cap, n, ap, support,
             need == 0 ? nullptr : (unsigned long long*)workspace, need == 0 ? (int64_t)0 : M);
  GDL_CHECK_LAUNCH("eval_ap_kernel");
  return GDL_OK;
}
