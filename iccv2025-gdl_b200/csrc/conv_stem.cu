// conv_stem.cu — the two stem convolutions (reference models/backbone.py:97-100:
// Conv2d(1|3 -> 64, kernel 7, stride 2, pad 3, bias=False)) as a space-to-depth implicit GEMM.
//
// A 7x7/s2 convolution over C channels equals a 4x4/s1 *valid* convolution over the 2x2
// space-to-depth image of the 3-padded input:
//     X[p, q, (dy,dx,c)] = x_pad3[2p+dy, 2q+dx, c]        (Hp = Ho + 3 rows, 4*C <= 16 channels)
//     y[ho, wo]          = sum_{a,b in 0..3} X[ho+a, wo+b, :] . W'[a,b,:],   W'[a,b,(dy,dx,c)] = w[2a+dy, 2b+dx, c]
// The layout kernel writes X directly (bf16, 16 channels = 32-byte pixels, padding materialised
// as zeros), so the GEMM K is 16 taps x 16 channels = 256 instead of the 448 of a tap-padded
// im2col, every tap is exactly ONE K=16 tcgen05.mma, and the 16 taps are 16 shifted views of a
// single TMA halo box {16 ch, 11 w, 19 h} (32-byte-swizzled, 6.7 KB).  The kernel is persistent,
// keeps the whole packed weight matrix (32 KB) resident in shared memory and is bound by the
// HBM write of its output, not by the tensor pipe.
//
// wgrad: per 128-pixel tile, dW'[co][(a,b,ch)] += dY[pix][co]^T . X_shift[pix][(a,ch)] with both
// operands MN-major (A = dY, 128-byte swizzle; B = four a-taps of the halo, 32-byte swizzle,
// N = 4 x 16); split over pixel ranges with deterministic fp32 partials.
#include "common.cuh"
#include "tma.cuh"

namespace gdl {
using namespace tc05;

constexpr int kSTileH = 16, kSTileW = 8;
constexpr int kSHaloW = 11, kSHaloH = 19;
constexpr int kSHaloBox = kSHaloW * kSHaloH * 32;           // 6688 bytes delivered
constexpr int kSHaloBytes = (kSHaloBox + 255) / 256 * 256;  // 6912 per stage
constexpr int kSWBytes = 16 * 64 * 32;                      // 16 taps x [64 co][16 ch]
constexpr int kSThreads = 192;

// ------------------------------------------------------------------------------------------
// layout: f32 [B,C,T,H,W] -> bf16 space-to-depth [B*T, Hp, Wp, 16]
// ------------------------------------------------------------------------------------------
// One CTA per output row (image bt, s2d row pp), one thread per s2d pixel: consecutive threads read consecutive pairs
// of source pixels of the two source rows 2pp-3, 2pp-2 of every channel (a warp covers 256 contiguous bytes per row) and
// write consecutive 32-byte pixels.  C is a template parameter so the 16 staged values stay in registers, and the only
// divisions are per CTA (the previous one-thread-per-pixel grid-stride version spent most of its issue slots on 64-bit
// div/mod and a runtime-indexed local array: 50 % issue utilisation at 19-29 % of DRAM bandwidth).
template <int C>
__global__ void __launch_bounds__(128) stem_layout_kernel(const float* __restrict__ src, bf16* __restrict__ dst,
                                                          int T, int H, int W, int Hp, int Wp) {
  const int row = blockIdx.x;
  const int bt = row / Hp, pp = row - bt * Hp;
  const int b = bt / T, t = bt - b * T;
  const int64_t HW = (int64_t)H * W;
  const float* base = src + ((int64_t)b * C * T + t) * HW;  // channel c: + c*T*HW
  const int h0 = 2 * pp - 3;
  for (int q = threadIdx.x; q < Wp; q += blockDim.x) {
    float f[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) f[k] = 0.f;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
      const int h = h0 + dy;
      if (h < 0 || h >= H) continue;
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const int w = 2 * q + dx - 3;
        if (w < 0 || w >= W) continue;
#pragma unroll
        for (int c = 0; c < C; ++c) f[(dy * 2 + dx) * C + c] = __ldg(base + (int64_t)c * T * HW + (int64_t)h * W + w);
      }
    }
    float lo[8], hi[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      lo[k] = f[k];
      hi[k] = f[8 + k];
    }
    uint4* o = reinterpret_cast<uint4*>(dst + ((int64_t)row * Wp + q) * 16);
    o[0] = pack8(lo);
    o[1] = pack8(hi);
  }
}

// fp32 OIHW [64][C][7][7] -> bf16 [64][256]  (k = (a*4+b)*16 + (dy*2+dx)*C + c)
__global__ void stem_pack_kernel(const float* __restrict__ w, const float* __restrict__ scale, bf16* __restrict__ wp, int C) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 64 * 256) return;
  int co = idx >> 8, k = idx & 255;
  int tap = k >> 4, ch = k & 15;
  int a = tap >> 2, b = tap & 3;
  float v = 0.f;
  if (ch < 4 * C) {
    int d = ch / C, c = ch - d * C;
    int r = 2 * a + (d >> 1), s = 2 * b + (d & 1);
    if (r < 7 && s < 7) v = w[((co * C + c) * 7 + r) * 7 + s];
    if (scale != nullptr) v *= scale[co];  // eval mode: BatchNorm scale folded into the weights
  }
  wp[idx] = __float2bfloat16_rn(v);
}

// ------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------
struct StemParams {
  CUtensorMap tm_x;    // X {16, Wp, Hp, N}, box {16, 11, 19, 1}, 32B swizzle
  CUtensorMap tm_w;    // packed weights {256, 64}, box {16, 64}, 32B swizzle
  CUtensorMap tm_out;  // y {64, Wo, Ho, N}, box {64, 8, 16, 1}, 128B swizzle
  float* stats;        // optional [gridDim.x][2][64]: per-CTA sum / sum of squares of the bf16 outputs (BatchNorm statistics)
  int N, Ho, Wo, tiles_h, tiles_w, tiles_total;
};

constexpr int kSFwdHaloStages = 8;
struct StemFwdSmem {
  static constexpr int W_OFF = 0;
  static constexpr int HALO_OFF = kSWBytes;
  static constexpr int OUT_OFF = (HALO_OFF + kSFwdHaloStages * kSHaloBytes + 1023) / 1024 * 1024;
  static constexpr int BAR_OFF = OUT_OFF + 128 * 128;
  static constexpr int STAT_OFF = BAR_OFF + 512;  // [4 warps][2][64] floats
  static constexpr int TOTAL = STAT_OFF + 2048 + 1024;
};

__global__ void __launch_bounds__(kSThreads, 1) stem_fwd_kernel(const __grid_constant__ StemParams p) {
  using L = StemFwdSmem;
  constexpr int HST = kSFwdHaloStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* halo_full = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
  uint64_t* halo_empty = halo_full + HST;
  uint64_t* tmem_full = halo_empty + HST;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* w_full = tmem_empty + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_full + 1);
  const int tid = threadIdx.x, warp = warp_uniform_idx();
  const int tiles_img = p.tiles_h * p.tiles_w;

  if (tid == 0) {
    for (int i = 0; i < HST; ++i) {
      mbar_init(&halo_full[i], 1);
      mbar_init(&halo_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 128);
    }
    mbar_init(w_full, 1);
    fence_mbar_init();
  }
  if (warp == 4) {
    tmem_alloc(tmem_slot, 128);
    tmem_relinquish();
  }
  if (tid == 5 * 32) {
    tma_prefetch_desc(&p.tm_x);
    tma_prefetch_desc(&p.tm_w);
    tma_prefetch_desc(&p.tm_out);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t smem_base = smem_u32(smem);

  if (warp == 5 && elect_one()) {
    // ---------------- TMA producer: weights once, then one halo per tile ----------------
    mbar_arrive_expect_tx(w_full, kSWBytes);
    for (int tap = 0; tap < 16; ++tap)
      tma_load_2d(smem_base + L::W_OFF + tap * 2048, &p.tm_w, w_full, tap * 16, 0);
    int it = 0;
    for (int t = blockIdx.x; t < p.tiles_total; t += gridDim.x, ++it) {
      const int n = t / tiles_img;
      const int rem = t - n * tiles_img;
      const int th = rem / p.tiles_w, tw = rem - th * p.tiles_w;
      const int hs = it % HST;
      if (it >= HST) mbar_wait(&halo_empty[hs], ((it / HST) - 1) & 1);
      mbar_arrive_expect_tx(&halo_full[hs], kSHaloBox);
      tma_load_4d(smem_base + L::HALO_OFF + hs * kSHaloBytes, &p.tm_x, &halo_full[hs], 0, tw * kSTileW,
                  th * kSTileH, n);
    }
  } else if (warp == 4 && elect_one()) {
    // ---------------- MMA issuer: 16 taps = 16 shifted views, one K=16 MMA each ----------------
    constexpr uint32_t idesc = make_idesc_bf16(128, 64, 0, 0);
    const uint32_t a_hi = desc_hi_sw32(kSHaloW * 32), b_hi = desc_hi_sw32(256);
    const uint32_t a_lo0 = desc_lo_sw128(smem_base + L::HALO_OFF, 16);
    const uint32_t b_lo0 = desc_lo_sw128(smem_base + L::W_OFF, 16);
    mbar_wait(w_full, 0);
    tc_fence_after();
    int it = 0;
    for (int t = blockIdx.x; t < p.tiles_total; t += gridDim.x, ++it) {
      const int acc = it & 1, hs = it % HST;
      if (it >= 2) {
        mbar_wait(&tmem_empty[acc], ((it >> 1) - 1) & 1);
        tc_fence_after();
      }
      mbar_wait(&halo_full[hs], (it / HST) & 1);
      tc_fence_after();
      const uint32_t a_lo = a_lo0 + hs * (kSHaloBytes >> 4);
#pragma unroll
      for (int tap = 0; tap < 16; ++tap) {
        const int a = tap >> 2, b = tap & 3;
        mma_bf16_ss(tmem_base + acc * 64, desc_join(a_lo + (((a * kSHaloW + b) * 32) >> 4), a_hi),
                    desc_join(b_lo0 + tap * (2048 >> 4), b_hi), idesc, tap != 0 ? 1u : 0u);
      }
      mma_commit(&halo_empty[hs]);
      mma_commit(&tmem_full[acc]);
    }
  } else if (warp < 4) {
    // ---------------- epilogue: TMEM -> bf16 -> swizzled smem -> TMA store ----------------
    // BatchNorm statistics (reference backbone.py:104 bn1, train mode) come out of the staged tile: each warp re-reads
    // the 32 rows it wrote by columns (lane = channel pair, conflict-free: one 128-byte row per load) and keeps the
    // sum / sum of squares of the bf16-rounded outputs in registers over all of the CTA's tiles; rows outside the
    // image are staged as zeros (the TMA store clips them anyway).  Fixed order of additions: deterministic.
    const int row = tid, sw = row & 7, lane = tid & 31;
    const uint32_t out_row = smem_base + L::OUT_OFF + row * 128;
    const bool want_stats = p.stats != nullptr;
    float ssum[2] = {0.f, 0.f}, ssq[2] = {0.f, 0.f};
    uint32_t col_off[8];  // byte offset of this lane's channel pair inside a staged row, per swizzle phase
#pragma unroll
    for (int k = 0; k < 8; ++k) col_off[k] = ((uint32_t)((lane >> 2) ^ k) << 4) + (lane & 3) * 4;
    const uint32_t warp_rows = smem_base + L::OUT_OFF + warp * 32 * 128;
    int it = 0;
    for (int t = blockIdx.x; t < p.tiles_total; t += gridDim.x, ++it) {
      const int n = t / tiles_img;
      const int rem = t - n * tiles_img;
      const int th = rem / p.tiles_w, tw = rem - th * p.tiles_w;
      const int acc = it & 1;
      const bool inside = (th * kSTileH + (row >> 3) < p.Ho) && (tw * kSTileW + (row & 7) < p.Wo);
      mbar_wait(&tmem_full[acc], (it >> 1) & 1);
      tc_fence_after();
      if (tid == 0) tma_store_wait_read();
      named_bar_sync(1, 128);
      const uint32_t trow = tmem_base + (uint32_t(warp * 32) << 16) + acc * 64;
#pragma unroll 1
      for (int c0 = 0; c0 < 64; c0 += 32) {
        uint32_t r[32];
        tmem_ld32(trow + c0, r);
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float f[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(r[q * 8 + i]);
          uint4 o = pack8(f);
          if (want_stats && !inside) o = make_uint4(0, 0, 0, 0);
          const int chunk = (c0 >> 3) + q;
          asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(out_row + ((chunk ^ sw) << 4)), "r"(o.x),
                       "r"(o.y), "r"(o.z), "r"(o.w)
                       : "memory");
        }
      }
      tc_fence_before();
      mbar_arrive(&tmem_empty[acc]);
      if (want_stats) {
        __syncwarp();
#pragma unroll
        for (int rr = 0; rr < 32; ++rr) {
          uint32_t w;
          asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(warp_rows + rr * 128 + col_off[rr & 7]) : "memory");
          const float lo = __uint_as_float(w << 16), hi = __uint_as_float(w & 0xffff0000u);
          ssum[0] += lo;
          ssq[0] = fmaf(lo, lo, ssq[0]);
          ssum[1] += hi;
          ssq[1] = fmaf(hi, hi, ssq[1]);
        }
      }
      fence_proxy_async();
      named_bar_sync(1, 128);
      if (tid == 0) {
        tma_store_4d(&p.tm_out, smem_base + L::OUT_OFF, 0, tw * kSTileW, th * kSTileH, n);
        tma_store_commit();
      }
    }
    if (tid == 0) tma_store_wait_all();
    if (want_stats) {  // combine the four warps in a fixed order: one partial row [2][64] per CTA
      float* sred = reinterpret_cast<float*>(smem + L::STAT_OFF);
      sred[warp * 128 + 2 * lane] = ssum[0];
      sred[warp * 128 + 2 * lane + 1] = ssum[1];
      sred[warp * 128 + 64 + 2 * lane] = ssq[0];
      sred[warp * 128 + 64 + 2 * lane + 1] = ssq[1];
      named_bar_sync(1, 128);
      p.stats[(size_t)blockIdx.x * 128 + tid] = (sred[tid] + sred[128 + tid]) + (sred[256 + tid] + sred[384 + tid]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, 128);
}

// ------------------------------------------------------------------------------------------
// wgrad
// ------------------------------------------------------------------------------------------
struct StemWgradParams {
  CUtensorMap tm_x;   // X, box {16, 11, 19, 1}, 32B swizzle
  CUtensorMap tm_dy;  // dY {64, Wo, Ho, N}, box {64, 8, 17, 1}, 128B swizzle (one row below the tile: the shifted M block)
  float* partial;     // [splits][4 a][64 co][64 (b,ch)]
  int N, Ho, Wo, tiles_h, tiles_w, tiles_total, tiles_per_split;
};
constexpr int kSWgStages = 4;
constexpr int kSWgDyRows = kSTileH + 1;
struct StemWgSmem {
  // per dY stage: 2 KB that stay zero (two 8-pixel K groups in front of the tile: the K step "rows -2, -1") + 17 tile rows
  static constexpr int DY_STAGE = 2048 + kSWgDyRows * 1024;
  static constexpr int DY_BYTES = kSWgDyRows * 1024;
  static constexpr int HALO_OFF = kSWgStages * DY_STAGE;
  static constexpr int BAR_OFF = (HALO_OFF + kSWgStages * kSHaloBytes + 1023) / 1024 * 1024;
  static constexpr int TOTAL = BAR_OFF + 512 + 1024;
};

// Every MMA uses all 128 rows of M and all of its operand bytes: M = {tap row a, tap row a-1} x 64 co — the second
// 64-row block of the MN-major A operand is the SAME dY tile one image row further (LBO = 1024 B), and
// sum_p dY[p + (1,0)] X[p + (a,b)] = sum_p' dY[p'] X[p' + (a-1,b)] — and N = 4 column taps b x 16 ch (LBO = 32 B: the next
// halo pixel).  Two accumulators (a = 1 | 0 and a = 3 | 2) instead of four half-empty ones: half the MMAs and half the
// shared-memory operand traffic, which bounded the kernel (ncu: L1/shared pipe 89 %, DRAM 36 %).  Shifted block coverage:
// tile rows 1..16 (row 16 = the next tile's row 0, or TMA zero fill below the image), so only row 0 of the IMAGE is
// missing for a-1: tiles of the first tile row run one more K step over "rows -2, -1", where block 0 reads the 2 KB of
// zeros kept in front of the tile and block 1 reads (zeros, row 0).
__global__ void __launch_bounds__(kSThreads, 1) stem_wgrad_kernel(const __grid_constant__ StemWgradParams p) {
  using L = StemWgSmem;
  constexpr int ST = kSWgStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
  uint64_t* empty = full + ST;
  uint64_t* tmem_full = empty + ST;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);
  const int tid = threadIdx.x, warp = warp_uniform_idx();
  const int tiles_img = p.tiles_h * p.tiles_w;
  const int t0 = blockIdx.x * p.tiles_per_split;
  const int t1 = min(t0 + p.tiles_per_split, p.tiles_total);

  {  // zero every operand byte once: the zero K groups in front of each dY tile, and finite values wherever the extra
     // K step's B descriptor points in front of a halo (0 x NaN would poison the accumulator)
    uint4* z = reinterpret_cast<uint4*>(smem);
    for (int i = tid; i < (L::BAR_OFF >> 4); i += kSThreads) z[i] = make_uint4(0, 0, 0, 0);
  }
  if (tid == 0) {
    for (int i = 0; i < ST; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(tmem_full, 1);
    fence_mbar_init();
  }
  if (warp == 4) {
    tmem_alloc(tmem_slot, 128);
    tmem_relinquish();
  }
  if (tid == 5 * 32) {
    tma_prefetch_desc(&p.tm_x);
    tma_prefetch_desc(&p.tm_dy);
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t smem_base = smem_u32(smem);

  if (warp == 5 && elect_one()) {
    int it = 0;
    for (int t = t0; t < t1; ++t, ++it) {
      const int n = t / tiles_img;
      const int rem = t - n * tiles_img;
      const int th = rem / p.tiles_w, tw = rem - th * p.tiles_w;
      const int st = it % ST;
      if (it >= ST) mbar_wait(&empty[st], ((it / ST) - 1) & 1);
      mbar_arrive_expect_tx(&full[st], kSHaloBox + L::DY_BYTES);
      tma_load_4d(smem_base + L::HALO_OFF + st * kSHaloBytes, &p.tm_x, &full[st], 0, tw * kSTileW, th * kSTileH, n);
      // pixels outside the image are zero-filled in dY, so they contribute nothing
      tma_load_4d(smem_base + st * L::DY_STAGE + 2048, &p.tm_dy, &full[st], 0, tw * kSTileW, th * kSTileH, n);
    }
  } else if (warp == 4 && elect_one()) {
    constexpr uint32_t idesc = make_idesc_bf16(128, 64, 1, 1);
    const uint32_t a_hi = desc_hi_sw128(1024);            // dY: MN-major, 128B rows, K groups of 8 pixels = tile rows
    const uint32_t b_hi = desc_hi_sw32(kSHaloW * 32);     // halo: K groups of 8 pixels one image row apart
    int it = 0;
    for (int t = t0; t < t1; ++t, ++it) {
      const int st = it % ST;
      const int rem = t % tiles_img;
      const int jstart = rem < p.tiles_w ? -1 : 0;  // first tile row of an image: the extra K step (see above)
      mbar_wait(&full[st], (it / ST) & 1);
      tc_fence_after();
      const uint32_t dy0 = smem_base + st * L::DY_STAGE + 2048;
      const uint32_t halo0 = smem_base + L::HALO_OFF + st * kSHaloBytes;
      for (int j = jstart; j < 8; ++j) {  // 16 pixels = tile rows 2j, 2j+1 (block 1: 2j+1, 2j+2)
        const uint32_t a_lo = desc_lo_sw128(dy0 + j * 2048, 1024);  // LBO: the second M block is one tile row further
#pragma unroll
        for (int ai = 0; ai < 2; ++ai) {
          const int a = 2 * ai + 1;
          const uint32_t b_lo = desc_lo_sw128(halo0 + (2 * j + a) * (kSHaloW * 32), 32);  // LBO: next column tap b
          mma_bf16_ss(tmem_base + ai * 64, desc_join(a_lo, a_hi), desc_join(b_lo, b_hi), idesc,
                      (it != 0 || j != jstart) ? 1u : 0u);
        }
      }
      mma_commit(&empty[st]);
    }
    mma_commit(tmem_full);
  } else if (warp < 4) {
    // row = (block, co): block 0 holds tap row a = 2*ai + 1, block 1 tap row a - 1
    mbar_wait(tmem_full, 0);
    tc_fence_after();
    const int blk = tid >> 6, co = tid & 63;
    const uint32_t trow = tmem_base + (uint32_t(warp * 32) << 16);
    for (int ai = 0; ai < 2; ++ai) {
      const int a = 2 * ai + 1 - blk;
      float* out = p.partial + (size_t)blockIdx.x * 4 * 64 * 64 + ((size_t)a * 64 + co) * 64;
#pragma unroll 1
      for (int c0 = 0; c0 < 64; c0 += 32) {
        uint32_t r[32];
        tmem_ld32(trow + ai * 64 + c0, r);
        tmem_ld_wait();
        if (t1 > t0) {
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<uint4*>(out + c0 + q * 4) = make_uint4(r[q * 4], r[q * 4 + 1], r[q * 4 + 2], r[q * 4 + 3]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, 128);
}

// partial [splits][a][co][b*16+ch] -> dw OIHW [64][C][7][7]
__global__ void stem_wgrad_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw, int splits,
                                         int C) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 64 * C * 49) return;
  int s = idx % 7;
  int r = (idx / 7) % 7;
  int c = (idx / 49) % C;
  int co = idx / (49 * C);
  int a = r >> 1, dy = r & 1, b = s >> 1, dx = s & 1;
  int ch = (dy * 2 + dx) * C + c;
  const size_t off = ((size_t)a * 64 + co) * 64 + b * 16 + ch;
  float acc = 0.f;
  for (int sp = 0; sp < splits; ++sp) acc += partial[(size_t)sp * 4 * 64 * 64 + off];
  dw[idx] = acc;
}

static int stem_splits(int tiles_total) {
  int splits = tiles_total < kNumSMs ? tiles_total : kNumSMs;
  return splits < 1 ? 1 : splits;
}

}  // namespace gdl

using namespace gdl;

extern "C" int gdl_stem_geometry(int H, int W, int* Ho, int* Wo, int* Hp, int* Wp) {
  if (H < 7 || W < 7 || !Ho || !Wo || !Hp || !Wp) return GDL_EINVAL;
  *Ho = (H + 6 - 7) / 2 + 1;
  *Wo = (W + 6 - 7) / 2 + 1;
  *Hp = *Ho + 3;
  *Wp = *Wo + 3;
  return GDL_OK;
}

extern "C" int gdl_stem_layout(const float* src, void* dst, int B, int C, int T, int H, int W, gdl_stream_t s) {
  GDL_REQUIRE(src && dst && B > 0 && C > 0 && C <= 4 && T > 0, "gdl_stem_layout: bad arguments");
  int Ho, Wo, Hp, Wp;
  GDL_REQUIRE(gdl_stem_geometry(H, W, &Ho, &Wo, &Hp, &Wp) == GDL_OK, "gdl_stem_layout: bad shape");
  const int64_t rows = (int64_t)B * T * Hp;
  GDL_REQUIRE(rows < ((int64_t)1 << 31), "gdl_stem_layout: too many rows");
  const cudaStream_t st = (cudaStream_t)s;
  switch (C) {
    case 1: stem_layout_kernel<1><<<(unsigned)rows, 128, 0, st>>>(src, (bf16*)dst, T, H, W, Hp, Wp); break;
    case 2: stem_layout_kernel<2><<<(unsigned)rows, 128, 0, st>>>(src, (bf16*)dst, T, H, W, Hp, Wp); break;
    case 3: stem_layout_kernel<3><<<(unsigned)rows, 128, 0, st>>>(src, (bf16*)dst, T, H, W, Hp, Wp); break;
    default: stem_layout_kernel<4><<<(unsigned)rows, 128, 0, st>>>(src, (bf16*)dst, T, H, W, Hp, Wp); break;
  }
  GDL_CHECK_LAUNCH("stem_layout_kernel");
  return GDL_OK;
}

extern "C" int gdl_stem_pack_weights(const float* w_oihw, void* w_packed, int C, gdl_stream_t s) {
  GDL_REQUIRE(w_oihw && w_packed && C > 0 && C <= 4, "gdl_stem_pack_weights: bad arguments");
  stem_pack_kernel<<<64, 256, 0, (cudaStream_t)s>>>(w_oihw, nullptr, (bf16*)w_packed, C);
  GDL_CHECK_LAUNCH("stem_pack_kernel");
  return GDL_OK;
}

extern "C" int gdl_stem_pack_weights_scaled(const float* w_oihw, const float* scale64, void* w_packed, int C,
                                            gdl_stream_t s) {
  GDL_REQUIRE(w_oihw && scale64 && w_packed && C >= 1 && C <= 4, "gdl_stem_pack_weights_scaled: bad arguments");
  stem_pack_kernel<<<64, 256, 0, (cudaStream_t)s>>>(w_oihw, scale64, (bf16*)w_packed, C);
  GDL_CHECK_LAUNCH("stem_pack_kernel(scaled)");
  return GDL_OK;
}

static int stem_fwd_impl(const void* x16, const void* w_packed, void* y, int N, int H, int W, float* stats, int* stats_rows,
                         gdl_stream_t s) {
  GDL_REQUIRE(x16 && w_packed && y && N > 0, "gdl_stem_fwd: bad arguments");
  int Ho, Wo, Hp, Wp;
  GDL_REQUIRE(gdl_stem_geometry(H, W, &Ho, &Wo, &Hp, &Wp) == GDL_OK, "gdl_stem_fwd: bad shape");
  const CUtensorMap* tx = tmap_nhwc16(x16, N, Hp, Wp, kSHaloW, kSHaloH);
  const CUtensorMap* tw = tmap_rows16(w_packed, 64, 256, 64);
  const CUtensorMap* to = tmap_nhwc(y, N, Ho, Wo, 64, kSTileW, kSTileH);
  if (!tx || !tw || !to) return GDL_ECUDA;
  StemParams p;
  p.tm_x = *tx; p.tm_w = *tw; p.tm_out = *to;
  p.stats = stats;
  p.N = N; p.Ho = Ho; p.Wo = Wo;
  p.tiles_h = (Ho + kSTileH - 1) / kSTileH;
  p.tiles_w = (Wo + kSTileW - 1) / kSTileW;
  p.tiles_total = N * p.tiles_h * p.tiles_w;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t err = cudaFuncSetAttribute(stem_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, StemFwdSmem::TOTAL);
    if (err != cudaSuccess) return cuda_fail(err, "cudaFuncSetAttribute(stem_fwd)");
    attr_set = true;
  }
  // two CTAs per SM (80 KB of shared memory, 128 TMEM columns each): the kernel is bound by its output writes,
  // and a second resident CTA hides their latency (measured 0.42 -> 0.32 ms on the visual stem)
  const int grid = p.tiles_total < 2 * kNumSMs ? p.tiles_total : 2 * kNumSMs;
  stem_fwd_kernel<<<grid, kSThreads, StemFwdSmem::TOTAL, (cudaStream_t)s>>>(p);
  GDL_CHECK_LAUNCH("stem_fwd_kernel");
  if (stats_rows) *stats_rows = grid;
  return GDL_OK;
}

extern "C" int gdl_stem_fwd(const void* x16, const void* w_packed, void* y, int N, int H, int W, gdl_stream_t s) {
  return stem_fwd_impl(x16, w_packed, y, N, H, W, nullptr, nullptr, s);
}

extern "C" int gdl_stem_fwd_stats(const void* x16, const void* w_packed, void* y, int N, int H, int W, float* bn_partial,
                                  int* bn_partial_rows, gdl_stream_t s) {
  GDL_REQUIRE(bn_partial && bn_partial_rows, "gdl_stem_fwd_stats: null pointer");
  return stem_fwd_impl(x16, w_packed, y, N, H, W, bn_partial, bn_partial_rows, s);
}

extern "C" int64_t gdl_stem_wgrad_workspace_bytes(int N, int H, int W) {
  int Ho, Wo, Hp, Wp;
  if (gdl_stem_geometry(H, W, &Ho, &Wo, &Hp, &Wp) != GDL_OK || N <= 0) return GDL_EINVAL;
  int tiles = N * ((Ho + kSTileH - 1) / kSTileH) * ((Wo + kSTileW - 1) / kSTileW);
  return (int64_t)stem_splits(tiles) * 4 * 64 * 64 * (int64_t)sizeof(float);
}

extern "C" int gdl_stem_wgrad(const void* x16, const void* dy, float* dw_oihw, int C, int N, int H, int W,
                              void* workspace, int64_t workspace_bytes, gdl_stream_t s) {
  GDL_REQUIRE(x16 && dy && dw_oihw && workspace && C > 0 && C <= 4 && N > 0, "gdl_stem_wgrad: bad arguments");
  int Ho, Wo, Hp, Wp;
  GDL_REQUIRE(gdl_stem_geometry(H, W, &Ho, &Wo, &Hp, &Wp) == GDL_OK, "gdl_stem_wgrad: bad shape");
  StemWgradParams p;
  const CUtensorMap* tx = tmap_nhwc16(x16, N, Hp, Wp, kSHaloW, kSHaloH);
  const CUtensorMap* td = tmap_nhwc(dy, N, Ho, Wo, 64, kSTileW, kSWgDyRows);
  if (!tx || !td) return GDL_ECUDA;
  p.tm_x = *tx; p.tm_dy = *td;
  p.partial = (float*)workspace;
  p.N = N; p.Ho = Ho; p.Wo = Wo;
  p.tiles_h = (Ho + kSTileH - 1) / kSTileH;
  p.tiles_w = (Wo + kSTileW - 1) / kSTileW;
  p.tiles_total = N * p.tiles_h * p.tiles_w;
  int splits = stem_splits(p.tiles_total);
  p.tiles_per_split = (p.tiles_total + splits - 1) / splits;
  splits = (p.tiles_total + p.tiles_per_split - 1) / p.tiles_per_split;
  if (workspace_bytes < (int64_t)splits * 4 * 64 * 64 * (int64_t)sizeof(float)) {
    set_last_error("gdl_stem_wgrad: workspace too small");
    return GDL_ENOMEM;
  }
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(stem_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         StemWgSmem::TOTAL);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(stem_wgrad)");
    attr_set = true;
  }
  stem_wgrad_kernel<<<splits, kSThreads, StemWgSmem::TOTAL, (cudaStream_t)s>>>(p);
  GDL_CHECK_LAUNCH("stem_wgrad_kernel");
  stem_wgrad_reduce_kernel<<<(64 * C * 49 + 255) / 256, 256, 0, (cudaStream_t)s>>>((const float*)workspace, dw_oihw, splits, C);
  GDL_CHECK_LAUNCH("stem_wgrad_reduce_kernel");
  return GDL_OK;
}
